#!/usr/bin/env python
"""bench.py -- ECDSA-P256 verifies/sec of the B200 verifier (BASELINE.json metric) and of the reference's CPU path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes what the last timed step of `value` returned -- the all-gathered validity bitmask, one float32 0/1
per signature in the order that step verified them -- as DIR/valid.npy.  The inputs are seeded, so two builds run with the
same arguments can be compared output for output.

A "step" is one pass of the hot path over one batch of B synthetic signatures per GPU (default B = 65 536, the
BASELINE.json configs[1] workload: K = 64 keys, SHA-256 digests of 1 KiB messages, low-S DER signatures).  With N > 1
every rank verifies its own B signatures (weak scaling) and the validity bitmask is all-gathered (NCCL) inside the
timed region.

Printed JSON (one line, rank 0):
  value        whole-job verifies/s, inputs resident in HBM, CUDA-event time summed over K steps (max over ranks);
  e2e          same metric through the C-ABI call fabgpu_bccsp_verify_batch with HOST buffers (raw DER signatures,
               digests, keys): host gates + pinned staging + H2D + kernel + D2H inside the timed region;
  roofline     HBM view of the verify kernel (algorithmic 160.125 B/verify) -- the path is integer-issue bound,
               so `roofline_int` carries the binding resource (217 600 32-bit MACs/verify vs the fma-pipe peak);
  cpu_baseline the oracle's C port (OpenSSL curve arithmetic + restated bccsp/sw gates) on this box's host cores.
--impl reference times that same CPU port as the reference arm (the reference itself is Go; no Go toolchain exists).
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "ECDSA-P256 verifies/sec"
ALG_BYTES_PER_VERIFY = 160.125          # SURVEY.md section 8(d): 5 x 32 B in, 1 bit out
ALG_MACS_PER_VERIFY = 217600            # SURVEY.md section 8(d): 3 400 modular multiplications x 64 MACs (generic kernel)


def alg_macs_cached(wg, wq):
    """key-table kernel: one mixed addition (8M + 3S = 11 field multiplications) per window of both tables + 3 for the final
    check, 64 32x32 MACs per field multiplication (the scalar inversion and the reductions are not counted)."""
    windows = (256 + wg - 1) // wg + (256 + wq - 1) // wq
    return (11 * windows + 3) * 64


KEYS = 64


def workload_string(B):
    """config.workload, identical for both arms (the driver compares the two strings)."""
    return "configs[1]: %d-signature batch per step and GPU, %d keys, SHA-256 digests of 1 KiB messages, low-S DER signatures" % (B, KEYS)

NCU_DRAM_BYTES_PER_LAUNCH_64K = 228455168 + 6074880   # ecdsa_verify_cached_kernel, profiles/r2_final_cached_ncu_summary.txt (dram read + write)
NCU_FMAHEAVY_BUSY = 0.6286              # sm__pipe_fmaheavy_cycles_active, % of elapsed, same capture: the binding unit of that kernel


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured", float(d.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback", 1965.0


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) >= 8:
                self.rows.append(f)

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit())
        reasons = []
        for i, name in ((4, "hw_slowdown"), (5, "hw_thermal_slowdown"), (6, "sw_thermal_slowdown"), (7, "sw_power_cap")):
            if any(r[i].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        mx = max([float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()] or [0.0])
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": reasons, "samples": len(sm)}


def pin_to_gpu_numa(dev_index):
    """One process per GPU: keep this rank's host threads (and, by first touch, its pinned staging buffers) on the CPU socket its
    GPU hangs off -- on an 8-GPU box GPUs 4-7 sit on NUMA node 1, and staging from the other socket halves the copy rate."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(dev_index)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        cpus = open("/sys/bus/pci/devices/%s/local_cpulist" % bdf).read().strip()
        ids = set()
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        if ids:
            os.sched_setaffinity(0, ids)
            return {"pci": bdf, "cpus": cpus}
    except Exception as e:                                               # not fatal: the run proceeds unpinned
        return {"error": str(e)[:120]}
    return None


def best_thread_count(w):
    """Host threads that give the CPU port its best throughput on this box (all logical CPUs is not always it)."""
    from oracle import fast
    ncpu = os.cpu_count() or 1
    cand = sorted({ncpu, max(1, ncpu // 2), max(1, ncpu // 4)}, reverse=True)
    n = min(w.n, 32768)
    best, best_rate = ncpu, 0.0
    for t in cand:
        rate = 0.0
        for _ in range(2):
            t0 = time.perf_counter()
            fast.verify_batch(w.keys_xy, w.key_idx[:n], w.digest[:n], w.dig_off()[:n + 1], w.sigs, w.sig_off[:n + 1], nthreads=t)
            rate = max(rate, n / (time.perf_counter() - t0))
        if rate > best_rate:
            best, best_rate = t, rate
    return best


def cpu_port_rate(w, threads, min_seconds=4.0):
    """verifies/s of the oracle's C port on `threads` host threads over the workload `w` (bounded sample)."""
    from oracle import fast
    fast.verify_batch(w.keys_xy, w.key_idx[:2048], w.digest[:2048], w.dig_off()[:2049], w.sigs, w.sig_off[:2049], nthreads=threads)  # warm
    done, t0 = 0, time.perf_counter()
    while True:
        st = fast.verify_batch(w.keys_xy, w.key_idx, w.digest, w.dig_off(), w.sigs, w.sig_off, nthreads=threads)
        done += w.n
        el = time.perf_counter() - t0
        if el >= min_seconds:
            break
    assert (st == 0).all()
    return done / el, done, el


def run_reference(args):
    """Reference arm: the reference's own CPU path is Go crypto/ecdsa behind bccsp/sw; Go is absent from this image, so
    the arm times the oracle's C port of it (restated gates + OpenSSL nistz256 arithmetic) on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from tools import workload
    w = workload.Workload(args.batch, KEYS, seed=workload.DEFAULT_SEED + 2)
    from oracle import fast
    cores = best_thread_count(w)
    for _ in range(args.warmup):
        fast.verify_batch(w.keys_xy, w.key_idx, w.digest, w.dig_off(), w.sigs, w.sig_off, nthreads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        st = fast.verify_batch(w.keys_xy, w.key_idx, w.digest, w.dig_off(), w.sigs, w.sig_off, nthreads=cores)
    el = time.perf_counter() - t0
    assert (st == 0).all()
    v = args.steps * w.n / el
    emit({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "verifies/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs (256-bit modular integer)",
        "data": "synthetic",
        "config": {"workload": workload_string(w.n), "batch_per_step": w.n,
                   "note": "the CPU arm runs on rank 0 only and verifies one batch per step whatever --gpus says (the GPU arm verifies one batch per GPU per step); both are rates"},
        "cpu_baseline": {"value": v, "unit": "verifies/s", "cores": cores, "kind": "port", "value_per_core": v / max(1, cores),
                         "sample": "%d steps x %d signatures through oracle/c (bccsp/sw gates + ecdsa.Verify steps on OpenSSL BN/EC primitives), %d of %d logical CPUs (best of all/half/quarter)" % (args.steps, w.n, cores, os.cpu_count() or 1)},
        "e2e": {"value": v, "unit": "verifies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


def run_gpu(args):
    import torch
    import torch.distributed as dist
    pkg = importlib.import_module("fabric-mod_b200")
    sharding = importlib.import_module("fabric-mod_b200.sharding")
    from tools import workload

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node %d for --gpus %d" % (args.gpus, args.gpus))
    if world > 1 and "FABGPU_GATE_THREADS" not in os.environ:       # ranks share the host: split its threads between them
        os.environ["FABGPU_GATE_THREADS"] = str(max(4, (os.cpu_count() or 8) // (2 * world)))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = pin_to_gpu_numa(local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    B = args.batch
    n_total = B * world
    # this rank's slice of the synthetic workload (rank-seeded so ranks do not verify identical bytes)
    w = workload.Workload(B, KEYS, seed=workload.DEFAULT_SEED + 2 + 1000 * rank)
    # one process per GPU shares the host: give each rank's staging pool its share of the cores (the pool spins briefly before
    # sleeping; eight ranks with the default 32 threads each would oversubscribe a 128-thread host)
    os.environ.setdefault("FABGPU_GATE_THREADS", str(max(4, min(32, (os.cpu_count() or 8) // (2 * world)))))
    ctx = pkg.binding.Context(max_batch=B, device_ids=[local])

    # ---- device-resident leg: ROT distinct input buffers (ROT x 10.5 MB = 168 MB > the 126 MB L2), steps back to back ----------------
    # The kernel's other input -- the window tables, 3.2 GB + 64 x 64 MiB, gathered at random -- is far larger than the L2 by itself.  The
    # same loop with a 256 MiB fill between steps (round 1's method) is timed beside it (config.value_l2_fill_between_steps): the fill
    # leaves the L2 full of DIRTY lines whose write-back competes with the next launch's table gathers, which no real batch stream does.
    ROT = 16
    host = [w.qx(), w.qy(), w.digest, w.r, w.s]
    bufs = []
    for k in range(ROT):
        perm = np.roll(np.arange(B), 997 * k)                # same tuples, different order => different bytes per buffer
        bufs.append([torch.from_numpy(np.ascontiguousarray(a[perm])).to(dev) for a in host])
    words = sharding.shard_words(n_total, world)
    assert words == B // 32
    local_mask = torch.zeros(words, dtype=torch.int32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev)

    # The provider registers a key once, when the identity is imported (KeyImport); steady-state batches then run the
    # key-table kernel.  `value` is that steady state; `value_generic` is the kernel for never-seen keys.
    t0 = time.perf_counter()
    slots = ctx.keys_register(w.keys_xy) & 0xFFF          # device-resident API takes raw slot indices
    key_register_ms = (time.perf_counter() - t0) * 1e3
    assert (slots >= 0).all()
    kslots = [torch.from_numpy(np.ascontiguousarray(slots[w.key_idx][np.roll(np.arange(B), 997 * k)])).to(dev) for k in range(ROT)]

    # N > 1: two ways to reassemble the bitmask, both timed with the same loop: the NCCL all-gather north_star names (the default `value`:
    # measured faster at every N on this pool's boxes, profiles/r2_scale.txt) and the library's own exchange over peer memory (P2P stores
    # from the verify kernel's epilogue, fabgpu_verify_p256_device_keyed_allgather; --collective p2p makes it the `value`).
    peer = None
    peer_note = None
    main_nccl = args.collective == "nccl"
    if world > 1:
        peer = sharding.PeerMaskExchange(ctx, n_total, world, rank, dev)
        if not peer.ok:                                            # no peer access on this box: every rank falls back to the NCCL all-gather
            peer_note, peer = "peer-memory exchange unavailable (%s): NCCL all-gather used" % (peer.error or "another rank failed"), None

    def step(k, generic=False, nccl=None):
        t = bufs[k % ROT]
        if nccl is None:
            nccl = main_nccl
        if peer is not None and not generic and not nccl:
            return peer.verify(True, kslots[k % ROT].data_ptr(), 0, 0, t[2].data_ptr(), t[3].data_ptr(), t[4].data_ptr(), B, stream.cuda_stream)
        if generic:
            ctx.verify_p256_device(t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr(), t[4].data_ptr(), B,
                                   local_mask.data_ptr(), 0, stream.cuda_stream)
        else:
            ctx.verify_p256_device_keyed(True, kslots[k % ROT].data_ptr(), 0, 0, t[2].data_ptr(), t[3].data_ptr(), t[4].data_ptr(), B,
                                         local_mask.data_ptr(), 0, stream.cuda_stream)
        return sharding.allgather_mask(local_mask, n_total, world)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    for k in range(args.warmup):
        full = step(k)
    sync_all()
    assert args.warmup == 0 or bool((full == -1).all()), "warm-up bitmask is not all-valid"
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    sync_all()
    wall0 = time.perf_counter()
    for k in range(args.steps):
        ev[k][0].record(stream)
        full = step(k)
        ev[k][1].record(stream)
    sync_all()
    wall = time.perf_counter() - wall0
    launches = ctx.launch_count() - launches0
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    assert bool((full == -1).all())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"valid": np.unpackbits(full.cpu().numpy().view(np.uint8), bitorder="little")[:n_total]})
    # the same loop with the L2 overwritten between steps (256 MiB fill, outside the event pairs)
    fev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    sync_all()
    for k in range(args.steps):
        flush.fill_(k & 0xFF)
        fev[k][0].record(stream)
        full = step(k)
        fev[k][1].record(stream)
    sync_all()
    fill_ms = sum(a.elapsed_time(b) for a, b in fev)
    assert bool((full == -1).all())
    # The same kernel with several batches in flight (one stream per batch, inputs resident, no flush): a 64k batch is 512 CTAs
    # on 592 resident CTA slots, so a launch on its own leaves part of the machine idle in its tail; concurrent streams fill it.
    # This is the regime the pipelined end-to-end call runs in, and why e2e can exceed the one-batch-at-a-time `value`.
    cstreams = [torch.cuda.Stream(device=dev) for _ in range(pkg.binding.SLOTS)]
    cmasks = [torch.zeros(words, dtype=torch.int32, device=dev) for _ in cstreams]
    csteps = max(len(cstreams), args.steps)
    def cstep(k):
        t = bufs[k % ROT]
        ctx.verify_p256_device_keyed(True, kslots[k % ROT].data_ptr(), 0, 0, t[2].data_ptr(), t[3].data_ptr(), t[4].data_ptr(), B,
                                     cmasks[k % len(cstreams)].data_ptr(), 0, cstreams[k % len(cstreams)].cuda_stream)
    for k in range(len(cstreams)):
        cstep(k)
    sync_all()
    c0 = torch.cuda.Event(enable_timing=True)
    cends = [torch.cuda.Event(enable_timing=True) for _ in cstreams]
    c0.record(stream)
    for cs in cstreams:
        cs.wait_event(c0)
    for k in range(csteps):
        cstep(k)
    for cs, e in zip(cstreams, cends):
        e.record(cs)
    sync_all()
    conc_ms = max(c0.elapsed_time(e) for e in cends)
    assert all(bool((m == -1).all()) for m in cmasks)
    # the same timed loop with the OTHER way of reassembling the bitmask (comparison; N > 1 only)
    nccl_ms = 0.0
    if peer is not None:
        for k in range(args.warmup):
            full = step(k, nccl=not main_nccl)
        nev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        sync_all()
        for k in range(args.steps):
            nev[k][0].record(stream)
            full = step(k, nccl=not main_nccl)
            nev[k][1].record(stream)
        sync_all()
        nccl_ms = sum(a.elapsed_time(b_) for a, b_ in nev)
        assert bool((full == -1).all())
    # generic kernel (no key tables), same hygiene, fewer steps
    gsteps = max(3, min(args.steps, 10))
    for k in range(2):
        step(k, generic=True)
    gev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(gsteps)]
    sync_all()
    for k in range(gsteps):
        flush.fill_(k & 0xFF)
        gev[k][0].record(stream)
        full = step(k, generic=True)
        gev[k][1].record(stream)
    sync_all()
    gen_ms = sum(a.elapsed_time(b) for a, b in gev)
    assert bool((full == -1).all())

    # small-table tier (keys that recur without being busy: 264 KiB per key, 33 mixed additions for u2*Q), same tuples, same hygiene
    small_ms = 0.0
    small_keys = 4096
    ssteps = max(3, min(args.steps, 10))
    if ctx.small_slot_capacity() >= small_keys:
        ws = workload.Workload(B, small_keys, seed=workload.DEFAULT_SEED + 11 + 1000 * rank, nthreads=os.cpu_count())
        t0 = time.perf_counter()
        codes = ctx.small_raw_codes(ctx.keys_register_small(ws.keys_xy))
        assert (codes <= -2).all()
        sbuf = [torch.from_numpy(a).to(dev) for a in (ws.digest, ws.r, ws.s)]
        sks = torch.from_numpy(np.ascontiguousarray(codes[ws.key_idx])).to(dev)
        def sstep():
            ctx.verify_p256_device_keyed(2, sks.data_ptr(), 0, 0, sbuf[0].data_ptr(), sbuf[1].data_ptr(), sbuf[2].data_ptr(), B,
                                         local_mask.data_ptr(), 0, stream.cuda_stream)
        sstep()
        torch.cuda.synchronize(dev)
        small_register_ms = (time.perf_counter() - t0) * 1e3       # build of 4 096 tables + first batch
        sstep()
        sev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(ssteps)]
        torch.cuda.synchronize(dev)
        for k in range(ssteps):
            flush.fill_(k & 0xFF)
            sev[k][0].record(stream)
            sstep()
            sev[k][1].record(stream)
        torch.cuda.synchronize(dev)
        small_ms = sum(a.elapsed_time(b) for a, b in sev)
        assert bool((local_mask == -1).all())
        del ws, sbuf, sks

    # ---- end-to-end leg: raw DER + digests + keys in host memory through the bccsp-level C-ABI call ----------
    # Headline form: the two halves of the call (fabgpu_bccsp_verify_batch_async / _wait) round-robin over the slots, one batch per slot
    # in flight -- every step still stages its host buffers, copies them H2D, runs gate + verify + status kernels and reads the
    # status bytes back D2H inside the timed region; the copies of step k+1 overlap the kernels of step k.  The one-call
    # synchronous form is timed beside it.
    e2e_steps = max(4, min(args.steps, 40))
    dig_off = w.dig_off()
    e2e_args = (w.keys_xy, w.key_idx, w.digest, dig_off, w.sigs, w.sig_off)
    for _ in range(2):
        st = ctx.bccsp_verify_batch(*e2e_args)
    assert (st == 0).all()
    sync_all()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        st = ctx.bccsp_verify_batch(*e2e_args)
    torch.cuda.synchronize(dev)
    e2e_sync_s = time.perf_counter() - t0
    assert (st == 0).all()
    e2e_phases = ctx.last_timing()
    S = pkg.binding.SLOTS                                                # batches in flight
    st_out = [np.full(B, 255, np.uint8) for _ in range(S)]
    for k in range(S):                                                   # warm every slot (first use allocates its buffers)
        ctx.bccsp_verify_batch_wait(k, ctx.bccsp_verify_batch_async(k, *e2e_args), st_out[k])

    def pipelined(submit):
        """S batches in flight round-robin over the slots; the loop is host-paced and the boxes are shared, so it is timed five times and
        the MEDIAN repetition is reported (all five are in the JSON line)."""
        reps = []
        for rep in range(5):
            sync_all()
            t0 = time.perf_counter()
            for k in range(e2e_steps):
                if k >= S:
                    ctx.bccsp_verify_batch_wait(k % S, B, st_out[k % S])    # the slot's previous batch (k - S)
                submit(k % S)
            for k in range(max(0, e2e_steps - S), e2e_steps):
                ctx.bccsp_verify_batch_wait(k % S, B, st_out[k % S])
            torch.cuda.synchronize(dev)
            reps.append(time.perf_counter() - t0)
        assert all((o == 0).all() for o in st_out)
        return reps

    # (a) the caller's arrays are ordinary (pageable) host memory: the library's staging threads copy them into its pinned buffers
    e2e_reps_pageable = pipelined(lambda sl: ctx.bccsp_verify_batch_async(sl, *e2e_args))
    # (b) HEADLINE: the batch already lies in the slots' pinned buffers (fabgpu_bccsp_batch_buffers, filled once -- what the Go
    #     provider's pre-pass does when it marshals a block): every step is H2D from pinned memory + gate + verify + status kernels + D2H
    KK = 0
    for k in range(S):
        for o in st_out:
            o[:] = 255
        KK, _ = ctx.bccsp_fill_batch_buffers(k, *e2e_args)
        ctx.bccsp_verify_batch_wait(k, ctx.bccsp_verify_batch_inplace_async(k, KK, B), st_out[k])
    e2e_reps = pipelined(lambda sl: ctx.bccsp_verify_batch_inplace_async(sl, KK, B))
    e2e_s = sorted(e2e_reps)[len(e2e_reps) // 2]
    e2e_pageable_s = sorted(e2e_reps_pageable)[len(e2e_reps_pageable) // 2]
    # (c) mix: half of the batch signed by the 64 busy identities (window tables), half by 4096 identities that sign 8 times each: too few
    #     for a window table (FABGPU_KEY_MIN_USES = 256), enough for a small one after four batches (FABGPU_SMALL_MIN_USES = 32 signatures seen) -- what a block with many client
    #     certificates looks like
    hot, cold = KEYS, 4096
    rng_m = np.random.default_rng(workload.DEFAULT_SEED + 77 + rank)
    kidx_m = np.concatenate([rng_m.integers(0, hot, size=B // 2), hot + (np.arange(B - B // 2) % cold)]).astype(np.int32)
    rng_m.shuffle(kidx_m)
    wm = workload.Workload(B, hot + cold, seed=workload.DEFAULT_SEED + 9 + 1000 * rank, key_idx=kidx_m)
    mixed_args = (wm.keys_xy, wm.key_idx, wm.digest, wm.dig_off(), wm.sigs, wm.sig_off)
    for _ in range(4):                                    # 4 x 8 signatures per cold identity: the 32 that earn a small table
        stm = ctx.bccsp_verify_batch(*mixed_args)
        assert (stm == 0).all()
    e2e_steps_saved, e2e_steps = e2e_steps, max(4, e2e_steps // 4)
    e2e_mixed_reps = pipelined(lambda sl: ctx.bccsp_verify_batch_async(sl, *mixed_args))
    e2e_mixed_steps, e2e_steps = e2e_steps, e2e_steps_saved
    e2e_mixed_s = sorted(e2e_mixed_reps)[len(e2e_mixed_reps) // 2]
    e2e_h2d = int(w.sig_off[B]) + int(dig_off[B]) + 4 * (B + 1) * 2 + 4 * B + 68 * KEYS
    e2e_d2h = B

    # ---- BASELINE.json configs[2]: block-validation replay, 10 k txs x 3 endorsements, 3-of-4 policy (rank 0 only) ----
    block_replay = None
    if rank == 0 and not args.no_block:
        from tools import blockgen
        os.environ["FABGPU_BLOCK_EVENTS"] = "1"        # per-stage CUDA-event times for the report below
        net = blockgen.Network()
        blk, binfo = blockgen.build_block(net, args.block_txs, 3, {}, seed=17)
        ctx.msp_configure([(i.serialized, i.mspid, i.xy, i.valid) for i in net.msp_table], net.policy_n_of(3), net.principals, net.channel)
        eblob, eoff = binfo["env_blob"], binfo["env_off"]           # Block.Data.Data, as TxValidator.Validate receives it
        pinned = ctx.block_buffer(len(eblob))
        pinned[:] = np.frombuffer(eblob, np.uint8)
        for _ in range(3):
            fl = ctx.validate_envelopes(pinned, eoff)
        assert fl.shape[0] == args.block_txs and not fl.any(), "block replay: not every transaction flag is VALID"
        breps = 10
        t0 = time.perf_counter()
        for _ in range(breps):
            fl = ctx.validate_envelopes(pinned, eoff)
        bms_single = (time.perf_counter() - t0) / breps * 1e3
        ph = ctx.block_timing()
        # several blocks in flight (fabgpu_validate_envelopes_async / fabgpu_validate_wait round-robin over the slots, one pinned buffer per
        # slot): the PCIe copy of block k+1 runs under the kernels of block k.  Every block is copied, walked, hashed, verified
        # and decided inside the timed region.
        bufs = [pinned]
        for k in range(1, S):
            pb = ctx.block_buffer(len(eblob), slot=k)
            pb[:] = np.frombuffer(eblob, np.uint8)
            bufs.append(pb)
        os.environ["FABGPU_BLOCK_EVENTS"] = "0"
        for k in range(S):
            ctx.validate_envelopes_async(k, bufs[k], eoff)
            assert not ctx.validate_wait(k, args.block_txs).any()
        breps2 = 30
        fls = []
        t0 = time.perf_counter()
        for k in range(breps2):
            if k >= S:
                fls.append(ctx.validate_wait(k % S, args.block_txs))
            ctx.validate_envelopes_async(k % S, bufs[k % S], eoff)
        for k in range(max(0, breps2 - S), breps2):
            fls.append(ctx.validate_wait(k % S, args.block_txs))
        bms = (time.perf_counter() - t0) / breps2 * 1e3
        assert len(fls) == breps2 and not any(f.any() for f in fls)
        block_replay = {"workload": "configs[2]: %d txs x (1 creator + 3 endorsement) signatures, 3-of-4 policy, block of %d bytes in pinned host memory" % (args.block_txs, len(blk)),
                        "api": "fabgpu_validate_envelopes_async + fabgpu_validate_wait, %d blocks in flight" % S, "ms_per_block": bms, "tx_per_s": args.block_txs / bms * 1e3,
                        "verifies_per_s": binfo["n_sigs"] / bms * 1e3, "all_flags_valid": True,
                        "single_call": {"api": "fabgpu_validate_envelopes (one blocking call per block)", "ms_per_block": bms_single,
                                        "tx_per_s": args.block_txs / bms_single * 1e3},
                        "device_stage_us": {"h2d_walk_creator_resolve_and_sha256": ph[5], "endorsement_resolve_and_sha256": ph[7], "verify_kernel": ph[8],
                                            "block_decide_kernel": ph[9]},
                        "host_us": {"enqueue": ph[0], "wait_for_device": ph[2], "duplicate_txid_pass": ph[3]}}
        # The same block shape when the channel's MSP holds 2 000 CLIENT certificates (5 transactions each) beside the 4 endorsing peers: more
        # identities than window-table slots.  The peers' keys are registered for window tables first (fabgpu_keys_register), the clients go to
        # the small tier (round 1: every identity of such an MSP stayed on the generic kernel).
        if not args.no_clients:
          try:                                            # a secondary leg: a failure here is reported in the line, it does not take the line away
              net2 = blockgen.Network(n_orgs=4, n_clients=2000, seed=0xC11E)
              blk2, binfo2 = blockgen.build_block(net2, args.block_txs, 3, {}, seed=19)
              ids2 = [(i.serialized, i.mspid, i.xy, i.valid) for i in net2.msp_table]
              eblob2, eoff2 = binfo2["env_blob"], binfo2["env_off"]

              def clients_leg(c):
                  c.keys_register(np.stack([np.frombuffer(p.xy, np.uint8) for p in net2.peers]))
                  c.msp_configure(ids2, net2.policy_n_of(3), net2.principals, net2.channel)
                  pin = c.block_buffer(len(eblob2))
                  pin[:] = np.frombuffer(eblob2, np.uint8)
                  for _ in range(3):
                      f2 = c.validate_envelopes(pin, eoff2)
                  assert f2.shape[0] == args.block_txs and not f2.any(), "block replay (clients): not every transaction flag is VALID"
                  t0_ = time.perf_counter()
                  for _ in range(10):
                      c.validate_envelopes(pin, eoff2)
                  return (time.perf_counter() - t0_) / 10 * 1e3, c.key_table_stats()
              ms_small, stats2 = clients_leg(ctx)
              os.environ["FABGPU_SMALL_SLOTS"] = "0"
              try:
                  ctx0 = pkg.binding.Context(max_batch=4096, device_ids=[local])
              finally:
                  del os.environ["FABGPU_SMALL_SLOTS"]
              ms_none, _ = clients_leg(ctx0)
              ctx0.close()
              block_replay["many_clients"] = {"workload": "%d txs x (1 creator + 3 endorsement) signatures; MSP of %d identities: 4 endorsing peers (window tables) + 2 000 client "
                                                          "certificates that sign 5 transactions each (small tables)" % (args.block_txs, len(ids2)),
                                              "api": "fabgpu_validate_envelopes (one blocking call per block)", "ms_per_block": ms_small, "tables": stats2,
                                              "ms_per_block_without_small_tables": ms_none,
                                              "without_note": "FABGPU_SMALL_SLOTS=0: the clients' 10 000 creator signatures take the generic kernel (255 doublings each)"}
          except Exception as ex:                         # noqa: BLE001 -- reported, not hidden
            block_replay["many_clients"] = {"error": repr(ex)}
    clocks = sampler.stop() if rank == 0 else None      # sampled across the three timed loops (key-table, generic, e2e)

    # ---- parity at the named multi-GPU shape (BASELINE.json configs[3] on 8 GPUs, configs[4] on 4; untimed) ----------------
    # Every rank verifies ITS contiguous shard of a batch with 5 % tampered r (+ the adversarial tail of tests/vectors.py on the
    # last rank) through the bccsp-level C-ABI call, the validity bitmask is all-gathered over NCCL exactly as in the timed
    # legs, and rank 0 compares it bit for bit with the oracle's C port run over all shards.
    parity = None
    if not args.no_parity:
        from tools import parity_workload as pw
        p_total, p_keys, p_name = pw.named_shape(world)
        shard = pw.Shard(rank, world, p_total, p_keys)
        st_shard = ctx.bccsp_verify_batch(*shard.args())
        p_words = sharding.shard_words(p_total, world)
        lw = np.zeros(p_words, np.uint32)
        bits = (st_shard == 0).astype(np.uint8)
        lw[: (shard.n + 31) // 32] = np.packbits(np.concatenate([bits, np.zeros((-shard.n) % 32, np.uint8)]).reshape(-1, 32), axis=1, bitorder="little").view("<u4").reshape(-1)
        full_mask = sharding.allgather_mask(torch.from_numpy(lw.view(np.int32)).to(dev), p_total, world).cpu().numpy().view(np.uint32)
        st_dev = torch.from_numpy(st_shard).to(dev)
        if world > 1:
            st_all = torch.empty(p_total, dtype=torch.uint8, device=dev)
            dist.all_gather_into_tensor(st_all, st_dev)
        else:
            st_all = st_dev
        st_all = st_all.cpu().numpy()
        if rank == 0:
            from oracle import fast
            ncpu = os.cpu_count() or 8
            exp, n_tamper, tail = [], 0, []
            for rk in range(world):
                sh = shard if rk == rank else pw.Shard(rk, world, p_total, p_keys)
                exp.append(pw.oracle_status(sh, min(ncpu, 64)))
                n_tamper += int(len(sh.tampered))
                tail += sh.tail
            exp = np.concatenate(exp)
            exp_mask = fast.valid_mask(exp)
            parity = {"workload": p_name + ", 5 % of r tampered (one bit), adversarial tail of tests/vectors.py on the last shard",
                      "n": int(p_total), "shards": world, "tampered": n_tamper, "tail_cases": len(tail),
                      "zeros": int(p_total - int((exp == 0).sum())), "mask_zeros_gpu": int(p_total - int(np.unpackbits(full_mask.view(np.uint8)).sum())),
                      "mask_equals_oracle": bool((full_mask == exp_mask).all()), "status_equals_oracle": bool((st_all == exp).all()),
                      "false_accepts": int(((st_all == 0) & (exp != 0)).sum()), "false_rejects": int(((st_all != 0) & (exp == 0)).sum()),
                      "collective": "all_gather_into_tensor of the uint32 mask words (%s), then of the status bytes" % ("NCCL" if world > 1 else "single rank"),
                      "oracle": "oracle/c (bccsp/sw gates + ecdsa.Verify steps on OpenSSL primitives); tail cross-checked with oracle/bccsp_sw.py"}
            assert parity["mask_equals_oracle"] and parity["status_equals_oracle"], "parity leg: GPU bitmask differs from the oracle: %r" % (parity,)
        sync_all()


    # ---- max over ranks ---------------------------------------------------------------------------------------
    times = torch.tensor([dev_ms, e2e_s * 1e3, wall * 1e3, gen_ms, key_register_ms, e2e_sync_s * 1e3, conc_ms, e2e_pageable_s * 1e3, nccl_ms, fill_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, wall_ms, gen_ms, key_register_ms, e2e_sync_ms, conc_ms, e2e_pageable_ms, nccl_ms, fill_ms = [float(x) for x in times.tolist()]

    if rank == 0:
        hbm_peak, peak_src, sm_max = _peaks()
        value = n_total * args.steps / (dev_ms * 1e-3)
        per_launch_s = dev_ms * 1e-3 / args.steps
        ach_gbs = B * ALG_BYTES_PER_VERIFY / per_launch_s / 1e9
        mac_peak = 148 * 4 * 16 * sm_max * 1e6                  # SURVEY 8(d): 148 SMs x 4 SMSP x 16 lanes/clk (IMAD, rt 2)
        wg, wq = pkg.binding.build_info()
        s_wb, s_nw, s_bytes = pkg.binding.Context.small_table_info()
        macs_cached = alg_macs_cached(wg, wq)
        n_gather = (256 + wg - 1) // wg + (256 + wq - 1) // wq
        ach_macs = B * macs_cached / per_launch_s
        gen_launch_s = gen_ms * 1e-3 / gsteps
        value_generic = n_total / gen_launch_s
        cores = best_thread_count(w)
        cpu_v, cpu_done, cpu_el = cpu_port_rate(w, cores)
        out = {
            "metric": METRIC, "value": value, "unit": "verifies/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32 limbs (256-bit modular integer)", "data": "synthetic",
            "config": {"workload": workload_string(B),
                       "batch_per_gpu": B, "global_batch": n_total,
                       "parallelism": ("batch split x%d + bitmask exchanged over peer memory (P2P stores from the verify kernel's epilogue, fabgpu_peer_mask_*)" % world)
                                      if (peer is not None and not main_nccl) else ("batch split x%d + NCCL all-gather of the bitmask" % world),
                       "collective": "p2p" if (peer is not None and not main_nccl) else "nccl",
                       "value_with_nccl_allgather": (n_total * args.steps / (nccl_ms * 1e-3)) if (nccl_ms and not main_nccl) else None,
                       "value_with_peer_memory_exchange": (n_total * args.steps / (nccl_ms * 1e-3)) if (nccl_ms and main_nccl) else None,
                       "collective_note": peer_note,
                       "timing": "per-step CUDA events on the launch stream, summed; steps back to back over %d rotating input buffers (%.0f MB > the 126 MB L2); "
                                 "the window tables the kernel gathers from (%.1f GB) are far larger than the L2 by themselves" % (
                                     ROT, ROT * B * 160 / 1e6, (((256 + wg - 1) // wg) * ((1 << wg) - 1) * 64 + KEYS * ((256 + wq - 1) // wq) * ((1 << wq) - 1) * 64) / 1e9),
                       "value_l2_fill_between_steps": n_total * args.steps / (fill_ms * 1e-3),
                       "value_l2_fill_note": "the same loop with a 256 MiB fill between steps (round 1's method): the fill leaves the L2 full of dirty lines whose write-back "
                                             "competes with the next launch's table gathers",
                       "wall_ms": wall_ms, "rank0_numa_pinning": numa},
            "e2e": {"value": n_total * e2e_steps / (e2e_ms * 1e-3), "unit": "verifies/s", "h2d_bytes_per_step": e2e_h2d * world, "d2h_bytes_per_step": e2e_d2h * world,
                    "api": "fabgpu_bccsp_verify_batch_inplace_async + _wait over the context's %d slots, that many batches in flight (raw DER signatures + digests + keys in the library's PINNED host buffers -> status bytes in host memory)" % pkg.binding.SLOTS,
                    "pageable_value": n_total * e2e_steps / (e2e_pageable_ms * 1e-3),
                    "pageable_api": "fabgpu_bccsp_verify_batch_async: the same pipeline fed from ordinary (pageable) host arrays; the library's staging threads copy them into the pinned buffers first",
                    "pageable_repetitions_verifies_per_s": [n_total * e2e_steps / t for t in e2e_reps_pageable],
                    "mixed_value_rank0": B * e2e_mixed_steps / e2e_mixed_s,
                    "mixed_what": "same pipeline (pageable arrays), per GPU: half of the %d signatures from the %d identities with window tables, half from %d identities that sign 8 times each "
                                  "(they earn SMALL tables once 32 of their signatures have been seen, i.e. during the warm-up calls; before the small tier they stayed on the generic kernel); rank 0's rate" % (B, hot, cold),
                    "steps": e2e_steps, "repetitions_verifies_per_s": [n_total * e2e_steps / t for t in e2e_reps], "reported": "median repetition (max over ranks)",
                    "sync_value": n_total * e2e_steps / (e2e_sync_ms * 1e-3), "sync_api": "fabgpu_bccsp_verify_batch, one blocking call per step",
                    "last_call_phases_us": {"key_lookup": e2e_phases[0], "host_staging_copy": e2e_phases[1], "h2d_gate_verify_status_d2h": e2e_phases[2], "status_copy": e2e_phases[3]},
                    "gates": "on the device (bccsp_gate_kernel); FABGPU_BCCSP_HOST_GATES=1 selects the host-thread gates"},
            "gpu_launches": int(launches),
            "value_concurrent": {"value": n_total * csteps / (conc_ms * 1e-3), "unit": "verifies/s", "steps": csteps,
                                 "what": "same kernel, device-resident inputs, %d batches in flight on %d streams, no L2 flush: the regime of the pipelined e2e call "
                                         "(a single 64k launch fills 512 of 592 resident CTA slots)" % (pkg.binding.SLOTS, pkg.binding.SLOTS)},
            "value_generic": value_generic,
            "value_small": (B * ssteps / (small_ms * 1e-3)) if small_ms else None,
            "small": {"what": "ecdsa_verify_small_kernel, rank 0: %d signatures from %d keys that own a SMALL table (%d windows of signed %d-bit digits, %d KiB per key): "
                              "%d + %d mixed additions per signature, no doublings; device-resident, L2 flushed between steps" % (
                                  B, small_keys, s_nw, s_wb, s_bytes // 1024, (256 + wg - 1) // wg, s_nw),
                      "ms_per_step": (small_ms / ssteps) if small_ms else None, "steps": ssteps,
                      "register_and_first_batch_ms": small_register_ms if small_ms else None, "tables": ctx.key_table_stats()},
            "generic": {"what": "ecdsa_verify_kernel: no per-key table (first sight of a key); 255 doublings + 52 additions per signature",
                        "ms_per_step": gen_ms / gsteps, "steps": gsteps},
            "key_tables": {"keys": KEYS, "register_ms_once": key_register_ms,
                           "what": "fabgpu_keys_register builds a %d-bit window table (%.1f MiB) per public key -- what KeyImport does once per identity" % (wq, ((256 + wq - 1) // wq) * ((1 << wq) - 1) * 64 / 2**20)},
            "roofline": {"bound": "hbm", "achieved": ach_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": ach_gbs / hbm_peak,
                         "traffic": (NCU_DRAM_BYTES_PER_LAUNCH_64K if B == 65536 else None),
                         "traffic_note": "dram read+write of one launch at batch 65536 from profiles/r2_final_cached_ncu_summary.txt; it exceeds the "
                                         "algorithmic 10.5 MB because the kernel gathers %d table points (64 B each) per signature from HBM-resident "
                                         "window tables (%.1f GB for G, %.0f MiB per key) by design -- that is what replaces 255 doublings" % (
                                             n_gather, ((256 + wg - 1) // wg) * ((1 << wg) - 1) * 64 / 1e9, ((256 + wq - 1) // wq) * ((1 << wq) - 1) * 64 / 2**20),
                         "peak_source": peak_src, "kernel": "ecdsa_verify_cached_kernel",
                         "note": "integer-issue bound, not HBM bound: see roofline_int"},
            "roofline_int": {"bound": "int32 mac (fma pipe)", "kernel": "ecdsa_verify_cached_kernel", "achieved": ach_macs / 1e12,
                             "peak": mac_peak / 1e12, "unit": "TMAC/s", "frac": ach_macs / mac_peak,
                             "macs_per_verify": macs_cached,
                             "binding_unit": {"name": "fmaheavy pipe (IMAD / IMAD.WIDE)", "busy_frac_of_elapsed_ncu": NCU_FMAHEAVY_BUSY,
                                              "note": "the multiplier's carry-chained wide MAC issues at 31 /clk/SM, half the plain IMAD.WIDE rate "
                                                      "(profiles/microbench/int_pipe_b200.txt); averaged over all 148 SMs the pipe is 63 % busy over the launch "
                                                      "(72 % on the 128 SMs the 128 CTAs of 512 threads occupy), ALU pipe 45 % (52 %)"},
                             "peak_source": "model: 148 SM x 64 IMAD/clk x %d MHz" % int(sm_max),
                             "generic_kernel": {"achieved": B * ALG_MACS_PER_VERIFY / gen_launch_s / 1e12,
                                                "frac": B * ALG_MACS_PER_VERIFY / gen_launch_s / mac_peak, "macs_per_verify": ALG_MACS_PER_VERIFY}},
            "cpu_baseline": {"value": cpu_v, "unit": "verifies/s", "cores": cores, "kind": "port", "value_per_core": cpu_v / max(1, cores),
                             "sample": "%d signatures in %.1f s through oracle/c (bccsp/sw gates + ecdsa.Verify steps on OpenSSL BN/EC primitives), %d of %d logical CPUs (best of all/half/quarter)" % (cpu_done, cpu_el, cores, os.cpu_count() or 1)},
            "clocks": clocks,
            "block_replay": block_replay,
            "parity": parity,
        }
        if block_replay:
            block_replay["cpu_port_ms_per_block_est"] = 4 * args.block_txs / cpu_v * 1e3
        emit(out)
    if peer is not None:
        sync_all()
        peer.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=65536, help="signatures per GPU per step")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--block-txs", type=int, default=10000, help="transactions in the block-replay leg (configs[2])")
    ap.add_argument("--no-block", action="store_true", help="skip the block-replay leg")
    ap.add_argument("--no-parity", action="store_true", help="skip the (untimed) named-shape parity leg")
    ap.add_argument("--no-clients", action="store_true", help="skip the block-replay variant with 2 000 client identities")
    ap.add_argument("--collective", default="nccl", choices=["p2p", "nccl"], help="N > 1: how the bitmask is reassembled in the timed loop (the other way is timed beside it)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the validity bits of the last timed step to DIR/valid.npy (GPU arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm")
    # The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version line on the first
    # collective), so everything but the result goes to stderr: fd 1 is pointed at fd 2 for the duration of the run and the
    # JSON line is written to the saved descriptor.
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    global _RESULT_FD
    _RESULT_FD = saved
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


_RESULT_FD = None
DUMP_BYTES = 64 << 20


def dump_outputs(dirname, arrays):
    """Writes each array as DIR/<name>.npy in float32.  Past 64 MB in all, each keeps a fixed, seeded sample of its entries (in
    their original order), so runs with the same arguments still write the same sample."""
    os.makedirs(dirname, exist_ok=True)
    cap = (DUMP_BYTES // len(arrays) - 4096) // 4                        # entries per array; 4096 B leaves room for the .npy header
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float32).reshape(-1)
        if a.size > cap:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))]
        np.save(os.path.join(dirname, name + ".npy"), a)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(line.decode()); sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_RESULT_FD, line)


if __name__ == "__main__":
    main()
