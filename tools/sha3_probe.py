"""SHA3 signature hash family: what it costs on the device (development tool, one GPU run):
    python tools/sha3_probe.py [--out FILE.json] [--block-txs 10000]
  * the card's name and power limit;
  * sha3_256_segments_kernel against sha256_segments_kernel on the creator payloads of the configs[2] block (10 000 x ~4.6 KB):
    kernel durations from torch.profiler's CUDA activity records, achieved GB/s over the payload bytes;
  * the configs[2] block replay (10 k txs x 3 endorsements, 3-of-4 policy) with every org on SHA2, every org on SHA3, and two of each:
    one blocking call per block and three blocks in flight, device stage times (FABGPU_BLOCK_EVENTS=1) and launches per block.
Prints one JSON document (and writes it to --out)."""
import argparse
import hashlib
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pkg = importlib.import_module("fabric-mod_b200")
from tools import blockgen  # noqa: E402

CONFIGS = {"all_sha2": {}, "all_sha3": {"Org%dMSP" % i: "SHA3" for i in range(1, 5)},
           "two_and_two": {"Org1MSP": "SHA3", "Org3MSP": "SHA3", "Org2MSP": "SHA2", "Org4MSP": "SHA2"}}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "nvidia-smi unavailable"


def payload_jobs(env_blob, env_off):
    """Creator-signature messages: the Payload field (Envelope field 1) of every envelope, as (off, 0, 0, len, 0, 0) jobs."""
    jobs = []
    for t in range(len(env_off) - 1):
        p = int(env_off[t])
        assert env_blob[p] == 0x0A                                 # field 1, length-delimited
        ln, sh, q = 0, 0, p + 1
        while True:
            c = env_blob[q]; q += 1
            ln |= (c & 0x7F) << sh; sh += 7
            if not c & 0x80:
                break
        jobs.append((q, 0, 0, ln, 0, 0))
    return np.array(jobs, np.uint32)


def kernel_times(ctx, buf, jobs, reps):
    """Median kernel duration (us) of each SHA kernel over `reps` calls, from the profiler's CUDA kernel records."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    for _ in range(3):                                             # module load, allocator
        ctx.sha256_segments(buf, jobs); ctx.sha3_256_segments(buf, jobs)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            ctx.sha256_segments(buf, jobs)
            ctx.sha3_256_segments(buf, jobs)
        torch.cuda.synchronize()
    durs = {"sha256_segments_kernel": [], "sha3_256_segments_kernel": []}
    for ev in prof.events():
        for k in durs:
            if k in ev.name and ev.device_type == torch.autograd.DeviceType.CUDA:
                durs[k].append(ev.device_time if hasattr(ev, "device_time") else ev.cuda_time)
    return {k: float(np.median(v)) if v else None for k, v in durs.items()}, {k: len(v) for k, v in durs.items()}


def block_leg(ctx, families, n_tx, slots):
    net = blockgen.Network(hash_families=families or None)
    blk, info = blockgen.build_block(net, n_tx, 3, {}, seed=17)
    ctx.msp_configure([(i.serialized, i.mspid, i.xy, i.valid) for i in net.msp_table], net.policy_n_of(3), net.principals, net.channel,
                      hash_families=families or None)
    eblob, eoff = info["env_blob"], info["env_off"]
    bufs = []
    for k in range(slots):
        b = ctx.block_buffer(len(eblob), slot=k)
        b[:] = np.frombuffer(eblob, np.uint8)
        bufs.append(b)
    os.environ["FABGPU_BLOCK_EVENTS"] = "1"
    for _ in range(3):
        fl = ctx.validate_envelopes(bufs[0], eoff)
    assert fl.shape[0] == n_tx and not fl.any(), "not every transaction flag is VALID"
    n0 = ctx.launch_count()
    ctx.validate_envelopes(bufs[0], eoff)
    launches = ctx.launch_count() - n0
    reps, stages = 10, []
    t0 = time.perf_counter()
    for _ in range(reps):
        ctx.validate_envelopes(bufs[0], eoff)
        stages.append(ctx.block_timing())
    ms_single = (time.perf_counter() - t0) / reps * 1e3
    st = np.median(np.array(stages), axis=0)
    os.environ["FABGPU_BLOCK_EVENTS"] = "0"
    for k in range(slots):
        ctx.validate_envelopes_async(k, bufs[k], eoff)
        assert not ctx.validate_wait(k, n_tx).any()
    reps2, fls = 30, []
    t0 = time.perf_counter()
    for k in range(reps2):
        if k >= slots:
            fls.append(ctx.validate_wait(k % slots, n_tx))
        ctx.validate_envelopes_async(k % slots, bufs[k % slots], eoff)
    for k in range(max(0, reps2 - slots), reps2):
        fls.append(ctx.validate_wait(k % slots, n_tx))
    ms_flight = (time.perf_counter() - t0) / reps2 * 1e3
    assert len(fls) == reps2 and not any(f.any() for f in fls)
    return {"families": families or "SHA2 (no fabgpu_msp_hash_families call)", "launches_per_block": int(launches),
            "single_call_ms_per_block": ms_single, "in_flight_ms_per_block": ms_flight, "blocks_in_flight": slots,
            "device_stage_us_median_of_%d" % reps: {"h2d_walk_creator_resolve_and_hash": st[5], "endorsement_resolve_and_hash": st[7],
                                                     "verify_kernel": st[8], "block_decide_kernel": st[9]}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--block-txs", type=int, default=10000)
    ap.add_argument("--reps", type=int, default=20, help="profiled calls per SHA kernel")
    args = ap.parse_args()
    ctx = pkg.binding.Context(max_batch=65536)
    res = {"card": card(), "block_txs": args.block_txs}
    net = blockgen.Network()
    _, info = blockgen.build_block(net, args.block_txs, 3, {}, seed=17)
    buf = np.frombuffer(info["env_blob"], np.uint8)
    jobs = payload_jobs(info["env_blob"], info["env_off"])
    nbytes = int(jobs[:, 3].sum())
    assert bytes(ctx.sha3_256_segments(buf, jobs[:1])[0]) == hashlib.sha3_256(bytes(buf[jobs[0, 0]: jobs[0, 0] + jobs[0, 3]])).digest()
    us, counts = kernel_times(ctx, buf, jobs, args.reps)
    res["sha_kernels"] = {
        "workload": "%d creator payloads of the configs[2] block, %d bytes in all (mean %.0f B), one thread per message" % (jobs.shape[0], nbytes, nbytes / jobs.shape[0]),
        "timing": "median kernel duration of %d calls each, torch.profiler CUDA kernel records" % args.reps,
        "l2_state": "warm: each call copies the %.0f MB buffer in (H2D) right before its kernel, and it fits the 126 MB L2" % (buf.shape[0] / 1e6),
        "kernel_us": us, "records": counts,
        "GB_per_s": {k: (nbytes / (v * 1e-6) / 1e9 if v else None) for k, v in us.items()},
        "sha3_over_sha256": (us["sha3_256_segments_kernel"] / us["sha256_segments_kernel"]) if all(us.values()) else None}
    print(json.dumps(res["sha_kernels"]), flush=True)
    res["block_replay"] = {}
    for name, fam in CONFIGS.items():
        res["block_replay"][name] = block_leg(ctx, fam, args.block_txs, pkg.binding.SLOTS)
        print(name, json.dumps(res["block_replay"][name]), flush=True)
    ctx.close()
    doc = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(doc + "\n")
    print(doc)


if __name__ == "__main__":
    main()
