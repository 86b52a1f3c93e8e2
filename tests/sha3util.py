"""Helpers for the tests of per-MSP signature hash families (SHA2 / SHA3): the oracle's block validator with each signature checked
over its signer's family, and the device block logic run on the host with the families installed."""
import ctypes
import hashlib
import os
import subprocess

import numpy as np

from oracle import bccsp_sw as o
from oracle import blockval as ob
from oracle import fast
from util import ROOT
import blockutil

_LIB = None


def lib():
    """tests/host_sim/libsha3_host.so: sha3.cuh + blockdev.cuh (through blockdev_host.cpp) built for the host."""
    global _LIB
    if _LIB is None:
        d = os.path.join(ROOT, "tests", "host_sim")
        so, src = os.path.join(d, "libsha3_host.so"), os.path.join(d, "sha3_host.cpp")
        csrc = os.path.join(ROOT, "fabric-mod_b200", "csrc")
        deps = [src, os.path.join(d, "blockdev_host.cpp"), os.path.join(csrc, "sha3.cuh"), os.path.join(csrc, "blockdev.cuh")]
        if not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(f) for f in deps):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, src])
        _LIB = ctypes.CDLL(so)
        _LIB.bd_new.restype = ctypes.c_void_p
    return _LIB


def host_sha3_segments(buf: bytes, jobs):
    """sha3_256_message (the per-job function of sha3_256_segments_kernel) on the host: jobs uint32[n,6] -> uint8[n,32]."""
    jobs = np.ascontiguousarray(jobs, np.uint32).reshape(-1, 6)
    b = np.zeros(len(buf) + 8, np.uint8)                     # slack: the block loader reads the aligned word past a range
    b[: len(buf)] = np.frombuffer(buf, np.uint8)
    out = np.zeros((jobs.shape[0], 32), np.uint8)
    lib().sha3_host_segments(blockutil._p(b), blockutil._p(jobs), jobs.shape[0], blockutil._p(out))
    return out


def digest(family, msg: bytes) -> bytes:
    return (hashlib.sha3_256 if family == "SHA3" else hashlib.sha256)(msg).digest()


def family_verify(identities, families):
    """identity.Verify with the signer's MSP family (msp/identities.go:169-196,216-224), as a `verify` hook of the oracle's block
    validator: the hook sees the signer's key, and every key here belongs to one MSP."""
    fam = {}
    for ser, mspid, xy, valid in identities:
        f = (families or {}).get(mspid, "SHA2")
        assert fam.setdefault(bytes(xy), f) == f, "one key in two MSPs of different families"

    def verify(xy, msg, sig):
        d = digest(fam.get(bytes(xy), "SHA2"), msg)
        st = fast.verify_batch(np.frombuffer(xy, np.uint8).reshape(1, 64), np.zeros(1, np.int32), np.frombuffer(d, np.uint8),
                               np.array([0, 32], np.uint32), np.frombuffer(sig, np.uint8) if sig else np.zeros(0, np.uint8),
                               np.array([0, len(sig)], np.uint32))
        return int(st[0]) == o.VALID
    return verify


def oracle_flags(blk, net, nodes, policies=None, families=None):
    """The oracle's flags for a device holding exactly net.msp_table, signatures checked over their signer's MSP family.  The tx id
    and the proposal hash stay SHA-256 (the oracle computes them so)."""
    ids = blockutil.identities_of(net)
    return ob.validate_block(blk, ids, net.channel, nodes, net.principals, verify=family_verify(ids + [(net.unknown.serialized, net.unknown.mspid,
                             net.unknown.xy, True)], families), policies=policies, known=[i[0] for i in ids])


def device_logic_flags(env_blob, env_off, identities, channel, nodes, principals, policies=None, families=None):
    """The device block logic (blockdev.cuh) run on the host with per-identity hash kinds from `families` ({mspid: "SHA2"|"SHA3"}).
    Each signature digest is computed with the kind resolve_job assigned to its job, not with the family known here.
    -> (flags, kinds, identities) with kinds / identities per signature job (identity -1: unused slot)."""
    from oracle import goasn1
    from util import pkg
    L = lib()
    idb, ido = blockutil._blob([bytes(i[0]) for i in identities])
    mb, mo = blockutil._blob([i[1].encode() for i in identities])
    keys = np.ascontiguousarray(np.frombuffer(b"".join(bytes(i[2]) for i in identities), np.uint8)).reshape(-1, 64)
    valid = np.array([1 if i[3] else 0 for i in identities], np.uint8)
    hash_kind = np.array([1 if (families or {}).get(i[1]) == "SHA3" else 0 for i in identities], np.uint8)
    nodes = np.ascontiguousarray(nodes, np.int32)
    pbb, pbo = blockutil._blob([p.encode() for p in principals])
    h = ctypes.c_void_p(L.bd_new(blockutil._p(idb), blockutil._p(ido), blockutil._p(mb), blockutil._p(mo), blockutil._p(valid), len(identities),
                                 blockutil._p(nodes), nodes.shape[0], blockutil._p(pbb), blockutil._p(pbo), len(principals), channel.encode()))
    groups = np.ascontiguousarray(pkg().binding.identity_groups(identities), np.int32)
    L.bd_groups(h, blockutil._p(groups), len(identities))
    if policies:
        names = sorted(policies)
        nb, no = blockutil._blob([n.encode() for n in names])
        roots = np.array([policies[n] for n in names], np.int32)
        L.bd_namespaces(h, blockutil._p(nb), blockutil._p(no), blockutil._p(roots), len(names))
    blob = np.frombuffer(env_blob, np.uint8) if len(env_blob) else np.zeros(1, np.uint8)
    env_off = np.ascontiguousarray(env_off, np.uint32)
    T = env_off.shape[0] - 1
    J = T + L.bd_plan_families(h, blockutil._p(blob), blockutil._p(env_off), T, blockutil._p(hash_kind))
    ident, gok = ctypes.c_int(0), ctypes.c_int(0)
    r = (ctypes.c_uint8 * 32)(); s = (ctypes.c_uint8 * 32)(); segs = (ctypes.c_uint32 * 12)()
    key_idx, digs, sigs, live, kinds, idents = [], [], [], [], [], []

    def msg(sg, base=0):
        return b"".join(env_blob[sg[base + k]: sg[base + k] + sg[base + 3 + k]] for k in range(3))
    for j in range(J):
        L.bd_job(h, j, ctypes.byref(ident), ctypes.byref(gok), r, s, segs)
        kinds.append(L.bd_job_kind(h, j))
        idents.append(ident.value)
        if ident.value < 0 or not gok.value:
            continue
        live.append(j)
        key_idx.append(ident.value)
        digs.append(digest("SHA3" if kinds[-1] == 1 else "SHA2", msg(segs)))
        sigs.append(goasn1.marshal_ecdsa_signature(int.from_bytes(bytes(r), "big"), int.from_bytes(bytes(s), "big")))
    sig_ok = np.zeros(max(J, 1), np.uint8)
    if live:
        soff = np.zeros(len(live) + 1, np.uint32); soff[1:] = np.cumsum([len(x) for x in sigs])
        st = fast.verify_batch(keys, np.array(key_idx, np.int32), np.frombuffer(b"".join(digs), np.uint8), (np.arange(len(live) + 1) * 32).astype(np.uint32),
                               np.frombuffer(b"".join(sigs), np.uint8), soff, nthreads=4)
        sig_ok[np.array(live)] = (st == o.VALID)
    chk = np.zeros((max(T, 1), 2, 32), np.uint8)
    for t in range(T):                                      # tx id and proposal hash: SHA-256 whatever the family
        L.bd_check(h, t, segs)
        chk[t, 0] = np.frombuffer(hashlib.sha256(msg(segs, 0)).digest(), np.uint8)
        chk[t, 1] = np.frombuffer(hashlib.sha256(msg(segs, 6)).digest(), np.uint8)
    flags = np.full(max(T, 1), 254, np.uint8)
    L.bd_decide(h, blockutil._p(sig_ok), blockutil._p(chk), blockutil._p(flags))
    L.bd_forget_kinds(h)
    L.bd_free(h)
    return flags[:T], np.array(kinds, np.int32), np.array(idents, np.int32)
