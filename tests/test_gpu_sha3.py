"""GPU: device SHA3-256 against hashlib, and the block pre-pass with per-MSP signature hash families (fabgpu_msp_hash_families)
against the oracle's validator with each signature checked over its signer's family."""
import ctypes
import hashlib
import random

import numpy as np
import pytest

from oracle import blockval as ob
from tools import blockgen
from util import pkg
import blockutil
import sha3util

pytestmark = pytest.mark.gpu

MIXED = {"Org1MSP": "SHA3", "Org3MSP": "SHA3", "Org2MSP": "SHA2", "Org4MSP": "SHA2"}
ALL_SHA3 = {"Org%dMSP" % i: "SHA3" for i in range(1, 5)}


@pytest.fixture(scope="module")
def ctx():
    c = pkg().binding.Context(max_batch=8192)
    yield c
    c.close()


def test_sha3_256_segments_vs_hashlib(ctx):
    rnd = random.Random(9)
    buf = bytes(rnd.getrandbits(8) for _ in range(20000))
    jobs, exp = [], []
    lens = [0, 1, 3, 4, 5, 31, 32, 33, 54, 55, 56, 57, 63, 64, 65, 119, 120, 127, 128, 129, 135, 136, 137, 271, 272, 273, 1000, 4097]
    for la in lens:
        for lb in (0, 1, 7, 64, 136, 333):
            for lc in (0, 5):
                oa, ob_, oc = rnd.randrange(0, 9000), rnd.randrange(0, 9000), rnd.randrange(0, 9000)
                jobs.append((oa, ob_, oc, la, lb, lc))
                exp.append(hashlib.sha3_256(buf[oa:oa + la] + buf[ob_:ob_ + lb] + buf[oc:oc + lc]).digest())
    got = ctx.sha3_256_segments(buf, np.array(jobs, np.uint32))
    assert [bytes(g) for g in got] == exp
    assert bytes(ctx.sha3_256_segments(b"abc", np.array([(0, 0, 0, 3, 0, 0)], np.uint32))[0]).hex() == \
        "3a985da74fe225b2045c172d6bd390bd855f086e3e9d525b46bfe24511431532"


def test_mixed_families_fault_classes_match_oracle(ctx):
    """Org1 / Org3 sign with SHA3-256, Org2 / Org4 with SHA-256: every fault class with per-namespace policies, through both entry
    points and through two slots in flight."""
    net = blockgen.Network(hash_families=MIXED)
    n = 3 * len(blockgen.FAULTS) + 4
    faults = blockutil.fault_map(n)
    blk, info = blockgen.build_block(net, n, 3, faults, seed=11)
    nodes, pol = net.policies_for(3)
    exp = sha3util.oracle_flags(blk, net, nodes, pol, MIXED)
    assert len(set(exp.tolist())) >= 10 and int((exp == ob.VALID).sum()) > n // 2
    ctx.msp_configure(blockutil.identities_of(net), nodes, net.principals, net.channel, policies=pol, hash_families=MIXED)
    assert ctx.validate_block(blk).tolist() == exp.tolist()
    assert ctx.validate_envelopes(info["env_blob"], info["env_off"]).tolist() == exp.tolist()
    rnd = random.Random(41)
    f2 = {t: rnd.choice(blockgen.FAULTS) for t in rnd.sample(range(1, 500), 60)}
    blk2, info2 = blockgen.build_block(net, 500, 3, f2, seed=42)
    exp2 = sha3util.oracle_flags(blk2, net, nodes, pol, MIXED)
    for _ in range(2):
        ctx.validate_envelopes_async(0, np.frombuffer(info["env_blob"], np.uint8), info["env_off"])
        ctx.validate_block_async(1, blk2)
        assert ctx.validate_wait(1, 500).tolist() == exp2.tolist()
        assert ctx.validate_wait(0, n).tolist() == exp.tolist()


def test_config3_block_all_sha3(ctx):
    # BASELINE.json configs[2] shape with every org on SHA3: 10 k txs x 3 endorsements, every flag VALID
    net = blockgen.Network(hash_families=ALL_SHA3)
    blk, info = blockgen.build_block(net, 10000, 3, {}, seed=17)
    ctx.msp_configure(blockutil.identities_of(net), net.policy_n_of(3), net.principals, net.channel, hash_families=ALL_SHA3)
    pinned = ctx.block_buffer(len(blk))
    pinned[:] = np.frombuffer(blk, np.uint8)
    got = ctx.validate_block(pinned)
    assert got.shape[0] == 10000 and (got == ob.VALID).all()
    # one flipped byte inside one endorsement signature flips exactly that transaction
    b = bytearray(blk)
    marker = net.peers[1].serialized
    pos = blk.index(marker, len(blk) // 2) + len(marker) + 10
    b[pos] ^= 0x20
    got2 = ctx.validate_block(bytes(b))
    exp2 = sha3util.oracle_flags(bytes(b), net, net.policy_n_of(3), None, ALL_SHA3)
    assert got2.tolist() == exp2.tolist() and int((got2 != ob.VALID).sum()) == 1


def _launches_per_block(c, blob, off):
    n0 = c.launch_count()
    c.validate_envelopes(blob, off)
    return c.launch_count() - n0


def test_launch_count():
    """A table with no SHA3 identity issues the launches of a SHA-256-only table; a SHA3 identity adds one SHA3-256 launch beside each
    of the two signature-message SHA-256 launches."""
    c = pkg().binding.Context(max_batch=4096)
    net = blockgen.Network(hash_families=MIXED)
    blk, info = blockgen.build_block(net, 300, 3, {}, seed=3)
    blob, off = np.frombuffer(info["env_blob"], np.uint8), info["env_off"]
    ids, nodes = blockutil.identities_of(net), net.policy_n_of(3)
    c.msp_configure(ids, nodes, net.principals, net.channel)
    base = _launches_per_block(c, blob, off)
    assert _launches_per_block(c, blob, off) == base
    c.msp_configure(ids, nodes, net.principals, net.channel, hash_families={"Org1MSP": "SHA2", "Org2MSP": "SHA2"})
    assert _launches_per_block(c, blob, off) == base
    c.msp_configure(ids, nodes, net.principals, net.channel, hash_families=MIXED)
    assert _launches_per_block(c, blob, off) == base + 2
    assert (c.validate_envelopes(blob, off) == ob.VALID).all()
    c.msp_hash_families({})                                                    # n_msps = 0: all-SHA2 again
    assert _launches_per_block(c, blob, off) == base
    c.close()


def test_hash_family_arguments_and_reset(ctx):
    binding = pkg().binding
    net = blockgen.Network(hash_families=MIXED)
    blk, _ = blockgen.build_block(net, 40, 3, {}, seed=9)
    ids, nodes = blockutil.identities_of(net), net.policy_n_of(3)
    ctx.msp_configure(ids, nodes, net.principals, net.channel, hash_families=MIXED)
    assert (ctx.validate_block(blk) == ob.VALID).all()

    def raw(names, fams):
        off = np.zeros(len(names) + 1, np.uint32)
        off[1:] = np.cumsum([len(n) for n in names])
        blob = np.frombuffer(b"".join(n.encode() for n in names) or b"\x00", np.uint8).copy()
        fam = np.array(fams or [0], np.uint8)
        return binding.lib().fabgpu_msp_hash_families(ctx._h, blob.ctypes.data_as(ctypes.c_void_p), off.ctypes.data_as(ctypes.c_void_p),
                                                       fam.ctypes.data_as(ctypes.c_void_p), ctypes.c_int(len(names)))
    assert raw(["Org1MSP"], [2]) == binding.E_ARG and "neither" in ctx.last_error()
    assert raw(["NoSuchMSP"], [1]) == binding.E_ARG and "NoSuchMSP" in ctx.last_error()
    assert raw(["Org1MSP", "Org1MSP"], [1, 0]) == binding.E_ARG and "two hash families" in ctx.last_error()
    with pytest.raises(binding.FabGpuError):
        ctx.msp_hash_families({"NoSuchMSP": "SHA3"})
    with pytest.raises(ValueError):
        ctx.msp_hash_families({"Org1MSP": "SHA-3"})
    # a refused call leaves the table as it was; one MSP listed twice with the same family is accepted
    assert (ctx.validate_block(blk) == ob.VALID).all()
    assert raw(["Org1MSP", "Org1MSP", "Org3MSP"], [1, 1, 1]) == binding.OK
    assert (ctx.validate_block(blk) == ob.VALID).all()
    # a second fabgpu_msp_configure without families resets every identity to SHA2: the SHA3 signatures no longer verify
    ctx.msp_configure(ids, nodes, net.principals, net.channel)
    exp_sha2 = ob.validate_block(blk, ids, net.channel, nodes, net.principals, known=[i[0] for i in ids])
    got = ctx.validate_block(blk)
    assert got.tolist() == exp_sha2.tolist() and not (got == ob.VALID).any()
