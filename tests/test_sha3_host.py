"""SHA3 signature hash family on the CPU: the SHA3-256 code of sha3.cuh built for the host against hashlib, and the device block logic
(blockdev.cuh) with per-MSP hash families against the oracle's validator with each signature checked over its signer's family."""
import hashlib
import random

from oracle import blockval as ob
from tools import blockgen
from tools import fabricpb as pb
import blockutil
import sha3util

FAMILIES = {"Org1MSP": "SHA3", "Org3MSP": "SHA3", "Org2MSP": "SHA2", "Org4MSP": "SHA2"}


def _check(buf, jobs):
    got = sha3util.host_sha3_segments(buf, jobs)
    exp = [hashlib.sha3_256(b"".join(buf[o:o + n] for o, n in zip(j[:3], j[3:]))).digest() for j in jobs]
    assert [bytes(g) for g in got] == exp


def test_fips202_examples():
    got = sha3util.host_sha3_segments(b"abc", [(0, 0, 0, 0, 0, 0), (0, 0, 0, 3, 0, 0)])
    assert bytes(got[0]).hex() == "a7ffc6f8bf1ed76651c14756a061d662f580ff4de43b49fa82d80a4b80f8434a"
    assert bytes(got[1]).hex() == "3a985da74fe225b2045c172d6bd390bd855f086e3e9d525b46bfe24511431532"


def test_every_length_0_to_600():
    rnd = random.Random(1)
    buf = bytes(rnd.getrandbits(8) for _ in range(2000))
    _check(buf, [(n % 7 + 3 * (n % 3), 0, 0, n, 0, 0) for n in range(601)])      # the start offset cycles through every alignment


def test_rate_edges_and_long_message():
    rnd = random.Random(2)
    buf = bytes(rnd.getrandbits(8) for _ in range(9000))
    jobs = [(off, 0, 0, n, 0, 0) for n in (135, 136, 137, 271, 272, 273, 4097) for off in (0, 1, 2, 3, 1001)]
    _check(buf, jobs)


def test_three_ranges_around_block_edges():
    rnd = random.Random(3)
    buf = bytes(rnd.getrandbits(8) for _ in range(6000))
    jobs = []
    for la in (0, 1, 135, 136, 137, 271, 272, 273):
        for lb in (0, 1, 134, 135, 136, 137, 272):
            for lc in (0, 1, 135, 136, 137):
                jobs.append((rnd.randrange(0, 2000), rnd.randrange(0, 2000), rnd.randrange(0, 2000), la, lb, lc))
    _check(buf, jobs)


def _mixed_block():
    net = blockgen.Network(hash_families=FAMILIES)
    n = 3 * len(blockgen.FAULTS) + 4
    faults = blockutil.fault_map(n)
    assert set(faults.values()) == set(blockgen.FAULTS)
    blk, info = blockgen.build_block(net, n, 3, faults, seed=11, nthreads=2)
    return net, faults, blk, info


def test_mixed_families_fault_classes_match_oracle():
    net, faults, blk, info = _mixed_block()
    ids = blockutil.identities_of(net)
    nodes, pol = net.policies_for(3)
    exp = sha3util.oracle_flags(blk, net, nodes, pol, FAMILIES)
    got, kinds, idents = sha3util.device_logic_flags(info["env_blob"], info["env_off"], ids, net.channel, nodes, net.principals, pol, FAMILIES)
    assert got.tolist() == exp.tolist()
    assert len(set(exp.tolist())) >= 10
    byf = {f: int(exp[t]) for t, f in faults.items()}
    # the tx-id and proposal-hash checks stay SHA-256: a SHA3 creator's transaction passes them, the faults are still caught
    assert byf["bad_txid"] == ob.BAD_PROPOSAL_TXID and byf["bad_proposal_hash"] == ob.INVALID_ENDORSER_TRANSACTION
    assert byf["dup_txid"] == ob.DUPLICATE_TXID and byf["bad_creator_sig"] == ob.BAD_CREATOR_SIGNATURE
    assert byf["bad_endorsement_sig"] == ob.ENDORSEMENT_POLICY_FAILURE
    T = len(exp)
    valid = [t for t in range(T) if exp[t] == ob.VALID]
    assert len(valid) > T // 2 and all(kinds[t] == 1 for t in valid)          # the client is an Org1MSP (SHA3) identity
    # every job's kind is its signer's MSP family: creator jobs [0, T), endorsement jobs after
    for j, (k, i) in enumerate(zip(kinds.tolist(), idents.tolist())):
        want = 0 if i < 0 else (1 if FAMILIES[ids[i][1]] == "SHA3" else 0)
        assert k == want, (j, k, i)
    end_kinds = kinds[T:][idents[T:] >= 0]
    assert (end_kinds == 1).sum() > 10 and (end_kinds == 0).sum() > 10


def test_sha3_block_without_families_is_sha2():
    """The table is what makes the difference: the same SHA3-signed block on a table with no families gives the flags the oracle
    gives when every MSP is SHA2 (most signatures fail), and the existing SHA-256-only host run agrees."""
    net, faults, blk, info = _mixed_block()
    ids = blockutil.identities_of(net)
    nodes, pol = net.policies_for(3)
    exp_sha2 = ob.validate_block(blk, ids, net.channel, nodes, net.principals, policies=pol, known=[i[0] for i in ids])
    got, kinds, _ = sha3util.device_logic_flags(info["env_blob"], info["env_off"], ids, net.channel, nodes, net.principals, pol, None)
    assert got.tolist() == exp_sha2.tolist()
    assert (kinds == 0).all()
    assert blockutil.device_logic_flags(info["env_blob"], info["env_off"], ids, net.channel, nodes, net.principals, pol).tolist() == exp_sha2.tolist()
    assert int((exp_sha2 == ob.VALID).sum()) == 0 and int((exp_sha2 == ob.BAD_CREATOR_SIGNATURE).sum()) > len(exp_sha2) // 2
    assert got.tolist() != sha3util.oracle_flags(blk, net, nodes, pol, FAMILIES).tolist()


def test_blockgen_without_families_is_unchanged():
    a, _ = blockgen.build_block(blockgen.Network(), 12, 3, {3: "bad_txid"}, seed=5, nthreads=2)
    b, _ = blockgen.build_block(blockgen.Network(hash_families=None), 12, 3, {3: "bad_txid"}, seed=5, nthreads=2)
    c, _ = blockgen.build_block(blockgen.Network(hash_families={"Org2MSP": "SHA2"}), 12, 3, {3: "bad_txid"}, seed=5, nthreads=2)
    d, _ = blockgen.build_block(blockgen.Network(hash_families={"Org2MSP": "SHA3"}), 12, 3, {3: "bad_txid"}, seed=5, nthreads=2)
    assert a == b == c and a != d
    envs = pb.parse(pb.parse(a, ob.S_BLOCK)["data"], ob.S_BLOCKDATA)["data"]
    assert len(envs) == 12
