"""Synthetic Fabric blocks for BASELINE.json configs[2] (block-validation replay: T transactions x E endorsements).

Builds what `protoutil.CreateSignedTx` + an orderer would produce (reference protoutil/txutils.go:134-295):
  * clients sign the marshalled Payload (txutils.go:223-236); endorsers sign  ProposalResponsePayload || endorser
    (txutils.go:266-275); tx id = hex(SHA-256(nonce || creator)) (proputils.go:357-364);
    proposal hash = SHA-256(channel_header || signature_header || chaincode_proposal_payload) (txutils.go:431-448);
  * identities are msp.SerializedIdentity{mspid, PEM certificate}; certificates are real self-signed P-256 X.509
    certificates when `cryptography` is importable, otherwise opaque PEM-shaped blobs of the same size (the validator
    only ever looks identities up in the MSP's table, as msp/cache does in steady state).
Not the oracle and not product code.  Faults can be injected per transaction to exercise every validation code on the
signature path."""
import hashlib
import os

import numpy as np

from . import fabricpb as pb
from . import workload

FAULTS = ("bad_creator_sig", "bad_endorsement_sig", "dup_endorser", "unknown_endorser", "unknown_creator", "bad_txid", "dup_txid",
          "bad_proposal_hash", "bad_payload", "wrong_channel", "two_bad_endorsements", "invalid_creator_cert", "high_s_endorsement",
          "empty_nonce", "config_update_type", "nonzero_epoch", "no_signature",
          # the plugin dispatcher's checks and per-chaincode policies (plugindispatcher/dispatcher.go:102-221)
          "bad_header_extension", "no_prp_extension", "bad_rwset", "cc_name_mismatch", "empty_cc_version", "event_wrong_cc", "dup_namespace",
          "writes_strict_namespace", "reads_strict_namespace", "writes_unknown_namespace", "same_cert_two_encodings", "many_endorsements")

CHAINCODE = "mycc"                 # the chaincode every synthetic transaction invokes
STRICT_NAMESPACE = "strictcc"      # a second chaincode whose policy wants one endorsement more than transactions carry
UNKNOWN_NAMESPACE = "ghostcc"      # a namespace without a chaincode definition in the table given to the device


def chaincode_id(name: str, version: str = "") -> bytes:
    return pb.f_bytes(2, name.encode()) + (pb.f_bytes(3, version.encode()) if version else b"")


def kv_rwset(n_reads=1, n_writes=1, tag=b"k") -> bytes:
    """kvrwset.KVRWSet{reads=1, writes=3}: KVRead{key=1}, KVWrite{key=1, value=3}."""
    out = b""
    for i in range(n_reads):
        out += pb.f_bytes(1, pb.f_bytes(1, tag + b"-r%d" % i))
    for i in range(n_writes):
        out += pb.f_bytes(3, pb.f_bytes(1, tag + b"-w%d" % i) + pb.f_bytes(3, b"value-%d" % i))
    return out


def tx_rwset(namespaces) -> bytes:
    """rwset.TxReadWriteSet{data_model=1 (KV = 0), ns_rwset=2}; namespaces: list of (name, n_reads, n_writes)."""
    return b"".join(pb.f_bytes(2, pb.f_bytes(1, name.encode()) + pb.f_bytes(2, kv_rwset(nr, nw, name.encode()))) for name, nr, nw in namespaces)


class Identity:
    def __init__(self, mspid, priv_index, xy, cert_pem, valid=True):
        self.mspid, self.priv_index, self.xy, self.cert_pem, self.valid = mspid, priv_index, xy, cert_pem, valid
        self.serialized = pb.serialized_identity(mspid, cert_pem)


def _pem_blob(tag: bytes, n=780) -> bytes:
    import base64
    raw = hashlib.sha256(tag).digest() * (n // 32 + 1)
    b64 = base64.encodebytes(raw[: n * 3 // 4])
    return b"-----BEGIN CERTIFICATE-----\n" + b64 + b"-----END CERTIFICATE-----\n"


def _der_sig(r: int, s: int) -> bytes:
    def der_int(v):
        b = v.to_bytes((v.bit_length() + 8) // 8 or 1, "big")
        return b"\x02" + bytes([len(b)]) + b
    body = der_int(r) + der_int(s)
    return b"\x30" + bytes([len(body)]) + body


class Network:
    """n_orgs endorsing orgs (one peer identity each) + n_clients client identities + one identity that is NOT in the
    MSP table ('unknown') and one whose certificate the MSP considers invalid.
    hash_families: {mspid: "SHA2" | "SHA3"}, the SignatureHashFamily of those MSPs (others SHA2): every signature is made over the
    digest of its signer's family, as identity.Sign does (msp/identities.go:216-224,251-280).  None: SHA-256 throughout."""

    def __init__(self, n_orgs=4, n_clients=1, seed=0xB10C, channel="fabgpu-channel", hash_families=None):
        self.channel = channel
        self.hash_families = dict(hash_families or {})
        self.n_orgs = n_orgs
        K = n_orgs + n_clients + 2
        L = workload.lib()
        import ctypes
        self.priv = np.zeros((K, 32), np.uint8)
        self.keys_xy = np.zeros((K, 64), np.uint8)
        L.siggen_keys(ctypes.c_uint64(seed), ctypes.c_int(K), self.priv.ctypes.data_as(ctypes.c_void_p), self.keys_xy.ctypes.data_as(ctypes.c_void_p))
        self.peers = [Identity("Org%dMSP" % (i + 1), i, bytes(self.keys_xy[i]), _pem_blob(b"peer%d" % i)) for i in range(n_orgs)]
        self.clients = [Identity("Org%dMSP" % (1 + i % n_orgs), n_orgs + i, bytes(self.keys_xy[n_orgs + i]), _pem_blob(b"client%d" % i))
                        for i in range(n_clients)]
        self.unknown = Identity("Org1MSP", K - 2, bytes(self.keys_xy[K - 2]), _pem_blob(b"unknown"))
        self.invalid_cert = Identity("Org2MSP", K - 1, bytes(self.keys_xy[K - 1]), _pem_blob(b"revoked"), valid=False)
        # every peer certificate once more in a byte-different PEM encoding (CRLF line ends): another serialization of the SAME
        # identity -- the reference de-duplicates on Mspid + certificate digest, not on the serialized bytes (policy.go:380-386)
        self.peers_alt = [Identity(p.mspid, p.priv_index, p.xy, p.cert_pem.replace(b"\n", b"\r\n")) for p in self.peers]
        self.msp_table = self.peers + self.clients + [self.invalid_cert] + self.peers_alt        # `unknown` deliberately absent
        self.principals = ["Org%dMSP" % (i + 1) for i in range(n_orgs)]
        # key index -> hash family of the MSP that key's identity belongs to
        self.key_family = {i.priv_index: self.hash_families.get(i.mspid, "SHA2") for i in self.msp_table + [self.unknown]}

    def digest(self, priv_index, msg: bytes) -> bytes:
        """What identity.Sign hashes before signing: SHA-256 or SHA3-256 per the signer's MSP family."""
        return (hashlib.sha3_256 if self.key_family.get(priv_index) == "SHA3" else hashlib.sha256)(msg).digest()

    def policies_for(self, n_endorsements):
        """(nodes, {namespace: root}): CHAINCODE wants n_endorsements of the orgs, STRICT_NAMESPACE one more; UNKNOWN_NAMESPACE has no entry."""
        a = self.policy_n_of(n_endorsements)
        b = self.policy_n_of(n_endorsements + 1).copy()
        b[0, 2] += a.shape[0]                                    # children of the second tree follow its root
        nodes = np.concatenate([a, b])
        return nodes, {CHAINCODE: 0, STRICT_NAMESPACE: int(a.shape[0])}

    def policy_n_of(self, n):
        """cauthdsl N-out-of over SignedBy(i) for every org: nodes as (type, n, first_child, n_children); type 0 = NOutOf, 1 = SignedBy."""
        nodes = [(0, n, 1, self.n_orgs)] + [(1, i, 0, 0) for i in range(self.n_orgs)]
        return np.array(nodes, np.int32)


def build_block(net: Network, n_tx: int, n_endorsements: int = 3, faults=None, seed=7, number=1, nthreads=None):
    """faults: {tx_index: fault_name}.  Returns (block_bytes, info) where info['expected_hint'][i] is the validation code the
    construction aims at (the oracle decides the truth)."""
    import ctypes
    faults = faults or {}
    rng = np.random.default_rng(seed)
    L = workload.lib()
    # ---- phase 1: build every message that must be signed ------------------------------------------------------
    txs = []
    sign_msgs, sign_keys = [], []
    for t in range(n_tx):
        f = faults.get(t)
        client = net.clients[t % len(net.clients)]
        if f == "unknown_creator":
            client = net.unknown
        if f == "invalid_creator_cert":
            client = net.invalid_cert
        nonce = bytes(rng.integers(0, 256, 24, dtype=np.uint8))
        if f == "dup_txid" and t > 0:
            nonce = txs[t - 1]["nonce"]
            client = txs[t - 1]["client"]
        creator = client.serialized
        txid = hashlib.sha256(nonce + creator).hexdigest()
        if f == "bad_txid":
            txid = hashlib.sha256(b"x" + nonce + creator).hexdigest()
        channel = net.channel if f != "wrong_channel" else "other-channel"
        htype = pb.HEADER_TYPE_ENDORSER_TRANSACTION if f != "config_update_type" else pb.HEADER_TYPE_CONFIG_UPDATE
        hext = pb.f_bytes(2, chaincode_id(CHAINCODE))                      # peer.ChaincodeHeaderExtension{chaincode_id = 2}
        if f == "bad_header_extension":
            hext = b"\x12\x7fshort"                                         # length prefix runs past the end
        chdr = pb.channel_header(htype, channel, txid, epoch=(5 if f == "nonzero_epoch" else 0), extension=hext)
        shdr = pb.signature_header(creator, b"" if f == "empty_nonce" else nonce)
        cpp = pb.f_bytes(1, b"invoke-args-" + bytes(rng.integers(0, 256, 40, dtype=np.uint8)))     # ChaincodeProposalPayload
        phash = hashlib.sha256(chdr + shdr + cpp).digest()
        if f == "bad_proposal_hash":
            phash = bytes(32)
        nss = [(CHAINCODE, 2, 2)]
        if f == "writes_strict_namespace":
            nss.append((STRICT_NAMESPACE, 0, 1))                            # cc-to-cc call that WRITES there: that policy applies too
        if f == "reads_strict_namespace":
            nss.append((STRICT_NAMESPACE, 2, 0))                            # only reads: the namespace is not validated
        if f == "writes_unknown_namespace":
            nss.append((UNKNOWN_NAMESPACE, 0, 1))
        if f == "dup_namespace":
            nss.append((CHAINCODE, 1, 0))
        rwset = tx_rwset(nss)
        if f == "bad_rwset":
            rwset = pb.f_bytes(2, b"\x0a\x7fnamespace-length-runs-past-the-end")
        ccact = pb.f_bytes(1, rwset) + pb.f_bytes(4, chaincode_id("othercc" if f == "cc_name_mismatch" else CHAINCODE, "" if f == "empty_cc_version" else "1.0"))
        if f == "event_wrong_cc":
            ccact += pb.f_bytes(2, pb.f_bytes(1, b"othercc") + pb.f_bytes(3, b"evt"))
        prp = pb.proposal_response_payload(phash, ccact)
        if f == "no_prp_extension":
            prp = pb.f_bytes(1, phash)
        # endorsers: the first n_endorsements orgs, rotated per tx
        order = [(t + k) % net.n_orgs for k in range(n_endorsements)]
        ends = [net.peers[o] for o in order]
        if f == "dup_endorser":
            ends[-1] = ends[0]
        if f == "unknown_endorser":
            ends[-1] = net.unknown
        if f == "same_cert_two_encodings":
            ends[-1] = net.peers_alt[order[0]]                             # the first endorser again, serialized differently
        if f == "many_endorsements":                                       # 21 endorsements: every org five times over (both encodings) + one
            ends = [(net.peers if (k // net.n_orgs) % 2 == 0 else net.peers_alt)[k % net.n_orgs] for k in range(5 * net.n_orgs + 1)]
        for e in ends:
            sign_msgs.append(prp + e.serialized)
            sign_keys.append(e.priv_index)
        txs.append(dict(fault=f, client=client, nonce=nonce, chdr=chdr, shdr=shdr, cpp=cpp, prp=prp, ends=ends, first_end_sig=len(sign_msgs) - len(ends)))
    # ---- phase 2: sign endorsements, assemble payloads, sign payloads ---------------------------------------------
    def sign_all(msgs, keys):
        n = len(msgs)
        dig = np.frombuffer(b"".join(net.digest(k, m) for m, k in zip(msgs, keys)), np.uint8).reshape(n, 32).copy()
        r = np.zeros((n, 32), np.uint8); s = np.zeros((n, 32), np.uint8)
        kidx = np.array(keys, np.int32)
        L.siggen_sign_batch(net.priv.ctypes.data_as(ctypes.c_void_p), kidx.ctypes.data_as(ctypes.c_void_p), dig.ctypes.data_as(ctypes.c_void_p),
                            ctypes.c_int(n), ctypes.c_uint64(seed + n), r.ctypes.data_as(ctypes.c_void_p), s.ctypes.data_as(ctypes.c_void_p),
                            ctypes.c_int(nthreads or min(os.cpu_count() or 1, 64)))
        off = np.zeros(n + 1, np.uint32); blob = np.zeros(72 * n + 8, np.uint8)
        L.siggen_der(r.ctypes.data_as(ctypes.c_void_p), s.ctypes.data_as(ctypes.c_void_p), ctypes.c_int(n), blob.ctypes.data_as(ctypes.c_void_p),
                     off.ctypes.data_as(ctypes.c_void_p))
        return [bytes(blob[off[i]:off[i + 1]]) for i in range(n)], r, s
    end_sigs, end_r, end_s = sign_all(sign_msgs, sign_keys)
    N_ORDER = 0xFFFFFFFF00000000FFFFFFFFFFFFFFFFBCE6FAADA7179E84F3B9CAC2FC632551
    payloads, payload_keys = [], []
    for t, tx in enumerate(txs):
        f = tx["fault"]
        sigs = end_sigs[tx["first_end_sig"]: tx["first_end_sig"] + len(tx["ends"])]
        if f in ("bad_endorsement_sig", "two_bad_endorsements"):
            for k in range(1 if f == "bad_endorsement_sig" else 2):
                b = bytearray(sigs[k]); b[-3] ^= 0x40; sigs[k] = bytes(b)
        if f == "high_s_endorsement":
            i0 = tx["first_end_sig"]
            rr = int.from_bytes(bytes(end_r[i0]), "big"); ss = N_ORDER - int.from_bytes(bytes(end_s[i0]), "big")
            sigs[0] = _der_sig(rr, ss)
        action = pb.chaincode_endorsed_action(tx["prp"], [pb.endorsement(e.serialized, sg) for e, sg in zip(tx["ends"], sigs)])
        cap = pb.chaincode_action_payload(tx["cpp"], action)
        data = pb.transaction([pb.transaction_action(tx["shdr"], cap)])
        pl = pb.payload(pb.header(tx["chdr"], tx["shdr"]), data)
        payloads.append(pl); payload_keys.append(tx["client"].priv_index)
    pay_sigs, _, _ = sign_all(payloads, payload_keys)
    envs = []
    for t, tx in enumerate(txs):
        f = tx["fault"]
        sg = pay_sigs[t]
        if f == "bad_creator_sig":
            b = bytearray(sg); b[-2] ^= 0x01; sg = bytes(b)
        if f == "no_signature":
            sg = b""
        env = pb.envelope(payloads[t], sg)
        if f == "bad_payload":
            env = pb.f_bytes(1, b"\xff\xff\xff\xff garbage that is not a Payload") + pb.f_bytes(2, sg)
        envs.append(env)
    env_off = np.zeros(len(envs) + 1, np.uint32)
    env_off[1:] = np.cumsum([len(e) for e in envs])
    return pb.block(number, envs), dict(n_tx=n_tx, faults=dict(faults), n_sigs=n_tx + sum(len(tx["ends"]) for tx in txs),
                                        env_blob=b"".join(envs), env_off=env_off)   # Block.Data.Data as the Go validator holds it
