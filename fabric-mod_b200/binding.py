"""ctypes binding of include/fabgpu_ecdsa.h (libfabgpu_ecdsa.so).  Fails loudly when the library is absent."""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# FABGPU_LIB: development knob, points the binding at another build of the same library (kernel A/B runs)
LIB_PATH = os.environ.get("FABGPU_LIB") or os.path.join(_HERE, "lib", "libfabgpu_ecdsa.so")
SLOTS = 3

OK, E_NO_DEVICE, E_CUDA, E_ARG, E_INJECTED = 0, -1, -2, -3, -4
HASH_SHA2, HASH_SHA3 = 0, 1          # FABGPU_HASH_*: the SignatureHashFamily of an MSP
HASH_FAMILIES = {"SHA2": HASH_SHA2, "SHA3": HASH_SHA3}
(ST_VALID, ST_INVALID, ST_ERR_NIL_KEY, ST_ERR_EMPTY_SIG, ST_ERR_EMPTY_DIGEST, ST_ERR_UNMARSHAL, ST_ERR_R_NOT_POSITIVE,
 ST_ERR_S_NOT_POSITIVE, ST_ERR_HIGH_S, ST_ERR_UNSUPPORTED_KEY, ST_ERR_OFF_CURVE) = range(11)

# every symbol include/fabgpu_ecdsa.h declares (tests/test_abi.py checks the header against this and the .so)
EXPORTS = [
    "fabgpu_init", "fabgpu_destroy", "fabgpu_last_error", "fabgpu_device_count", "fabgpu_max_batch",
    "fabgpu_host_buffers", "fabgpu_verify_p256", "fabgpu_verify_p256_async", "fabgpu_wait", "fabgpu_verify_p256_host",
    "fabgpu_verify_p256_device", "fabgpu_bccsp_verify_batch", "fabgpu_bccsp_verify", "fabgpu_gate_signature",
    "fabgpu_test_fieldop", "fabgpu_test_table_entries", "fabgpu_launch_count",
    "fabgpu_keys_register", "fabgpu_key_slot_capacity", "fabgpu_host_key_slots", "fabgpu_verify_p256_keyed",
    "fabgpu_verify_p256_keyed_async", "fabgpu_verify_p256_device_keyed", "fabgpu_last_timing", "fabgpu_build_info",
    "fabgpu_msp_configure", "fabgpu_validate_block", "fabgpu_validate_envelopes", "fabgpu_block_buffer", "fabgpu_block_timing", "fabgpu_sha256_segments",
    "fabgpu_bccsp_verify_batch_async", "fabgpu_bccsp_verify_batch_wait", "fabgpu_bccsp_batch_buffers", "fabgpu_bccsp_verify_batch_inplace_async",
    "fabgpu_msp_identity_groups", "fabgpu_namespace_policies", "fabgpu_msp_hash_families", "fabgpu_sha3_256_segments",
    "fabgpu_peer_mask_create", "fabgpu_peer_mask_open", "fabgpu_peer_mask_close", "fabgpu_verify_p256_device_keyed_allgather",
    "fabgpu_validate_block_async", "fabgpu_validate_envelopes_async", "fabgpu_validate_wait", "fabgpu_block_buffer_slot",
    "fabgpu_keys_register_small", "fabgpu_small_slot_capacity", "fabgpu_key_table_stats", "fabgpu_small_table_info",
]


class FabGpuError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("fabgpu error %d: %s" % (code, msg))
        self.code = code


def build(extra=""):
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    env = dict(os.environ)
    args = ["make", "-s", "-C", os.path.join(_HERE, "csrc")]
    if extra:
        args.append("EXTRA=" + extra)
    subprocess.check_call(args, env=env)


_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise FabGpuError(E_NO_DEVICE, "%s is missing: run __graft_entry__.build() (there is no CPU fallback)" % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        L.fabgpu_last_error.restype = ctypes.c_char_p
        L.fabgpu_last_error.argtypes = [ctypes.c_void_p]
        L.fabgpu_max_batch.restype = ctypes.c_size_t
        L.fabgpu_max_batch.argtypes = [ctypes.c_void_p]
        L.fabgpu_launch_count.restype = ctypes.c_ulonglong
        L.fabgpu_launch_count.argtypes = [ctypes.c_void_p]
        L.fabgpu_destroy.argtypes = [ctypes.c_void_p]
        L.fabgpu_destroy.restype = None
        L.fabgpu_device_count.argtypes = [ctypes.c_void_p]
        _LIB = L
    return _LIB


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None


def identity_groups(identities):
    """De-duplication groups for fabgpu_msp_identity_groups: identities = [(serialized SerializedIdentity bytes, mspid, ...)].  Two table
    entries get the same group id when they are the same certificate of the same MSP in byte-different encodings -- the reference's
    policy evaluation de-duplicates signers on Mspid + Id with Id = digest of the certificate's DER (common/policies/policy.go:380-386,
    msp/identities.go:55-76), not on the serialized bytes.  Entries whose PEM does not parse are their own group."""
    import base64
    import hashlib
    import re

    def id_bytes(ser):
        off, out = 0, b""
        while off < len(ser):                                   # SerializedIdentity{mspid = 1, id_bytes = 2}
            key = ser[off]; off += 1
            if key & 7 != 2:
                return None
            ln, shift = 0, 0
            while True:
                c = ser[off]; off += 1
                ln |= (c & 0x7F) << shift
                shift += 7
                if not c & 0x80:
                    break
            if key >> 3 == 2:
                out = ser[off:off + ln]
            off += ln
        return out

    keys, groups = {}, np.zeros(len(identities), np.int32)
    for i, it in enumerate(identities):
        ser, mspid = bytes(it[0]), it[1]
        k = (mspid, ser)
        try:
            m = re.search(rb"-----BEGIN CERTIFICATE-----(.*?)-----END CERTIFICATE-----", id_bytes(ser) or b"", re.S)
            if m:
                k = (mspid, hashlib.sha256(base64.b64decode(b"".join(m.group(1).split()))).digest())
        except Exception:
            pass
        groups[i] = keys.setdefault(k, len(keys))
    return groups


def build_info():
    """(window bits of the G table, window bits of the per-key tables) this library was compiled with."""
    a, b = ctypes.c_int(0), ctypes.c_int(0)
    lib().fabgpu_build_info(ctypes.byref(a), ctypes.byref(b))
    return a.value, b.value


def gate_signature(sig: bytes):
    """fabgpu_gate_signature: host gates only (no GPU).  Returns (status, r32, s32)."""
    r = (ctypes.c_uint8 * 32)()
    s = (ctypes.c_uint8 * 32)()
    buf = (ctypes.c_uint8 * max(1, len(sig))).from_buffer_copy(sig if len(sig) else b"\x00")
    st = lib().fabgpu_gate_signature(buf, ctypes.c_size_t(len(sig)), r, s)
    return st, bytes(r), bytes(s)


class Context:
    """fabgpu_ctx owner.  device_ids=None -> CUDA device 0."""

    def __init__(self, max_batch=65536, device_ids=None):
        L = lib()
        self._h = ctypes.c_void_p()
        if device_ids:
            arr = (ctypes.c_int * len(device_ids))(*device_ids)
            rc = L.fabgpu_init(arr, ctypes.c_int(len(device_ids)), ctypes.c_size_t(max_batch), ctypes.byref(self._h))
        else:
            rc = L.fabgpu_init(None, ctypes.c_int(0), ctypes.c_size_t(max_batch), ctypes.byref(self._h))
        if rc != OK:
            raise FabGpuError(rc, (L.fabgpu_last_error(None) or b"").decode())
        self.max_batch = max_batch

    def close(self):
        if self._h:
            lib().fabgpu_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != OK:
            raise FabGpuError(rc, (lib().fabgpu_last_error(self._h) or b"").decode())

    def last_error(self):
        return (lib().fabgpu_last_error(self._h) or b"").decode()

    def launch_count(self):
        return int(lib().fabgpu_launch_count(self._h))

    def device_count(self):
        return int(lib().fabgpu_device_count(self._h))

    # ---- leaf -------------------------------------------------------------------------------------------
    def host_buffers(self, slot=0):
        """numpy views (no copy) of the slot's pinned SoA buffers: dict qx,qy,e,r,s -> uint8[max_batch,32]; mask, offcurve."""
        ptrs = [ctypes.POINTER(ctypes.c_uint8)() for _ in range(5)]
        mask = ctypes.POINTER(ctypes.c_uint32)()
        off = ctypes.POINTER(ctypes.c_uint32)()
        self._ck(lib().fabgpu_host_buffers(self._h, ctypes.c_int(slot), *[ctypes.byref(p) for p in ptrs], ctypes.byref(mask), ctypes.byref(off)))
        out = {}
        for name, p in zip(("qx", "qy", "e", "r", "s"), ptrs):
            out[name] = np.ctypeslib.as_array(p, shape=(self.max_batch, 32))
        words = (self.max_batch + 31) // 32
        out["mask"] = np.ctypeslib.as_array(mask, shape=(words,))
        out["offcurve"] = np.ctypeslib.as_array(off, shape=(words,))
        return out

    def verify_p256(self, slot, n):
        self._ck(lib().fabgpu_verify_p256(self._h, ctypes.c_int(slot), ctypes.c_size_t(n)))

    def verify_p256_async(self, slot, n):
        self._ck(lib().fabgpu_verify_p256_async(self._h, ctypes.c_int(slot), ctypes.c_size_t(n)))

    def wait(self, slot):
        self._ck(lib().fabgpu_wait(self._h, ctypes.c_int(slot)))

    def verify_p256_host(self, qx, qy, e, r, s):
        """SoA uint8[n,32] arrays in ordinary host memory -> (mask uint32[ceil(n/32)], offcurve uint32[...])."""
        arrs = [np.ascontiguousarray(a, dtype=np.uint8).reshape(-1, 32) for a in (qx, qy, e, r, s)]
        n = arrs[0].shape[0]
        assert all(a.shape[0] == n for a in arrs)
        words = (n + 31) // 32
        mask = np.zeros(max(words, 1), np.uint32)
        off = np.zeros(max(words, 1), np.uint32)
        self._ck(lib().fabgpu_verify_p256_host(self._h, *[_p(a) for a in arrs], ctypes.c_size_t(n), _p(mask), _p(off)))
        return mask[:words], off[:words]

    def verify_p256_device(self, d_qx, d_qy, d_e, d_r, d_s, n, d_mask, d_off=0, stream=0, dev_index=0):
        """Raw device pointers (ints).  Enqueues on `stream` (a cudaStream_t as int) and returns immediately."""
        self._ck(lib().fabgpu_verify_p256_device(self._h, ctypes.c_int(dev_index), ctypes.c_void_p(d_qx), ctypes.c_void_p(d_qy),
                                                 ctypes.c_void_p(d_e), ctypes.c_void_p(d_r), ctypes.c_void_p(d_s), ctypes.c_size_t(n),
                                                 ctypes.c_void_p(d_mask), ctypes.c_void_p(d_off), ctypes.c_void_p(stream)))

    # ---- per-key tables ---------------------------------------------------------------------------------
    def keys_register(self, keys_xy):
        """uint8[K,64] -> int32[K] table slots (-1 = no table)."""
        keys_xy = np.ascontiguousarray(keys_xy, dtype=np.uint8).reshape(-1, 64)
        slots = np.full(keys_xy.shape[0], -1, np.int32)
        self._ck(lib().fabgpu_keys_register(self._h, _p(keys_xy), ctypes.c_int(keys_xy.shape[0]), _p(slots)))
        return slots

    def key_slot_capacity(self):
        return int(lib().fabgpu_key_slot_capacity(self._h))

    def keys_register_small(self, keys_xy):
        """uint8[K,64] -> int32[K] small-table handles (<= -2; -1 = no slot could be had)."""
        keys_xy = np.ascontiguousarray(keys_xy, dtype=np.uint8).reshape(-1, 64)
        handles = np.full(keys_xy.shape[0], -1, np.int32)
        self._ck(lib().fabgpu_keys_register_small(self._h, _p(keys_xy), ctypes.c_int(keys_xy.shape[0]), _p(handles)))
        return handles

    @staticmethod
    def small_raw_codes(handles):
        """small handles -> the raw device codes fabgpu_verify_p256_device_keyed takes (-2 - slot)."""
        h = np.asarray(handles, np.int64)
        return np.where(h <= -2, -2 - ((-2 - h) & 0xFFFFF), -1).astype(np.int32)

    def key_table_stats(self):
        """{'big': window tables alive, 'small': small tables alive, 'small_built': ..., 'small_recycled': ...}"""
        out = (ctypes.c_ulonglong * 4)()
        self._ck(lib().fabgpu_key_table_stats(self._h, out))
        return {"big": int(out[0]), "small": int(out[1]), "small_built": int(out[2]), "small_recycled": int(out[3])}

    @staticmethod
    def small_table_info():
        """(signed window bits, windows, bytes per table) of the small key tables."""
        wb, nw, nb = ctypes.c_int(0), ctypes.c_int(0), ctypes.c_size_t(0)
        lib().fabgpu_small_table_info(ctypes.byref(wb), ctypes.byref(nw), ctypes.byref(nb))
        return wb.value, nw.value, nb.value

    def small_slot_capacity(self):
        return int(lib().fabgpu_small_slot_capacity(self._h))

    def host_key_slots(self, slot=0):
        p = ctypes.POINTER(ctypes.c_int32)()
        self._ck(lib().fabgpu_host_key_slots(self._h, ctypes.c_int(slot), ctypes.byref(p)))
        return np.ctypeslib.as_array(p, shape=(self.max_batch,))

    def verify_p256_keyed(self, slot, n):
        self._ck(lib().fabgpu_verify_p256_keyed(self._h, ctypes.c_int(slot), ctypes.c_size_t(n)))

    def verify_p256_keyed_async(self, slot, n):
        self._ck(lib().fabgpu_verify_p256_keyed_async(self._h, ctypes.c_int(slot), ctypes.c_size_t(n)))

    def verify_p256_device_keyed(self, all_cached, d_key_slot, d_qx, d_qy, d_e, d_r, d_s, n, d_mask, d_off=0, stream=0, dev_index=0):
        self._ck(lib().fabgpu_verify_p256_device_keyed(self._h, ctypes.c_int(dev_index), ctypes.c_int(int(all_cached)),
                                                       ctypes.c_void_p(d_key_slot), ctypes.c_void_p(d_qx), ctypes.c_void_p(d_qy),
                                                       ctypes.c_void_p(d_e), ctypes.c_void_p(d_r), ctypes.c_void_p(d_s), ctypes.c_size_t(n),
                                                       ctypes.c_void_p(d_mask), ctypes.c_void_p(d_off), ctypes.c_void_p(stream)))

    # ---- bitmask exchange over peer memory (one process per GPU) ------------------------------------------
    def peer_mask_create(self, world, rank, words_per_rank, dev_index=0):
        h = np.zeros(64, np.uint8)
        self._ck(lib().fabgpu_peer_mask_create(self._h, ctypes.c_int(dev_index), ctypes.c_int(world), ctypes.c_int(rank), ctypes.c_size_t(words_per_rank), _p(h)))
        return h

    def peer_mask_open(self, handles, dev_index=0):
        handles = np.ascontiguousarray(handles, dtype=np.uint8).reshape(-1)
        self._ck(lib().fabgpu_peer_mask_open(self._h, ctypes.c_int(dev_index), _p(handles)))

    def peer_mask_close(self, dev_index=0):
        self._ck(lib().fabgpu_peer_mask_close(self._h, ctypes.c_int(dev_index)))

    def verify_p256_device_keyed_allgather(self, all_cached, d_key_slot, d_qx, d_qy, d_e, d_r, d_s, n, step, stream=0, dev_index=0):
        """Returns the device pointer (int) of the assembled world x words_per_rank mask words of this step."""
        out = ctypes.c_void_p(0)
        self._ck(lib().fabgpu_verify_p256_device_keyed_allgather(self._h, ctypes.c_int(dev_index), ctypes.c_int(1 if all_cached else 0), ctypes.c_void_p(d_key_slot),
                                                                 ctypes.c_void_p(d_qx), ctypes.c_void_p(d_qy), ctypes.c_void_p(d_e), ctypes.c_void_p(d_r),
                                                                 ctypes.c_void_p(d_s), ctypes.c_size_t(n), ctypes.c_uint32(step), ctypes.byref(out), ctypes.c_void_p(stream)))
        return int(out.value or 0)

    # ---- bccsp level ------------------------------------------------------------------------------------
    @staticmethod
    def _batch_args(keys_xy, key_idx, digests, dig_off, sigs, sig_off):
        keys_xy = np.ascontiguousarray(keys_xy, dtype=np.uint8).reshape(-1, 64)
        key_idx = np.ascontiguousarray(key_idx, dtype=np.int32)
        digests = np.ascontiguousarray(digests, dtype=np.uint8).reshape(-1)
        sigs = np.ascontiguousarray(sigs, dtype=np.uint8).reshape(-1)
        dig_off = np.ascontiguousarray(dig_off, dtype=np.uint32)
        sig_off = np.ascontiguousarray(sig_off, dtype=np.uint32)
        if digests.size == 0:
            digests = np.zeros(1, np.uint8)
        if sigs.size == 0:
            sigs = np.zeros(1, np.uint8)
        return keys_xy, key_idx, digests, dig_off, sigs, sig_off

    def bccsp_verify_batch(self, keys_xy, key_idx, digests, dig_off, sigs, sig_off):
        keys_xy, key_idx, digests, dig_off, sigs, sig_off = self._batch_args(keys_xy, key_idx, digests, dig_off, sigs, sig_off)
        n = key_idx.shape[0]
        status = np.full(max(n, 1), 255, np.uint8)
        self._ck(lib().fabgpu_bccsp_verify_batch(self._h, _p(keys_xy), ctypes.c_int(keys_xy.shape[0]), _p(key_idx), _p(digests), _p(dig_off),
                                                 _p(sigs), _p(sig_off), ctypes.c_size_t(n), _p(status)))
        return status[:n]

    def bccsp_verify_batch_async(self, slot, keys_xy, key_idx, digests, dig_off, sigs, sig_off):
        """First half of bccsp_verify_batch on one of the FABGPU_SLOTS slots; returns n for the matching _wait."""
        keys_xy, key_idx, digests, dig_off, sigs, sig_off = self._batch_args(keys_xy, key_idx, digests, dig_off, sigs, sig_off)
        n = key_idx.shape[0]
        self._ck(lib().fabgpu_bccsp_verify_batch_async(self._h, ctypes.c_int(slot), _p(keys_xy), ctypes.c_int(keys_xy.shape[0]), _p(key_idx),
                                                       _p(digests), _p(dig_off), _p(sigs), _p(sig_off), ctypes.c_size_t(n)))
        return n

    def bccsp_verify_batch_wait(self, slot, n, out=None):
        status = out if out is not None else np.full(max(n, 1), 255, np.uint8)
        self._ck(lib().fabgpu_bccsp_verify_batch_wait(self._h, ctypes.c_int(slot), _p(status), ctypes.c_size_t(n)))
        return status[:n]

    def bccsp_batch_buffers(self, slot, n_cap, sig_bytes_cap, dig_bytes_cap, k_cap):
        """numpy views (no copy) of the slot's pinned batch buffers: dict keys_xy uint8[k_cap,64], key_idx int32[n_cap], digests uint8[dig_bytes_cap],
        dig_off uint32[n_cap+1], sigs uint8[sig_bytes_cap], sig_off uint32[n_cap+1].  Fill them, then bccsp_verify_batch_inplace_async."""
        pk, pd, ps = (ctypes.POINTER(ctypes.c_uint8)() for _ in range(3))
        pi = ctypes.POINTER(ctypes.c_int32)()
        pdo, pso = ctypes.POINTER(ctypes.c_uint32)(), ctypes.POINTER(ctypes.c_uint32)()
        self._ck(lib().fabgpu_bccsp_batch_buffers(self._h, ctypes.c_int(slot), ctypes.c_size_t(n_cap), ctypes.c_size_t(sig_bytes_cap), ctypes.c_size_t(dig_bytes_cap),
                                                  ctypes.c_int(k_cap), ctypes.byref(pk), ctypes.byref(pi), ctypes.byref(pd), ctypes.byref(pdo), ctypes.byref(ps), ctypes.byref(pso)))
        A = np.ctypeslib.as_array
        return {"keys_xy": A(pk, shape=(max(k_cap, 1), 64)), "key_idx": A(pi, shape=(max(n_cap, 1),)), "digests": A(pd, shape=(max(dig_bytes_cap, 1),)),
                "dig_off": A(pdo, shape=(n_cap + 1,)), "sigs": A(ps, shape=(max(sig_bytes_cap, 1),)), "sig_off": A(pso, shape=(n_cap + 1,))}

    def bccsp_fill_batch_buffers(self, slot, keys_xy, key_idx, digests, dig_off, sigs, sig_off):
        """Convenience: reserve + copy a batch into the slot's pinned buffers once; returns (K, n) for bccsp_verify_batch_inplace_async."""
        keys_xy, key_idx, digests, dig_off, sigs, sig_off = self._batch_args(keys_xy, key_idx, digests, dig_off, sigs, sig_off)
        n, K = key_idx.shape[0], keys_xy.shape[0]
        hb = self.bccsp_batch_buffers(slot, n, int(sig_off[n]), int(dig_off[n]), K)
        hb["keys_xy"][:K] = keys_xy; hb["key_idx"][:n] = key_idx
        hb["digests"][: int(dig_off[n])] = digests[: int(dig_off[n])]; hb["dig_off"][: n + 1] = dig_off
        hb["sigs"][: int(sig_off[n])] = sigs[: int(sig_off[n])]; hb["sig_off"][: n + 1] = sig_off
        return K, n

    def bccsp_verify_batch_inplace_async(self, slot, K, n):
        self._ck(lib().fabgpu_bccsp_verify_batch_inplace_async(self._h, ctypes.c_int(slot), ctypes.c_int(K), ctypes.c_size_t(n)))
        return n

    def bccsp_verify(self, key_xy, sig, digest):
        """One sw.CSP.Verify call -> (valid: bool, err: str|None) with the reference's error strings."""
        valid = ctypes.c_int(0)
        err = ctypes.create_string_buffer(1024)
        kb = (ctypes.c_uint8 * 64).from_buffer_copy(key_xy) if key_xy is not None else None
        sb = (ctypes.c_uint8 * max(1, len(sig or b""))).from_buffer_copy(sig if sig else b"\x00")
        db = (ctypes.c_uint8 * max(1, len(digest or b""))).from_buffer_copy(digest if digest else b"\x00")
        self._ck(lib().fabgpu_bccsp_verify(self._h, kb, sb, ctypes.c_size_t(len(sig or b"")), db, ctypes.c_size_t(len(digest or b"")),
                                           ctypes.byref(valid), err, ctypes.c_size_t(1024)))
        e = err.value.decode()
        return bool(valid.value), (e if e else None)

    # ---- block level ------------------------------------------------------------------------------------
    def msp_configure(self, identities, policy_nodes, principals, channel, policies=None, hash_families=None):
        """identities: list of (serialized: bytes, mspid: str, key_xy: 64 bytes, valid: bool).  policy_nodes may hold several policy
        trees; policies = {namespace: root node index} names the tree of each chaincode namespace (None: node 0 for every namespace).
        The identities' de-duplication groups (Mspid + certificate, identity_groups) are installed as well.
        hash_families = {mspid: "SHA2" | "SHA3"}: the SignatureHashFamily of those MSPs (fabgpu_msp_hash_families); None or an MSP
        left out: SHA2."""
        def blob(items):
            off = np.zeros(len(items) + 1, np.uint32)
            off[1:] = np.cumsum([len(x) for x in items])
            b = np.frombuffer(b"".join(items) or b"\x00", np.uint8)
            return np.ascontiguousarray(b), off
        idb, ido = blob([bytes(i[0]) for i in identities])
        mb, mo = blob([i[1].encode() for i in identities])
        keys = np.ascontiguousarray(np.frombuffer(b"".join(bytes(i[2]) for i in identities) or b"\x00" * 64, np.uint8))
        valid = np.array([1 if i[3] else 0 for i in identities] or [0], np.uint8)
        nodes = np.ascontiguousarray(policy_nodes, dtype=np.int32).reshape(-1, 4)
        pbb, pbo = blob([p.encode() for p in principals])
        self._ck(lib().fabgpu_msp_configure(self._h, _p(idb), _p(ido), _p(mb), _p(mo), _p(keys), _p(valid), ctypes.c_int(len(identities)),
                                            _p(nodes), ctypes.c_int(nodes.shape[0]), _p(pbb), _p(pbo), ctypes.c_int(len(principals)),
                                            ctypes.c_char_p(channel.encode())))
        if identities:
            groups = np.ascontiguousarray(identity_groups(identities), np.int32)
            self._ck(lib().fabgpu_msp_identity_groups(self._h, _p(groups), ctypes.c_int(len(identities))))
        names = sorted(policies) if policies else []
        nb, no = blob([n.encode() for n in names])
        roots = np.array([policies[n] for n in names] or [0], np.int32)
        self._ck(lib().fabgpu_namespace_policies(self._h, _p(nb), _p(no), _p(roots), ctypes.c_int(len(names))))
        if hash_families is not None:
            self.msp_hash_families(hash_families)

    def msp_hash_families(self, hash_families):
        """{mspid: "SHA2" | "SHA3"} -> fabgpu_msp_hash_families (after msp_configure; {} restores all-SHA2)."""
        unknown = {f for f in hash_families.values() if f not in HASH_FAMILIES}
        if unknown:
            raise ValueError("hash family must be SHA2 or SHA3, got %s" % sorted(map(str, unknown)))
        names = sorted(hash_families)
        off = np.zeros(len(names) + 1, np.uint32)
        off[1:] = np.cumsum([len(n.encode()) for n in names])
        mb = np.ascontiguousarray(np.frombuffer(b"".join(n.encode() for n in names) or b"\x00", np.uint8))
        fam = np.array([HASH_FAMILIES[hash_families[n]] for n in names] or [0], np.uint8)
        self._ck(lib().fabgpu_msp_hash_families(self._h, _p(mb), _p(off), _p(fam), ctypes.c_int(len(names))))

    def block_buffer(self, nbytes, slot=0):
        """Pinned staging buffer (numpy view) for block bytes; one per slot."""
        p = ctypes.POINTER(ctypes.c_uint8)()
        self._ck(lib().fabgpu_block_buffer_slot(self._h, ctypes.c_int(slot), ctypes.c_size_t(nbytes), ctypes.byref(p)))
        return np.ctypeslib.as_array(p, shape=(nbytes,))

    def validate_envelopes_async(self, slot, blob, env_off):
        """First half of validate_envelopes on one of the FABGPU_SLOTS slots.  `blob` must stay alive and unchanged until
        validate_wait(slot) returns (it is kept referenced here).  Returns the number of envelopes."""
        arr = np.frombuffer(blob, np.uint8) if isinstance(blob, (bytes, bytearray)) else blob
        env_off = np.ascontiguousarray(env_off, dtype=np.uint32)
        n_env = env_off.shape[0] - 1
        self._inflight = getattr(self, "_inflight", {})
        self._inflight[slot] = (arr, env_off)
        self._ck(lib().fabgpu_validate_envelopes_async(self._h, ctypes.c_int(slot), _p(arr), _p(env_off), ctypes.c_size_t(n_env)))
        return n_env

    def validate_block_async(self, slot, block):
        arr = np.frombuffer(block, np.uint8) if isinstance(block, (bytes, bytearray)) else block
        self._inflight = getattr(self, "_inflight", {})
        self._inflight[slot] = (arr,)
        self._ck(lib().fabgpu_validate_block_async(self._h, ctypes.c_int(slot), _p(arr), ctypes.c_size_t(arr.shape[0])))
        return max(16, arr.shape[0] // 2)

    def validate_wait(self, slot, max_tx):
        flags = np.full(max(max_tx, 1), 254, np.uint8)
        n = ctypes.c_size_t(0)
        try:
            self._ck(lib().fabgpu_validate_wait(self._h, ctypes.c_int(slot), _p(flags), ctypes.c_size_t(flags.shape[0]), ctypes.byref(n)))
        finally:
            getattr(self, "_inflight", {}).pop(slot, None)
        return flags[: n.value]

    def validate_block(self, block, max_tx=None):
        """block: bytes or a uint8 numpy array (e.g. a slice of block_buffer()).  Returns the TRANSACTIONS_FILTER bytes."""
        arr = np.frombuffer(block, np.uint8) if isinstance(block, (bytes, bytearray)) else block
        cap = max_tx or max(16, arr.shape[0] // 64)
        flags = np.full(cap, 254, np.uint8)
        n = ctypes.c_size_t(0)
        self._ck(lib().fabgpu_validate_block(self._h, _p(arr), ctypes.c_size_t(arr.shape[0]), _p(flags), ctypes.c_size_t(cap), ctypes.byref(n)))
        return flags[: n.value]

    def validate_envelopes(self, blob, env_off):
        """blob: uint8 array holding the envelopes back to back; env_off: uint32[n+1].  Returns the flags."""
        arr = np.frombuffer(blob, np.uint8) if isinstance(blob, (bytes, bytearray)) else blob
        env_off = np.ascontiguousarray(env_off, dtype=np.uint32)
        n_env = env_off.shape[0] - 1
        flags = np.full(max(n_env, 1), 254, np.uint8)
        n = ctypes.c_size_t(0)
        self._ck(lib().fabgpu_validate_envelopes(self._h, _p(arr), _p(env_off), ctypes.c_size_t(n_env), _p(flags), ctypes.c_size_t(max(n_env, 1)),
                                                 ctypes.byref(n)))
        return flags[: n.value]

    def block_timing(self):
        out = (ctypes.c_double * 10)()
        self._ck(lib().fabgpu_block_timing(self._h, out))
        return [float(x) for x in out]

    def sha256_segments(self, buf, jobs):
        """jobs: uint32[n,6] (off0,off1,off2,len0,len1,len2) -> uint8[n,32]."""
        buf = np.ascontiguousarray(np.frombuffer(buf, np.uint8) if isinstance(buf, (bytes, bytearray)) else buf)
        jobs = np.ascontiguousarray(jobs, dtype=np.uint32).reshape(-1, 6)
        out = np.zeros((jobs.shape[0], 32), np.uint8)
        self._ck(lib().fabgpu_sha256_segments(self._h, _p(buf), ctypes.c_size_t(buf.shape[0]), _p(jobs), ctypes.c_size_t(jobs.shape[0]), _p(out)))
        return out

    def sha3_256_segments(self, buf, jobs):
        """jobs: uint32[n,6] (off0,off1,off2,len0,len1,len2) -> uint8[n,32] SHA3-256 digests."""
        buf = np.ascontiguousarray(np.frombuffer(buf, np.uint8) if isinstance(buf, (bytes, bytearray)) else buf)
        jobs = np.ascontiguousarray(jobs, dtype=np.uint32).reshape(-1, 6)
        out = np.zeros((jobs.shape[0], 32), np.uint8)
        self._ck(lib().fabgpu_sha3_256_segments(self._h, _p(buf), ctypes.c_size_t(buf.shape[0]), _p(jobs), ctypes.c_size_t(jobs.shape[0]), _p(out)))
        return out

    def last_timing(self):
        """[key lookup, host gates, device, scatter] microseconds of the last bccsp_verify_batch call."""
        out = (ctypes.c_double * 4)()
        self._ck(lib().fabgpu_last_timing(self._h, out))
        return [float(x) for x in out]

    # ---- test hooks -------------------------------------------------------------------------------------
    def test_fieldop(self, op, a, b):
        a = np.ascontiguousarray(a, dtype=np.uint8).reshape(-1, 32)
        b = np.ascontiguousarray(b, dtype=np.uint8).reshape(-1, 32)
        out = np.zeros_like(a)
        self._ck(lib().fabgpu_test_fieldop(self._h, ctypes.c_int(op), _p(a), _p(b), ctypes.c_size_t(a.shape[0]), _p(out)))
        return out

    def test_table_entries(self, key_slot, window, digit):
        """Sampled window-table entries (key_slot < 0: generator table) -> (n, 16) little-endian u32 limbs, X then Y, Montgomery form."""
        window = np.ascontiguousarray(window, dtype=np.uint32)
        digit = np.ascontiguousarray(digit, dtype=np.uint32)
        out = np.zeros((window.shape[0], 64), np.uint8)
        self._ck(lib().fabgpu_test_table_entries(self._h, ctypes.c_int(key_slot), _p(window), _p(digit), ctypes.c_size_t(window.shape[0]), _p(out)))
        return out.view("<u4").reshape(-1, 16)
