// Device-side block pre-pass: the same walk, gates and decisions as blockval.cpp / bccsp_host.cpp, written once as
// host+device code so that (a) the GPU runs it with one thread per transaction straight on the block bytes that are in
// HBM anyway (SURVEY.md section 8f ranks 1 and 3: block pre-pass, DER / low-S gates on the device) and (b) tests can run
// the identical code on the CPU-only build box (tests/host_sim/blockdev_host.cpp).
//
// Reference semantics restated here (see blockval.hpp for the full list):
//   ValidateTransaction / checkSignatureFromCreator / validateEndorserTransaction   core/common/validation/msgvalidation.go:26-320
//   KeyLevelValidator signature set        core/common/validation/statebased/validator_keylevel.go:243-259
//   SignatureSetToValidIdentities          common/policies/policy.go:365-402
//   cauthdsl evaluator                     common/cauthdsl/cauthdsl.go:24-92
//   UnmarshalECDSASignature / IsLowS       bccsp/utils/ecdsa.go:43-92 (Go encoding/asn1 DER rules)
// No STL, no allocation: everything is offsets into the block buffer and fixed-size records.
#pragma once
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define BD_HD __host__ __device__ __forceinline__
#else
#define BD_HD inline
#endif

namespace fabgpu { namespace bdev {

enum : uint8_t {
    TXC_VALID = 0, TXC_BAD_PAYLOAD = 2, TXC_BAD_COMMON_HEADER = 3, TXC_BAD_CREATOR_SIGNATURE = 4, TXC_INVALID_ENDORSER_TRANSACTION = 5,
    TXC_UNSUPPORTED_TX_PAYLOAD = 7, TXC_BAD_PROPOSAL_TXID = 8, TXC_DUPLICATE_TXID = 9, TXC_ENDORSEMENT_POLICY_FAILURE = 10,
    TXC_TARGET_CHAIN_NOT_FOUND = 14, TXC_BAD_HEADER_EXTENSION = 19, TXC_BAD_RESPONSE_PAYLOAD = 21, TXC_BAD_RWSET = 22, TXC_ILLEGAL_WRITESET = 23,
    TXC_INVALID_CHAINCODE = 25, TXC_NOT_VALIDATED = 254, TXC_INVALID_OTHER_REASON = 255
};

#define BD_MAX_SIGNERS 64       // distinct verified signers one policy evaluation handles (`used` is a 64-bit mask); more -> CPU validator
#define BD_MAX_NS 4             // namespaces validated per transaction (the invoked chaincode + those it writes to); more -> CPU validator
#define BD_MAX_NS_SEEN 8        // namespaces of one read/write set checked for duplicates; more -> CPU validator
#define BD_ENDS_HINT 16         // job-array sizing: expected endorsements per transaction (the capacity is a parameter, see JobArrays::J_cap)

struct Seg { uint32_t off, len; };

// ---- MSP view on the device --------------------------------------------------------------------------------------------
struct MspDev {
    const uint8_t* id_blob;       // serialized identities back to back
    const uint32_t* id_off;       // n_ids + 1
    const int32_t* key_slot;      // per identity: big-table slot (>= 0), small-table code (<= -2) or -1
    const uint8_t* valid;         // per identity: identity.Validate()
    const int32_t* msp_code;      // per identity: code of its MSP id (equal ids <=> equal codes)
    const int32_t* group;         // per identity: de-duplication id -- Mspid + certificate (policy.go:380-386): two serializations of one
                                  // certificate share it; null = every table entry is its own group
    const uint8_t* keys_xy;       // per identity: X || Y (64 bytes), for signatures whose key has no table
    const uint8_t* hash_kind = nullptr;   // per identity: hash of identity.Verify, 0 = SHA-256, 1 = SHA3-256 (the MSP's SignatureHashFamily,
                                          // msp/identities.go:169-196,216-224); null = SHA-256 for every identity
    const uint64_t* ht_hash;      // open-addressing table, size ht_size (power of two); 0 = empty
    const int32_t* ht_idx;
    uint32_t ht_size;
    int32_t n_ids;
};

// Hash of a serialized identity from 16 + 32 + 32 + 24 sampled bytes.  A SerializedIdentity is the MSP id followed by a PEM certificate: every
// identity of an MSP starts with the same bytes and ends with the same "-----END CERTIFICATE-----" footer, so head and tail alone (round 1) put all
// of an MSP's identities into ONE probe chain -- harmless with a dozen identities, 1.7 ms per block with 2 000 client certificates (the creator
// pass of block_resolve_kernel: 1 696 us against 46 us, profiles/r2_block_many_clients_launches.csv).  The two inner windows fall into the base64
// body: the middle (subject / public key) and the end of the signature just before the footer.
BD_HD uint64_t sample_hash(const uint8_t* p, uint32_t n)
{
    uint64_t h = 1469598103934665603ull ^ n;
    const uint32_t head = n < 16 ? n : 16, tail = n < 24 ? n : 24;
    for (uint32_t i = 0; i < head; i++) h = (h ^ p[i]) * 1099511628211ull;
    if (n >= 160) {
        for (uint32_t i = n / 2 - 16; i < n / 2 + 16; i++) h = (h ^ p[i]) * 1099511628211ull;
        for (uint32_t i = n - 72; i < n - 40; i++) h = (h ^ p[i]) * 1099511628211ull;
    }
    for (uint32_t i = n - tail; i < n; i++) h = (h ^ p[i]) * 1099511628211ull;
    return h ? h : 1;
}

BD_HD bool bytes_equal(const uint8_t* a, const uint8_t* b, uint32_t n)
{
#if defined(__CUDA_ARCH__)
    // ~1 KiB identities are compared four times per transaction: go by aligned 32-bit words on both sides, re-aligning
    // each stream with a funnel shift (reads stay inside the 4-byte-aligned words that contain the ranges).
    if (n >= 8) {
        const uint32_t sa = 8u * (uint32_t)((uintptr_t)a & 3u), sb = 8u * (uint32_t)((uintptr_t)b & 3u);
        const uint32_t* pa = reinterpret_cast<const uint32_t*>((uintptr_t)a & ~(uintptr_t)3);
        const uint32_t* pb = reinterpret_cast<const uint32_t*>((uintptr_t)b & ~(uintptr_t)3);
        const uint32_t words = n >> 2;
        // Eight words per step with no exit in between: the sixteen-plus loads of a step are in flight together (with an
        // exit test after every word each ~1 KiB identity cost ~275 dependent HBM round trips).
        uint32_t k = 0;
        for (; k + 8 <= words; k += 8) {
            uint32_t xa[9], xb[9];
#pragma unroll
            for (int q = 0; q < 9; q++) { xa[q] = pa[k + q]; xb[q] = pb[k + q]; }    // word k+8 lies inside the range or its slack
            uint32_t diff = 0;
#pragma unroll
            for (int q = 0; q < 8; q++) diff |= __funnelshift_r(xa[q], xa[q + 1], sa) ^ __funnelshift_r(xb[q], xb[q + 1], sb);
            if (diff) return false;
        }
        for (; k < words; k++) {
            const uint32_t wa = __funnelshift_r(pa[k], pa[k + 1], sa), wb = __funnelshift_r(pb[k], pb[k + 1], sb);
            if (wa != wb) return false;
        }
        for (uint32_t i = words << 2; i < n; i++) if (a[i] != b[i]) return false;
        return true;
    }
#endif
    for (uint32_t i = 0; i < n; i++) if (a[i] != b[i]) return false;
    return true;
}

BD_HD int32_t msp_find(const MspDev& m, const uint8_t* p, uint32_t n)
{
    if (m.ht_size == 0) return -1;
    const uint64_t h = sample_hash(p, n);
    for (uint32_t probe = 0, pos = (uint32_t)h & (m.ht_size - 1); probe < m.ht_size; probe++, pos = (pos + 1) & (m.ht_size - 1)) {
        const uint64_t k = m.ht_hash[pos];
        if (k == 0) return -1;
        if (k != h) continue;
        const int32_t i = m.ht_idx[pos];
        const uint32_t len = m.id_off[i + 1] - m.id_off[i];
        if (len == n && bytes_equal(m.id_blob + m.id_off[i], p, n)) return i;
    }
    return -1;
}

// ---- protobuf wire reader ------------------------------------------------------------------------------------------------
struct Reader {
    const uint8_t* base; uint32_t pos, end; bool ok;
    BD_HD bool varint(uint64_t& v)
    {
        v = 0;
        for (int shift = 0; shift < 70; shift += 7) {
            if (pos >= end) { ok = false; return false; }
            const uint8_t c = base[pos++];
            v |= (uint64_t)(c & 0x7f) << shift;
            if (!(c & 0x80)) return true;
        }
        ok = false; return false;
    }
    BD_HD bool next(uint32_t& field, uint32_t& wt, uint64_t& val, Seg& bytes)
    {
        if (pos >= end) return false;
        uint64_t key;
        if (!varint(key)) return false;
        field = (uint32_t)(key >> 3); wt = (uint32_t)(key & 7);
        if (field == 0) { ok = false; return false; }
        if (wt == 0) return varint(val);
        if (wt == 1) { if (end - pos < 8) { ok = false; return false; } pos += 8; return true; }
        if (wt == 5) { if (end - pos < 4) { ok = false; return false; } pos += 4; return true; }
        if (wt == 2) {
            uint64_t ln;
            if (!varint(ln)) return false;
            if ((uint64_t)(end - pos) < ln) { ok = false; return false; }
            bytes.off = pos; bytes.len = (uint32_t)ln; pos += (uint32_t)ln;
            return true;
        }
        ok = false; return false;
    }
};

// Up to 3 selected length-delimited fields (last occurrence wins) and up to 2 varint fields of one message.
struct Sel { uint32_t f[3]; Seg s[3]; bool present[3]; uint32_t uf[2]; uint64_t uv[2]; };

BD_HD bool parse_sel(const uint8_t* base, Seg msg, Sel& sel)
{
    Reader r; r.base = base; r.pos = msg.off; r.end = msg.off + msg.len; r.ok = true;
    for (int i = 0; i < 3; i++) { sel.s[i].off = 0; sel.s[i].len = 0; sel.present[i] = false; }
    sel.uv[0] = sel.uv[1] = 0;
    uint32_t f, wt; uint64_t v = 0; Seg b; b.off = b.len = 0;
    while (r.next(f, wt, v, b)) {
        bool hit = false;
        for (int i = 0; i < 2 && !hit; i++) if (sel.uf[i] && sel.uf[i] == f) { if (wt != 0) return false; sel.uv[i] = v; hit = true; }
        for (int i = 0; i < 3 && !hit; i++) if (sel.f[i] && sel.f[i] == f) { if (wt != 2) return false; sel.s[i] = b; sel.present[i] = true; hit = true; }
    }
    return r.ok;
}
BD_HD Sel make_sel(uint32_t f0, uint32_t f1 = 0, uint32_t f2 = 0, uint32_t u0 = 0, uint32_t u1 = 0)
{
    Sel s; s.f[0] = f0; s.f[1] = f1; s.f[2] = f2; s.uf[0] = u0; s.uf[1] = u1; return s;
}

// ---- DER gate (Go encoding/asn1 rules; bccsp/utils/ecdsa.go:43-92, bccsp/sw/ecdsa.go:42-54) -----------------------------
// Returns true when every gate passes (r, s written as 32 big-endian bytes).  false covers unmarshal errors, R <= 0,
// S <= 0, high S and r >= 2^256: at block level all of those make identity.Verify fail alike.
BD_HD bool der_tag_len(const uint8_t* b, uint32_t n, uint32_t& off, uint32_t& cls, bool& compound, uint32_t& tag, uint32_t& length)
{
    if (off >= n) return false;
    uint8_t c = b[off++];
    cls = c >> 6; compound = (c & 0x20) != 0; tag = c & 0x1f;
    if (tag == 0x1f) {
        uint64_t t = 0; int shifted = 0;
        for (;;) {
            if (off >= n || shifted == 5) return false;
            c = b[off++];
            if (shifted == 0 && c == 0x80) return false;
            t = (t << 7) | (c & 0x7f); shifted++;
            if (!(c & 0x80)) break;
        }
        if (t > 0x7fffffffull || t < 0x1f) return false;
        tag = (uint32_t)t;
    }
    if (off >= n) return false;
    c = b[off++];
    if (!(c & 0x80)) { length = c & 0x7f; return true; }
    const int nb = c & 0x7f;
    if (nb == 0) return false;
    uint32_t L = 0;
    for (int i = 0; i < nb; i++) {
        if (off >= n) return false;
        c = b[off++];
        if (L >= (1u << 23)) return false;
        L = (L << 8) | c;
        if (L == 0) return false;
    }
    if (L < 0x80) return false;
    length = L;
    return true;
}

BD_HD bool der_int(const uint8_t* b, uint32_t n, uint32_t& off, uint32_t& vo, uint32_t& vl)
{
    if (off == n) return false;
    uint32_t cls, tag, len; bool compound;
    if (!der_tag_len(b, n, off, cls, compound, tag, len)) return false;
    if ((uint64_t)off + len > n) return false;
    if (cls != 0 || tag != 2 || compound || len == 0) return false;
    const uint8_t* p = b + off;
    if (len > 1 && ((p[0] == 0 && !(p[1] & 0x80)) || (p[0] == 0xff && (p[1] & 0x80)))) return false;
    vo = off; vl = len; off += len;
    return true;
}

// Gate outcome as the status code of include/fabgpu_ecdsa.h: 0 = every gate passed (ask the curve arithmetic),
// 1 = (false, nil) because r >= 2^256, 5 = unmarshal error, 6 / 7 = R / S not positive, 8 = high S.
// Order of checks as in bccsp/sw/ecdsa.go:41-54: unmarshal, R > 0, S > 0, then low-S, then ecdsa.Verify's range checks.
BD_HD int gate_signature_status(const uint8_t* sig, uint32_t n, uint8_t* r32, uint8_t* s32)
{
    const uint8_t half[32] = {0x7F, 0xFF, 0xFF, 0xFF, 0x80, 0x00, 0x00, 0x00, 0x7F, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF,
                              0xDE, 0x73, 0x7D, 0x56, 0xD3, 0x8B, 0xCF, 0x42, 0x79, 0xDC, 0xE5, 0x61, 0x7E, 0x31, 0x92, 0xA8};
    if (n == 0) return 5;
    uint32_t off = 0, cls, tag, len; bool compound;
    if (!der_tag_len(sig, n, off, cls, compound, tag, len)) return 5;
    if ((uint64_t)off + len > n) return 5;
    if (cls != 0 || tag != 16 || !compound) return 5;
    const uint8_t* inner = sig + off;
    uint32_t io = 0, ro, rl, so, sl;
    if (!der_int(inner, len, io, ro, rl)) return 5;
    if (!der_int(inner, len, io, so, sl)) return 5;
    const uint8_t* rp = inner + ro; const uint8_t* sp = inner + so;
    const bool r_neg = (rp[0] & 0x80) != 0, s_neg = (sp[0] & 0x80) != 0;
    while (rl > 0 && *rp == 0) { rp++; rl--; }
    while (sl > 0 && *sp == 0) { sp++; sl--; }
    if (r_neg || rl == 0) return 6;                               // R must be larger than zero
    if (s_neg || sl == 0) return 7;                               // S must be larger than zero
    if (sl > 32) return 8;                                        // s >= 2^256 > N/2
    for (int i = 0; i < 32; i++) s32[i] = 0;
    for (uint32_t i = 0; i < sl; i++) s32[32 - sl + i] = sp[i];
    for (int i = 0; i < 32; i++) {                                // s <= N >> 1
        if (s32[i] < half[i]) break;
        if (s32[i] > half[i]) return 8;
    }
    if (rl > 32) return 1;                                        // r >= 2^256 can never be < N: (false, nil)
    for (int i = 0; i < 32; i++) r32[i] = 0;
    for (uint32_t i = 0; i < rl; i++) r32[32 - rl + i] = rp[i];
    return 0;
}

BD_HD bool gate_signature(const uint8_t* sig, uint32_t n, uint8_t* r32, uint8_t* s32)
{
    return gate_signature_status(sig, n, r32, s32) == 0;
}

// ---- per-transaction plan --------------------------------------------------------------------------------------------------
struct ShaJobD { uint32_t off[3]; uint32_t len[3]; };

struct TxDev {
    uint8_t early;                 // decided by structure alone, else TXC_NOT_VALIDATED
    uint8_t htype;
    uint8_t endorser_parse_ok, channel_ok, endorsements_parse_ok, overflow;
    uint8_t disp;                  // plugin dispatcher's structural verdict (dispatcher.go:102-179): TXC_VALID or the code it returns
    uint8_t n_ns;                  // namespaces to validate: wr_ns[0] = the invoked chaincode, then the others it writes to
    int32_t creator_identity;      // -1 unknown
    int32_t creator_has_job;       // creator job index is the transaction index when 1
    Seg txid_ascii;
    Seg phash_claimed;
    uint32_t first_end_job;        // endorsement jobs [first_end_job, first_end_job + n_end_jobs), in endorsement order
    uint32_t n_end_jobs;           // (endorsements without signature bytes get none: they can never verify)
    Seg wr_ns[BD_MAX_NS];
};

// Everything plan_tx writes for one transaction besides TxDev: job records live in caller-provided arrays.
struct JobArrays {
    ShaJobD* sha;                  // [J_cap + 2 T]: signature messages, then (txid, proposal hash) per transaction
    uint8_t* r; uint8_t* s;        // [J_cap x 32]
    int32_t* key_slot;             // [J_cap]
    int32_t* identity;             // [J_cap]
    uint8_t* qx; uint8_t* qy;      // [J_cap x 32] or null: filled only for keys without a table (generic kernel)
    uint8_t* gate_ok;              // [J_cap]
    uint8_t* kind = nullptr;       // [J_cap] or null: hash of each signature message, from its signer's MspDev::hash_kind
    uint32_t J_cap;                // capacity; creator jobs occupy [0, T), endorsement jobs [T, T + n_end)
    uint32_t T;
};

// What the walk leaves for one signature; identity lookup and DER gate are done per job by resolve_job (four times
// more threads than transactions: the walk alone exposed too little parallelism -- ncu: 2 warps/SM, issue active 3 %).
struct RawJob { Seg ident; Seg sig; uint32_t tx; int32_t k; };   // k = -1: creator signature, else endorsement index; tx = 0xffffffff: unused slot

// Wire scan of one message: known fields must carry their wire type (Go's proto.Unmarshal fails otherwise); on_bytes(field, seg)
// is called for every length-delimited KNOWN field in order.  bytes_mask / varint_mask: bit f = field f is known with that type.
template <typename F>
BD_HD bool scan_msg(const uint8_t* base, Seg msg, uint32_t bytes_mask, uint32_t varint_mask, F on_bytes)
{
    Reader r; r.base = base; r.pos = msg.off; r.end = msg.off + msg.len; r.ok = true;
    uint32_t f, wt; uint64_t v = 0; Seg b; b.off = b.len = 0;
    while (r.next(f, wt, v, b)) {
        if (f < 32 && ((bytes_mask >> f) & 1u)) { if (wt != 2) return false; on_bytes(f, b); }
        else if (f < 32 && ((varint_mask >> f) & 1u)) { if (wt != 0) return false; }
    }
    return r.ok;
}
#define BD_F(n) (1u << (n))

BD_HD bool seg_equal(const uint8_t* base, Seg a, Seg b)
{
    if (a.len != b.len) return false;
    for (uint32_t i = 0; i < a.len; i++) if (base[a.off + i] != base[b.off + i]) return false;
    return true;
}

// The plugin dispatcher's structural checks (plugindispatcher/dispatcher.go:102-179), in its order.  chdr_ext: ChannelHeader.extension;
// prp / prp_ext: ProposalResponsePayload bytes and its extension (peer.ChaincodeAction).  Fills tx.disp, tx.wr_ns, tx.n_ns.
BD_HD void dispatch_plan(const uint8_t* base, Seg chdr_ext, bool has_prp, bool has_prp_ext, Seg prp_ext, TxDev& tx)
{
    tx.disp = TXC_VALID; tx.n_ns = 0;
    // hdrExt = ChaincodeHeaderExtension{chaincode_id = 2}, its ChaincodeID{path = 1, name = 2, version = 3} parsed with it
    Seg h_ccid; h_ccid.off = h_ccid.len = 0; bool has_h_ccid = false;
    if (!scan_msg(base, chdr_ext, BD_F(2), 0, [&](uint32_t, Seg b) { h_ccid = b; has_h_ccid = true; })) { tx.disp = TXC_BAD_HEADER_EXTENSION; return; }
    Seg h_name; h_name.off = h_name.len = 0;
    if (has_h_ccid && !scan_msg(base, h_ccid, BD_F(1) | BD_F(2) | BD_F(3), 0, [&](uint32_t f, Seg b) { if (f == 2) h_name = b; })) { tx.disp = TXC_BAD_HEADER_EXTENSION; return; }
    // respPayload = GetActionFromEnvelope: ChaincodeAction{results = 1, events = 2, response = 3, chaincode_id = 4}
    if (!has_prp || !has_prp_ext) { tx.disp = TXC_BAD_RESPONSE_PAYLOAD; return; }
    Seg results, events, r_ccid; results.off = results.len = events.off = events.len = r_ccid.off = r_ccid.len = 0;
    bool has_events = false, has_r_ccid = false;
    if (!scan_msg(base, prp_ext, BD_F(1) | BD_F(2) | BD_F(3) | BD_F(4), 0, [&](uint32_t f, Seg b) {
            if (f == 1) results = b; else if (f == 2) { events = b; has_events = true; } else if (f == 4) { r_ccid = b; has_r_ccid = true; } })) {
        tx.disp = TXC_BAD_RESPONSE_PAYLOAD; return;
    }
    Seg r_name, r_ver; r_name.off = r_name.len = r_ver.off = r_ver.len = 0;
    if (has_r_ccid && !scan_msg(base, r_ccid, BD_F(1) | BD_F(2) | BD_F(3), 0, [&](uint32_t f, Seg b) { if (f == 2) r_name = b; else if (f == 3) r_ver = b; })) {
        tx.disp = TXC_BAD_RESPONSE_PAYLOAD; return;
    }
    // txRWSet.FromProtoBytes(results): TxReadWriteSet{data_model = 1, ns_rwset = 2}, every namespace with its KVRWSet and hashed collections
    Seg seen[BD_MAX_NS_SEEN]; bool wrote[BD_MAX_NS_SEEN]; uint32_t n_seen = 0; bool too_many = false, rw_ok = true;
    const bool top_ok = scan_msg(base, results, BD_F(2), BD_F(1), [&](uint32_t, Seg nsb) {
        if (!rw_ok) return;
        Seg name, kv; name.off = name.len = kv.off = kv.len = 0;
        bool writes = false;
        // NsReadWriteSet{namespace = 1, rwset = 2, collection_hashed_rwset = 3}
        if (!scan_msg(base, nsb, BD_F(1) | BD_F(2) | BD_F(3), 0, [&](uint32_t f, Seg b) {
                if (f == 1) name = b; else if (f == 2) kv = b;
                else {                                                  // CollectionHashedReadWriteSet{collection_name = 1, hashed_rwset = 2, pvt_rwset_hash = 3}
                    Seg hashed; hashed.off = hashed.len = 0;
                    if (!scan_msg(base, b, BD_F(1) | BD_F(2) | BD_F(3), 0, [&](uint32_t g, Seg c) { if (g == 2) hashed = c; })) { rw_ok = false; return; }
                    // HashedRWSet{hashed_reads = 1, hashed_writes = 2, metadata_writes = 3}
                    if (!scan_msg(base, hashed, BD_F(1) | BD_F(2) | BD_F(3), 0, [&](uint32_t g, Seg) { if (g == 2 || g == 3) writes = true; })) rw_ok = false;
                } })) { rw_ok = false; return; }
        if (!rw_ok) return;
        // KVRWSet{reads = 1, range_queries_info = 2, writes = 3, metadata_writes = 4}
        if (!scan_msg(base, kv, BD_F(1) | BD_F(2) | BD_F(3) | BD_F(4), 0, [&](uint32_t g, Seg) { if (g == 3 || g == 4) writes = true; })) { rw_ok = false; return; }
        if (n_seen < BD_MAX_NS_SEEN) { seen[n_seen] = name; wrote[n_seen] = writes; n_seen++; } else too_many = true;
    });
    if (!top_ok || !rw_ok) { tx.disp = TXC_BAD_RWSET; return; }
    if (!has_h_ccid || !has_r_ccid) { tx.disp = TXC_INVALID_OTHER_REASON; return; }
    if (h_name.len == 0 || !seg_equal(base, h_name, r_name) || r_ver.len == 0) { tx.disp = TXC_INVALID_CHAINCODE; return; }
    if (has_events) {                                                  // ChaincodeEvent{chaincode_id = 1 (string), tx_id = 2, event_name = 3, payload = 4}
        Seg ev_cc; ev_cc.off = ev_cc.len = 0;
        if (!scan_msg(base, events, BD_F(1) | BD_F(2) | BD_F(3) | BD_F(4), 0, [&](uint32_t f, Seg b) { if (f == 1) ev_cc = b; }) || !seg_equal(base, ev_cc, h_name)) {
            tx.disp = TXC_INVALID_OTHER_REASON; return;
        }
    }
    if (too_many) { tx.disp = TXC_NOT_VALIDATED; return; }              // more namespaces than the device tracks: CPU validator
    tx.wr_ns[0] = h_name; tx.n_ns = 1;
    for (uint32_t i = 0; i < n_seen; i++) {
        for (uint32_t j = 0; j < i; j++) if (seg_equal(base, seen[i], seen[j])) { tx.disp = TXC_ILLEGAL_WRITESET; return; }
    }
    for (uint32_t i = 0; i < n_seen; i++) {
        if (!wrote[i] || seg_equal(base, seen[i], h_name)) continue;
        if (tx.n_ns >= BD_MAX_NS) { tx.disp = TXC_NOT_VALIDATED; return; }
        tx.wr_ns[tx.n_ns++] = seen[i];
    }
}

// alloc_end(n) must return the first index of n fresh endorsement-job slots (atomicAdd on the device, a counter on the host)
template <typename Alloc>
BD_HD void walk_tx(const uint8_t* base, Seg env, uint32_t t, const uint8_t* channel, uint32_t channel_len, TxDev& tx, RawJob* raw,
                   JobArrays& ja, Alloc alloc_end)
{
    tx.early = TXC_NOT_VALIDATED; tx.htype = 0; tx.endorser_parse_ok = 0; tx.channel_ok = 0; tx.endorsements_parse_ok = 1; tx.overflow = 0;
    tx.disp = TXC_VALID; tx.n_ns = 0; tx.creator_identity = -1; tx.creator_has_job = 0; tx.first_end_job = 0; tx.n_end_jobs = 0;
    tx.txid_ascii.off = tx.txid_ascii.len = 0; tx.phash_claimed.off = tx.phash_claimed.len = 0;
    {
        ShaJobD z; for (int k = 0; k < 3; k++) { z.off[k] = 0; z.len[k] = 0; }
        ja.sha[t] = z; ja.sha[ja.J_cap + 2 * t] = z; ja.sha[ja.J_cap + 2 * t + 1] = z;
        raw[t].tx = 0xffffffffu; raw[t].k = -1;
    }
    Sel e = make_sel(1, 2);                                           // Envelope{payload=1, signature=2}
    if (!parse_sel(base, env, e)) { tx.early = TXC_INVALID_OTHER_REASON; return; }
    const Seg payload = e.s[0], signature = e.s[1];
    Sel p = make_sel(1, 2);                                           // Payload{header=1, data=2}
    if (!parse_sel(base, payload, p)) { tx.early = TXC_BAD_PAYLOAD; return; }
    if (!p.present[0]) { tx.early = TXC_BAD_COMMON_HEADER; return; }
    const Seg data = p.s[1]; const bool has_data = p.present[1];
    Sel h = make_sel(1, 2);                                           // Header{channel_header=1, signature_header=2}
    if (!parse_sel(base, p.s[0], h)) { tx.early = TXC_BAD_COMMON_HEADER; return; }
    const Seg chdr_b = h.s[0], shdr_b = h.s[1]; const bool has_chdr = h.present[0];
    Sel ch = make_sel(4, 5, 7, 1, 6);                                 // ChannelHeader{type=1, channel_id=4, tx_id=5, epoch=6, extension=7}
    if (!parse_sel(base, chdr_b, ch)) { tx.early = TXC_BAD_COMMON_HEADER; return; }
    Sel sh = make_sel(1, 2);                                          // SignatureHeader{creator=1, nonce=2}
    if (!parse_sel(base, shdr_b, sh)) { tx.early = TXC_BAD_COMMON_HEADER; return; }
    const Seg creator = sh.s[0], nonce = sh.s[1];
    const uint32_t ht = (uint32_t)ch.uv[0];
    if (!(ht == 1 || ht == 2 || ht == 3) || ch.uv[1] != 0 || nonce.len == 0 || creator.len == 0) { tx.early = TXC_BAD_COMMON_HEADER; return; }
    tx.htype = (uint8_t)ht;
    if (signature.len > 0 && payload.len > 0) {                       // creator job: slot t (identity resolved per job)
        raw[t].ident = creator; raw[t].sig = signature; raw[t].tx = t; raw[t].k = -1;
        ShaJobD& sj = ja.sha[t]; sj.off[0] = payload.off; sj.len[0] = payload.len;
        tx.creator_has_job = 1;
    }
    if (ht != 3) return;
    tx.txid_ascii = ch.s[1];
    { ShaJobD& a = ja.sha[ja.J_cap + 2 * t]; a.off[0] = nonce.off; a.len[0] = nonce.len; a.off[1] = creator.off; a.len[1] = creator.len; }
    tx.channel_ok = (ch.s[0].len == channel_len && bytes_equal(base + ch.s[0].off, channel, channel_len)) ? 1 : 0;
    if (!has_data) return;
    Seg action0; action0.off = action0.len = 0; uint32_t n_actions = 0;   // Transaction{repeated actions=1}: exactly one
    {
        Reader r; r.base = base; r.pos = data.off; r.end = data.off + data.len; r.ok = true;
        uint32_t f, wt; uint64_t v; Seg b;
        while (r.next(f, wt, v, b)) { if (f == 1) { if (wt != 2) { r.ok = false; break; } action0 = b; n_actions++; } }
        if (!r.ok || n_actions != 1) return;
    }
    Sel ta = make_sel(1, 2);                                          // TransactionAction{header=1, payload=2}
    if (!parse_sel(base, action0, ta)) return;
    Sel ah = make_sel(1, 2);
    if (!parse_sel(base, ta.s[0], ah) || ah.s[1].len == 0 || ah.s[0].len == 0) return;
    Sel cap = make_sel(1, 2);                                         // ChaincodeActionPayload{chaincode_proposal_payload=1, action=2}
    if (!parse_sel(base, ta.s[1], cap) || !cap.present[1]) return;
    Seg prp; prp.off = prp.len = 0; uint32_t n_end = 0; bool has_prp = false;   // ChaincodeEndorsedAction{prp=1, repeated endorsements=2}
    {
        Reader r; r.base = base; r.pos = cap.s[1].off; r.end = cap.s[1].off + cap.s[1].len; r.ok = true;
        uint32_t f, wt; uint64_t v; Seg b;
        while (r.next(f, wt, v, b)) {
            if (f == 1) { if (wt != 2) { r.ok = false; break; } prp = b; has_prp = true; }
            else if (f == 2) { if (wt != 2) { r.ok = false; break; } n_end++; }
        }
        if (!r.ok) return;
    }
    Sel pr = make_sel(1, 2);                                          // ProposalResponsePayload{proposal_hash=1, extension=2}
    if (!parse_sel(base, prp, pr)) return;
    if (!has_chdr || !ta.present[0] || !cap.present[0]) return;       // GetProposalHash2 "nil arguments"
    { ShaJobD& b = ja.sha[ja.J_cap + 2 * t + 1];
      b.off[0] = chdr_b.off; b.len[0] = chdr_b.len; b.off[1] = ta.s[0].off; b.len[1] = ta.s[0].len; b.off[2] = cap.s[0].off; b.len[2] = cap.s[0].len; }
    tx.phash_claimed = pr.s[0];
    tx.endorser_parse_ok = 1;
    dispatch_plan(base, ch.s[2], has_prp, pr.present[1], pr.s[1], tx);
    // endorsements: one pass to count those that carry a signature, one to emit their jobs (contiguous, in endorsement order)
    uint32_t n_jobs = 0;
    {
        Reader r; r.base = base; r.pos = cap.s[1].off; r.end = cap.s[1].off + cap.s[1].len; r.ok = true;
        uint32_t f, wt; uint64_t v; Seg b;
        while (r.next(f, wt, v, b)) {
            if (f != 2) continue;
            Sel en = make_sel(1, 2);                                  // Endorsement{endorser=1, signature=2}
            if (!parse_sel(base, b, en)) { tx.endorsements_parse_ok = 0; break; }
            // an endorsement without signature bytes can never verify: whatever its identity, it contributes nothing
            if (en.s[1].len > 0) n_jobs++;
        }
    }
    if (!tx.endorsements_parse_ok || n_jobs == 0) return;
    uint32_t j = alloc_end(n_jobs);
    if (j + n_jobs > ja.J_cap || j + n_jobs < j) { tx.overflow = 1; return; }          // job arrays full: this transaction goes to the CPU validator
    tx.first_end_job = j; tx.n_end_jobs = n_jobs;
    {
        Reader r; r.base = base; r.pos = cap.s[1].off; r.end = cap.s[1].off + cap.s[1].len; r.ok = true;
        uint32_t f, wt; uint64_t v; Seg b; int32_t k = 0;
        while (r.next(f, wt, v, b)) {
            if (f != 2) continue;
            Sel en = make_sel(1, 2);
            parse_sel(base, b, en);
            if (en.s[1].len == 0) continue;
            raw[j].ident = en.s[0]; raw[j].sig = en.s[1]; raw[j].tx = t; raw[j].k = k++;
            ShaJobD& sj = ja.sha[j];
            sj.off[0] = prp.off; sj.len[0] = prp.len; sj.off[1] = en.s[0].off; sj.len[1] = en.s[0].len; sj.off[2] = 0; sj.len[2] = 0;
            j++;
        }
    }
}

// One signature job: identity lookup in the MSP table, DER / low-S gate, operands for the verify kernel, and (creator jobs) the
// identity index written back into the transaction record.
BD_HD void resolve_job(const uint8_t* base, uint32_t j, const RawJob* raw, const MspDev& msp, JobArrays& ja, TxDev* txs)
{
    const RawJob rj = raw[j];
    int32_t identity = -1;
    bool ok = false;
    uint8_t rr[32], ss[32];
    if (rj.tx != 0xffffffffu) {
        identity = msp_find(msp, base + rj.ident.off, rj.ident.len);
        if (rj.k < 0) txs[rj.tx].creator_identity = identity;
        if (identity >= 0) ok = gate_signature(base + rj.sig.off, rj.sig.len, rr, ss);
    }
    uint32_t* r4 = reinterpret_cast<uint32_t*>(ja.r + 32 * (size_t)j);
    uint32_t* s4 = reinterpret_cast<uint32_t*>(ja.s + 32 * (size_t)j);
    for (int k = 0; k < 8; k++) {
        r4[k] = ok ? ((uint32_t)rr[4 * k] | ((uint32_t)rr[4 * k + 1] << 8) | ((uint32_t)rr[4 * k + 2] << 16) | ((uint32_t)rr[4 * k + 3] << 24)) : 0u;
        s4[k] = ok ? ((uint32_t)ss[4 * k] | ((uint32_t)ss[4 * k + 1] << 8) | ((uint32_t)ss[4 * k + 2] << 16) | ((uint32_t)ss[4 * k + 3] << 24)) : 0u;
    }
    ja.gate_ok[j] = ok ? 1 : 0;
    ja.identity[j] = identity;
    // creator jobs hash with the creator's MSP family, endorsement jobs with the endorser's: the identity that verifies the signature
    if (ja.kind) ja.kind[j] = (identity >= 0 && msp.hash_kind) ? msp.hash_kind[identity] : 0;
    const int32_t slot = (identity >= 0 && ok) ? msp.key_slot[identity] : -1;
    ja.key_slot[j] = slot;
    if (identity >= 0 && ok && slot == -1 && ja.qx) {
        for (int i = 0; i < 32; i++) { ja.qx[32 * (size_t)j + i] = msp.keys_xy[64 * (size_t)identity + i]; ja.qy[32 * (size_t)j + i] = msp.keys_xy[64 * (size_t)identity + 32 + i]; }
    }
}

// ---- policy evaluator: cauthdsl.go:24-92, `used` as a bit mask over at most BD_MAX_SIGNERS signers ------------------------
// Several policies share one node array (one tree per chaincode namespace); ns_* name the root of each.
struct PolicyDev {
    const int32_t* nodes; int32_t n_nodes; const int32_t* principal_code; int32_t n_principals;
    const uint8_t* ns_blob; const uint32_t* ns_off; const int32_t* ns_root; int32_t n_ns;     // n_ns = 0: one policy (root 0) for every namespace
};

BD_HD bool eval_policy(const PolicyDev& pol, int idx, const int32_t* signer_code, int n_signers, uint64_t& used, int depth)
{
    if (idx < 0 || idx >= pol.n_nodes || depth > 12) return false;
    const int32_t type = pol.nodes[4 * idx], n = pol.nodes[4 * idx + 1], first = pol.nodes[4 * idx + 2], cnt = pol.nodes[4 * idx + 3];
    if (type == 0) {
        int verified = 0;
        for (int c = first; c < first + cnt; c++) {
            uint64_t scratch = used;
            if (eval_policy(pol, c, signer_code, n_signers, scratch, depth + 1)) { verified++; used = scratch; }
        }
        return verified >= n;
    }
    if (n < 0 || n >= pol.n_principals) return false;
    const int32_t want = pol.principal_code[n];
    for (int i = 0; i < n_signers; i++) {
        if (used & (1ull << i)) continue;
        if (signer_code[i] < 0 || signer_code[i] != want) continue;
        used |= 1ull << i;
        return true;
    }
    return false;
}

// root node of namespace `ns`'s policy, -1 when the table has no chaincode definition for it
BD_HD int32_t policy_root(const PolicyDev& pol, const uint8_t* base, Seg ns)
{
    if (pol.n_ns == 0) return pol.n_nodes > 0 ? 0 : -1;
    for (int32_t i = 0; i < pol.n_ns; i++) {
        const uint32_t o = pol.ns_off[i], l = pol.ns_off[i + 1] - o;
        if (l != ns.len) continue;
        bool eq = true;
        for (uint32_t k = 0; k < l && eq; k++) eq = pol.ns_blob[o + k] == base[ns.off + k];
        if (eq) return pol.ns_root[i];
    }
    return -1;
}

// ---- per-transaction decision ---------------------------------------------------------------------------------------------
// sig_ok(j): signature job j verified (gate and curve).  job_identity: JobArrays::identity.  digests: 32 bytes per SHA job.
// An identity the table does not hold, or a namespace without a policy entry, cannot be decided here: TXC_NOT_VALIDATED hands the
// transaction to the CPU validator (the reference deserialises and validates ANY certificate of the channel's CAs,
// msgvalidation.go:40-57, and reads chaincode definitions from the ledger, dispatcher.go:224-277).
template <typename SigOk>
BD_HD uint8_t decide_tx(const uint8_t* base, const TxDev& tx, uint32_t t, const MspDev& msp, const PolicyDev& pol, SigOk sig_ok,
                        const int32_t* job_identity, const uint8_t* digests, uint32_t J_cap, uint64_t* txid_hash_out)
{
    const char hex[] = "0123456789abcdef";
    if (tx.early != TXC_NOT_VALIDATED) return tx.early;
    if (!tx.creator_has_job) return TXC_BAD_CREATOR_SIGNATURE;        // "nil arguments"
    if (tx.creator_identity < 0) return TXC_NOT_VALIDATED;            // not in the device's MSP table
    if (!msp.valid[tx.creator_identity] || !sig_ok(t)) return TXC_BAD_CREATOR_SIGNATURE;
    if (tx.htype == 1) return TXC_NOT_VALIDATED;                      // config transaction: CPU validator
    if (tx.htype != 3) return TXC_UNSUPPORTED_TX_PAYLOAD;
    {
        const uint8_t* dg = digests + 32 * (size_t)(J_cap + 2 * t);
        bool same = tx.txid_ascii.len == 64;
        for (int k = 0; same && k < 32; k++)
            same = base[tx.txid_ascii.off + 2 * k] == (uint8_t)hex[dg[k] >> 4] && base[tx.txid_ascii.off + 2 * k + 1] == (uint8_t)hex[dg[k] & 15];
        if (!same) return TXC_BAD_PROPOSAL_TXID;
    }
    if (!tx.endorser_parse_ok) return TXC_INVALID_ENDORSER_TRANSACTION;
    if (tx.phash_claimed.len != 32 || !bytes_equal(base + tx.phash_claimed.off, digests + 32 * (size_t)(J_cap + 2 * t + 1), 32))
        return TXC_INVALID_ENDORSER_TRANSACTION;
    if (!tx.channel_ok) return TXC_TARGET_CHAIN_NOT_FOUND;
    if (tx.disp != TXC_VALID) return tx.disp;                         // the plugin dispatcher's own checks
    if (!tx.endorsements_parse_ok) return TXC_INVALID_OTHER_REASON;
    if (tx.overflow) return TXC_NOT_VALIDATED;                        // job arrays were full: CPU validator
    int32_t roots[BD_MAX_NS];
    for (int i = 0; i < tx.n_ns; i++) {
        roots[i] = policy_root(pol, base, tx.wr_ns[i]);
        if (roots[i] < 0) return TXC_NOT_VALIDATED;                   // no chaincode definition on the device
    }
    // SignatureSetToValidIdentities (policy.go:365-402): in order; de-duplicated by Mspid + Id against the identities that already
    // VERIFIED; a failed signature drops that entry only.  One set per transaction, shared by every namespace's evaluation.
    int32_t signer_code[BD_MAX_SIGNERS]; int n_signers = 0;
    for (uint32_t i = 0; i < tx.n_end_jobs; i++) {
        const uint32_t j = tx.first_end_job + i;
        const int32_t idn = job_identity[j];
        if (idn < 0) return TXC_NOT_VALIDATED;
        const int32_t grp = msp.group ? msp.group[idn] : idn;
        bool dup = false;
        for (uint32_t i2 = 0; i2 < i && !dup; i2++) {
            const uint32_t j2 = tx.first_end_job + i2;
            const int32_t id2 = job_identity[j2];
            dup = (msp.group ? msp.group[id2] : id2) == grp && sig_ok(j2);
        }
        if (dup) continue;
        if (!sig_ok(j)) continue;
        if (n_signers >= BD_MAX_SIGNERS) return TXC_NOT_VALIDATED;
        signer_code[n_signers++] = msp.valid[idn] ? msp.msp_code[idn] : -1;
    }
    for (int i = 0; i < tx.n_ns; i++) {
        uint64_t used = 0;
        if (!eval_policy(pol, roots[i], signer_code, n_signers, used, 0)) return TXC_ENDORSEMENT_POLICY_FAILURE;
    }
    uint64_t hsh = 1469598103934665603ull;
    for (uint32_t k = 0; k < tx.txid_ascii.len; k++) hsh = (hsh ^ base[tx.txid_ascii.off + k]) * 1099511628211ull;
    *txid_hash_out = hsh;
    return TXC_VALID;
}

} }  // namespace fabgpu::bdev
