/* fabgpu_ecdsa.h -- C ABI of the B200 batch ECDSA-P256 verifier (libfabgpu_ecdsa.so).
 *
 * Drop-in boundary for ONE path of trustbloc/fabric-mod: signature verification behind
 *     bccsp.BCCSP.Verify(k, signature, digest, opts) (bool, error)         reference bccsp/bccsp.go:123-125
 * as implemented by the software provider
 *     sw.CSP.Verify -> verifyECDSA -> crypto/ecdsa.Verify                   reference bccsp/sw/impl.go:247-270,
 *                                                                           bccsp/sw/ecdsa.go:41-57
 * and reached from msp identity.Verify (reference msp/identities.go:169-196).  The reference has no native
 * code on this path; these entry points are what a cgo provider (INTEGRATION.md, go/bccsp/gpu) binds, in the
 * same way bccsp/pkcs11 binds an HSM library (reference bccsp/pkcs11/pkcs11.go:36-87,241-262).
 *
 * Conventions
 *   - plain pointers and sizes only; no CUDA or torch types.  `cuda_stream` arguments are a cudaStream_t
 *     passed as void* (NULL = CUDA's default stream, as in the runtime API).
 *   - every function returns FABGPU_OK (0) or a negative FABGPU_E_* code.  A negative code means "could not
 *     decide": the caller MUST fall back to the CPU provider for that batch.  A device fault is never
 *     reported as "signature invalid" (SURVEY.md section 5: that would fork the ledger).
 *   - big integers cross the boundary as 32-byte big-endian strings, structure-of-arrays: element i of an
 *     array lives at bytes [32*i, 32*i+32).
 *   - validity bitmask: signature i -> bit (i % 32) of uint32 word (i / 32); 1 = VALID, i.e. (true, nil).
 *   - there is NO CPU fallback inside this library: without a usable CUDA device fabgpu_init fails.
 */
#ifndef FABGPU_ECDSA_H
#define FABGPU_ECDSA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct fabgpu_ctx fabgpu_ctx;

enum {
    FABGPU_OK = 0,
    FABGPU_E_NO_DEVICE = -1,   /* no CUDA device / driver, or device id out of range */
    FABGPU_E_CUDA = -2,        /* a CUDA call failed; see fabgpu_last_error */
    FABGPU_E_ARG = -3,         /* bad argument (NULL, n > max_batch, bad slot ...) */
    FABGPU_E_INJECTED = -4     /* FABGPU_FAULT_INJECT=1 is set: every verify call fails (fault-injection tests) */
};

/* Per-signature status of the bccsp-level entry points: the (bool, error) pair of sw.CSP.Verify as one byte.
 * Error kinds follow reference bccsp/sw/impl.go:249-266, bccsp/sw/ecdsa.go:42-54, bccsp/utils/ecdsa.go:43-92. */
enum {
    FABGPU_ST_VALID = 0,              /* (true,  nil) */
    FABGPU_ST_INVALID = 1,            /* (false, nil): well-formed but wrong, incl. r >= N, point at infinity */
    FABGPU_ST_ERR_NIL_KEY = 2,        /* "Invalid Key. It must not be nil." */
    FABGPU_ST_ERR_EMPTY_SIG = 3,      /* "Invalid signature. Cannot be empty." */
    FABGPU_ST_ERR_EMPTY_DIGEST = 4,   /* "Invalid digest. Cannot be empty." */
    FABGPU_ST_ERR_UNMARSHAL = 5,      /* "Failed unmashalling signature [...]" (asn1) */
    FABGPU_ST_ERR_R_NOT_POSITIVE = 6, /* "invalid signature, R must be larger than zero" */
    FABGPU_ST_ERR_S_NOT_POSITIVE = 7, /* "invalid signature, S must be larger than zero" */
    FABGPU_ST_ERR_HIGH_S = 8,         /* "Invalid S. Must be smaller than half the order [..][..]." */
    FABGPU_ST_ERR_UNSUPPORTED_KEY = 9,/* not a P-256 key: delegate to the embedded sw provider */
    FABGPU_ST_ERR_OFF_CURVE = 10      /* public key is not a curve point: outside the reference's defined behaviour, delegate to CPU */
};

/* ---- lifetime ---------------------------------------------------------------------------------------- */

/* Creates a context on the given CUDA devices (device_ids == NULL && n_dev == 0: device 0).  Allocates, per
 * device, the fixed-base table, device SoA buffers and pinned host SoA buffers for `max_batch` signatures per
 * slot (FABGPU_SLOTS slots), and builds the table on the device.  A batch given to the host-buffer entry points
 * is split into contiguous, 32-aligned ranges across the context's devices. */
int fabgpu_init(const int* device_ids, int n_dev, size_t max_batch, fabgpu_ctx** out);
void fabgpu_destroy(fabgpu_ctx* ctx);
/* Last error text of this context (or of the failed fabgpu_init when ctx == NULL). Never NULL. */
const char* fabgpu_last_error(const fabgpu_ctx* ctx);
int fabgpu_device_count(const fabgpu_ctx* ctx);
size_t fabgpu_max_batch(const fabgpu_ctx* ctx);

#define FABGPU_SLOTS 3

/* ---- leaf: pre-gated SoA tuples -> bitmask (replaces the crypto/ecdsa.Verify call at bccsp/sw/ecdsa.go:56) */

/* Pinned, library-owned host SoA buffers of one slot (cgo cannot hand Go memory to an async copy).  Each of
 * qx,qy,e,r,s has max_batch*32 bytes; mask and offcurve have ceil(max_batch/32) words.  Caller pre-conditions,
 * established by the host gates exactly as the reference does before calling ecdsa.Verify: 0 < r, 0 < s <= N/2,
 * r < 2^256 (longer r is INVALID without asking the GPU), e = leftmost min(len,32) digest bytes left-padded. */
int fabgpu_host_buffers(fabgpu_ctx* ctx, int slot, uint8_t** qx, uint8_t** qy, uint8_t** e, uint8_t** r,
                        uint8_t** s, uint32_t** mask, uint32_t** offcurve);
/* H2D + kernel + D2H for the first n tuples of the slot's pinned buffers; synchronous. */
int fabgpu_verify_p256(fabgpu_ctx* ctx, int slot, size_t n);
/* Same, asynchronous: returns after enqueueing; fabgpu_wait blocks until the slot's mask is complete. */
int fabgpu_verify_p256_async(fabgpu_ctx* ctx, int slot, size_t n);
int fabgpu_wait(fabgpu_ctx* ctx, int slot);
/* Convenience for callers whose tuples sit in ordinary host memory: copies through slot 0. */
int fabgpu_verify_p256_host(fabgpu_ctx* ctx, const uint8_t* qx, const uint8_t* qy, const uint8_t* e,
                            const uint8_t* r, const uint8_t* s, size_t n, uint32_t* mask, uint32_t* offcurve);
/* Inputs and outputs already resident in the memory of context device `dev_index`; enqueues on `cuda_stream`
 * and returns without synchronising.  offcurve may be NULL. */
int fabgpu_verify_p256_device(fabgpu_ctx* ctx, int dev_index, const void* d_qx, const void* d_qy, const void* d_e,
                              const void* d_r, const void* d_s, size_t n, void* d_mask, void* d_offcurve,
                              void* cuda_stream);

/* ---- per-key fixed-base tables (SURVEY.md section 8f rank 4; what KeyImport does once per identity) -----------
 * Identities repeat heavily in Fabric (the reference caches them: msp/cache/cache.go:38-129; keys are imported once,
 * bccsp/sw/keyimport.go:114-134, msp/mspimpl.go:420).  A registered key gets a window table on every device of the
 * context, after which u2*Q is fixed-base like u1*G.  Results are identical to the generic kernel; only speed differs. */

/* Looks up / builds tables for K keys (X||Y, 64 bytes each).  slots_out[k] >= 0 is the key's HANDLE
 * ((generation << 12) | slot); -1 means "no table" (not a curve point, or more distinct keys than
 * fabgpu_key_slot_capacity in one call) -- such signatures simply take the generic kernel.  Least-recently-used slots are
 * recycled; a handle issued before its slot was recycled is detected by the pinned-slot entry points and treated as -1,
 * so a stale handle costs speed, never correctness.  Capacity: env FABGPU_KEY_SLOTS (default 256, at most 4096). */
int fabgpu_keys_register(fabgpu_ctx* ctx, const uint8_t* keys_xy, int K, int32_t* slots_out);
int fabgpu_key_slot_capacity(const fabgpu_ctx* ctx);
/* The tier between "never seen" and a window table: a SMALL table (33 windows of signed 8-bit digits, 264 KiB, built in
 * about 1.5 us of GPU time) makes u2*Q 33 mixed additions and no doublings.  Meant for keys that recur without being busy -- client /
 * creator certificates, thousands of identities with a few signatures per block each (the reference caches exactly those identities:
 * msp/cache/cache.go:38-129).  handles_out[k] <= -2 is the key's small HANDLE (-2 - ((generation << 20) | slot)), -1 = no slot could
 * be had; every entry point that takes key handles accepts both kinds.  A key that is not a curve point still gets a handle: its
 * signatures are reported off-curve, exactly as by the generic kernel.  The build is enqueued, not waited for; consumers are ordered
 * behind it on the device.  fabgpu_bccsp_verify_batch* give a key a small table by themselves once FABGPU_SMALL_MIN_USES (default 32: the
 * point where the key has cost as much on the generic kernel as its table does) of its signatures have been seen without a window table; fabgpu_msp_configure uses small tables when the MSP holds more identities
 * than window-table slots.  Capacity: env FABGPU_SMALL_SLOTS (default 16 384 = 4.4 GB per device; 0 turns the tier off); least recently
 * used tables are recycled in bulk (stale handles are detected like the big ones). */
int fabgpu_keys_register_small(fabgpu_ctx* ctx, const uint8_t* keys_xy, int K, int32_t* handles_out);
int fabgpu_small_slot_capacity(const fabgpu_ctx* ctx);
/* Build constants of the small tables: signed window width in bits, number of windows, bytes per table. */
void fabgpu_small_table_info(int* window_bits, int* windows, size_t* table_bytes);
/* out[0] = window tables alive, out[1] = small tables alive, out[2] = small tables built so far, out[3] = small tables recycled. */
int fabgpu_key_table_stats(fabgpu_ctx* ctx, unsigned long long out[4]);
/* Pinned int32[max_batch] of one slot: key_slot[i] = handle of signature i's key (from fabgpu_keys_register), or -1.
 * Only the _keyed entry points read it (they replace handles by live slot indices in place); callers overwrite all n
 * entries per batch and still fill Qx/Qy, which the generic kernel uses whenever a handle is -1 or stale. */
int fabgpu_host_key_slots(fabgpu_ctx* ctx, int slot, int32_t** key_slot);
int fabgpu_verify_p256_keyed(fabgpu_ctx* ctx, int slot, size_t n);
int fabgpu_verify_p256_keyed_async(fabgpu_ctx* ctx, int slot, size_t n);
/* Device-resident form: d_key_slot holds raw slot indices (handle & 0xfff) that the caller obtained from
 * fabgpu_keys_register and knows to be live: RAW slots are not re-validated, so the caller must not let a registration that could
 * recycle them (fabgpu_keys_register of new keys, fabgpu_msp_configure, a fabgpu_bccsp_verify_batch* call that tables new keys) run
 * between obtaining the slots and the completion of this launch.  The handle-taking entry points (fabgpu_verify_p256_keyed*,
 * fabgpu_bccsp_verify_batch*, fabgpu_validate_*) hold the library's slot-table lock from resolution to enqueue and need no such care.
 * all_cached = 1 promises every d_key_slot[i] >= 0 (d_qx/d_qy may then be NULL); all_cached = 2 promises every d_key_slot[i] <= -2,
 * the raw code of a small table: -2 - (slot bits of a small handle, i.e. (-2 - handle) & 0xfffff); all_cached = 0: any mix (this form has
 * no compaction scratch: every signature without a WINDOW table -- codes -1 and <= -2 alike -- goes through the generic arithmetic
 * and reads d_qx/d_qy). */
int fabgpu_verify_p256_device_keyed(fabgpu_ctx* ctx, int dev_index, int all_cached, const void* d_key_slot, const void* d_qx,
                                    const void* d_qy, const void* d_e, const void* d_r, const void* d_s, size_t n,
                                    void* d_mask, void* d_offcurve, void* cuda_stream);

/* ---- validity bitmask across GPUs driven by separate processes (one process per GPU, SURVEY.md section 8e) ----------------
 * The reference has no counterpart (its verifier is per-signature, bccsp/sw/ecdsa.go:41-57); BASELINE.json's north_star asks for
 * the batch to be split across the GPUs of a box and the bitmask to be reassembled.  The consumer of the bitmask is the HOST
 * (the Go provider reads it from pinned memory), so the single-process form (one context, several devices: fabgpu_verify_p256*)
 * needs no device-to-device collective at all.  For the one-process-per-GPU form the library exchanges the mask words itself,
 * over peer memory: every rank creates a receive buffer and exports it (CUDA IPC), maps the others', and the verify kernel's
 * epilogue stores each ballot word into the buffer of every rank (P2P writes over NVLink / NVSwitch), followed by a step flag;
 * a wait kernel on the same stream returns when all ranks' words of that step have landed.  No NCCL call on the data path
 * (fabric-mod_b200/sharding.py keeps the NCCL all-gather as the alternative).
 *   _create: this rank's buffer for `world` ranks x words_per_rank mask words; writes its IPC handle (FABGPU_IPC_HANDLE_BYTES).
 *   _open:   handles = world x FABGPU_IPC_HANDLE_BYTES bytes, rank-major (the caller exchanges them, e.g. over its process group).
 *   _allgather: fabgpu_verify_p256_device_keyed for this rank's n signatures (n <= 32 x words_per_rank), then the exchange;
 *            `step` must be 1, 2, 3, ... in lock step on all ranks; *d_full_mask = device pointer to world x words_per_rank
 *            words, valid once the stream has run (until step + 2 is launched: two generations).  A peer that never publishes
 *            makes the NEXT call fail with FABGPU_E_CUDA instead of hanging the GPU. */
#define FABGPU_IPC_HANDLE_BYTES 64
int fabgpu_peer_mask_create(fabgpu_ctx* ctx, int dev_index, int world, int rank, size_t words_per_rank,
                            uint8_t handle_out[FABGPU_IPC_HANDLE_BYTES]);
int fabgpu_peer_mask_open(fabgpu_ctx* ctx, int dev_index, const uint8_t* handles);
int fabgpu_peer_mask_close(fabgpu_ctx* ctx, int dev_index);
int fabgpu_verify_p256_device_keyed_allgather(fabgpu_ctx* ctx, int dev_index, int all_cached, const void* d_key_slot,
                                              const void* d_qx, const void* d_qy, const void* d_e, const void* d_r,
                                              const void* d_s, size_t n, uint32_t step, void** d_full_mask, void* cuda_stream);

/* ---- bccsp level: raw DER signatures + digests + keys -> three-valued status (sw.CSP.Verify semantics) -- */

/* keys_xy: K x 64 bytes (X || Y, big-endian).  key_idx[i] in [0,K), or < 0 for a nil key.  digests / sigs are
 * concatenations indexed by (n+1)-entry offset tables.  status[i] receives FABGPU_ST_*.  The gates (DER per Go
 * encoding/asn1, positivity, low-S, r < 2^256) run in a kernel in front of the verify kernel (on the context's host
 * threads for multi-device contexts or with FABGPU_BCCSP_HOST_GATES=1); survivors are verified.  Keys used by at least
 * FABGPU_KEY_MIN_USES (env, default 256; negative disables) signatures of the call get a window table automatically.
 * A call of >= 24576 signatures is cut into one chunk per slot internally when all slots are free. */
int fabgpu_bccsp_verify_batch(fabgpu_ctx* ctx, const uint8_t* keys_xy, int K, const int32_t* key_idx,
                              const uint8_t* digests, const uint32_t* dig_off, const uint8_t* sigs,
                              const uint32_t* sig_off, size_t n, uint8_t* status);
/* The same call in two halves, for a caller that keeps the GPU fed (the Go provider's aggregator): _async stages the
 * batch into the slot's pinned buffers and enqueues copies + kernels + the status read-back on the slot's stream, then
 * returns -- the caller's arrays are not referenced afterwards; _wait blocks until that batch is done and writes its n
 * status bytes.  With the FABGPU_SLOTS slots used round-robin, the staging and copies of the next batches overlap the kernels of batch i.
 * A slot holds one batch at a time (FABGPU_E_ARG otherwise); fabgpu_bccsp_verify_batch itself is _async + _wait on slot 0. */
int fabgpu_bccsp_verify_batch_async(fabgpu_ctx* ctx, int slot, const uint8_t* keys_xy, int K, const int32_t* key_idx,
                                    const uint8_t* digests, const uint32_t* dig_off, const uint8_t* sigs,
                                    const uint32_t* sig_off, size_t n);
int fabgpu_bccsp_verify_batch_wait(fabgpu_ctx* ctx, int slot, uint8_t* status, size_t n);
/* Zero-copy form of the pair above (what the Go provider's block pre-pass and bench.py's e2e leg use): the library hands out
 * the slot's PINNED staging buffers, the caller writes the batch there -- keys (K x 64 B), key index per signature, digest and
 * DER blobs with their offset tables (offsets start at 0) -- and _inplace_async enqueues the copies and kernels straight from
 * them; no second host copy, no staging threads.  The buffers stay valid (and keep their contents) until a later
 * fabgpu_bccsp_batch_buffers call asks for larger capacities; they must not be rewritten while the slot's batch is in flight.
 * Single-device contexts; completion and statuses through fabgpu_bccsp_verify_batch_wait. */
int fabgpu_bccsp_batch_buffers(fabgpu_ctx* ctx, int slot, size_t n_cap, size_t sig_bytes_cap, size_t dig_bytes_cap, int k_cap,
                               uint8_t** keys_xy, int32_t** key_idx, uint8_t** digests, uint32_t** dig_off, uint8_t** sigs,
                               uint32_t** sig_off);
int fabgpu_bccsp_verify_batch_inplace_async(fabgpu_ctx* ctx, int slot, int K, size_t n);
/* Single call with the reference's exact error strings (sw.CSP.Verify).  key_xy == NULL is the nil key.
 * *valid and err (NUL-terminated, truncated to errcap) mirror the Go (bool, error) pair; err[0] == 0 is nil. */
int fabgpu_bccsp_verify(fabgpu_ctx* ctx, const uint8_t* key_xy, const uint8_t* sig, size_t sig_len,
                        const uint8_t* digest, size_t digest_len, int* valid, char* err, size_t errcap);
/* The host gate alone (no GPU): parses one DER signature the way utils.UnmarshalECDSASignature + IsLowS do and,
 * on success, writes r and s as 32-byte big-endian.  Returns a FABGPU_ST_* code: FABGPU_ST_VALID means "gates
 * passed, ask the GPU"; FABGPU_ST_INVALID means r >= 2^256 (cannot be < N). */
int fabgpu_gate_signature(const uint8_t* sig, size_t sig_len, uint8_t r_out[32], uint8_t s_out[32]);

/* ---- block level: the signature pre-pass of TxValidator.Validate (SURVEY.md section 8a rows a11-a14, 8f ranks 1-2) ----
 * One call verifies every signature of a serialized common.Block as ONE GPU batch -- creator signatures
 * (core/common/validation/msgvalidation.go:26-64) and endorsement signatures (statebased/validator_keylevel.go:243-259,
 * common/policies/policy.go:365-402) -- with the SHA-256 of each signed message computed on the device straight from the
 * block bytes, then replays the reference's per-transaction decision order (msgvalidation.go:248-320, v20/validator.go:
 * 300-455, cauthdsl.go:24-92, markTXIdDuplicates) and writes the TRANSACTIONS_FILTER bytes (peer.TxValidationCode).
 * Outside the pre-pass, exactly as mocked in the reference's unit tests: ledger lookups, chaincode definitions, rw-sets,
 * key-level policies.  Config transactions are flagged 254 (NOT_VALIDATED) and must be validated by the CPU validator. */

/* Installs the MSP view and the endorsement policy used by fabgpu_validate_block.
 * identities: n_ids serialized msp.SerializedIdentity byte strings (id_blob + (n_ids+1) offsets) exactly as they appear in
 * SignatureHeader.creator / Endorsement.endorser, their MSP ids, P-256 keys (X||Y) and the outcome of identity.Validate().
 * policy_nodes: n_nodes x 4 int32 (type, n, first_child, n_children); type 0 = NOutOf(n) over children
 * [first_child, first_child + n_children), type 1 = SignedBy(principal n); node 0 is the root.  Principals are MSP ids
 * (ROLE member).  Every identity's key gets a window table when the MSP fits the window-table pool (n_ids <= fabgpu_key_slot_capacity);
 * a larger MSP -- thousands of client certificates -- goes to the small tier instead, except the identities whose key already owns a
 * window table: register the few busy keys (the endorsing peers) with fabgpu_keys_register BEFORE this call and they keep it. */
int fabgpu_msp_configure(fabgpu_ctx* ctx, const uint8_t* id_blob, const uint32_t* id_off, const uint8_t* mspid_blob,
                         const uint32_t* mspid_off, const uint8_t* keys_xy, const uint8_t* valid, int n_ids,
                         const int32_t* policy_nodes, int n_nodes, const uint8_t* principal_blob, const uint32_t* principal_off,
                         int n_principals, const char* channel_id);
/* Two optional refinements of the table fabgpu_msp_configure installed (call them after it; each drains the block slots first):
 *   _identity_groups: group[i] = de-duplication id of identity i.  The reference de-duplicates a transaction's signers on
 *       Mspid + certificate digest (common/policies/policy.go:380-386), so two byte-different serializations of ONE certificate
 *       must share a group; without this call every table entry is its own group.
 *   _namespace_policies: the endorsement policy of each chaincode namespace (what the plugin dispatcher looks up per namespace a
 *       transaction writes to, core/committer/txvalidator/v20/plugindispatcher/dispatcher.go:166-221,265-277): ns_root[i] is the
 *       root node -- an index into the node array given to fabgpu_msp_configure, which may hold several trees -- of namespace i's
 *       policy.  n_ns = 0 restores "node 0 is the policy of every namespace".  A transaction that needs a namespace without an
 *       entry is flagged 254 (NOT_VALIDATED): the CPU validator reads the chaincode definition from the ledger. */
int fabgpu_msp_identity_groups(fabgpu_ctx* ctx, const int32_t* group, int n_ids);
int fabgpu_namespace_policies(fabgpu_ctx* ctx, const uint8_t* ns_blob, const uint32_t* ns_off, const int32_t* ns_root, int n_ns);
/* A third refinement, called the same way: the hash each MSP's identities sign with.  identity.Verify hashes the signed message
 * with the SignatureHashFamily of the signer's MSP configuration (FabricMSPConfig.CryptoConfig.SignatureHashFamily;
 * msp/identities.go:169-196,216-224): "SHA2" -> SHA-256, "SHA3" -> SHA3-256.  family[i] (FABGPU_HASH_SHA2 or FABGPU_HASH_SHA3)
 * is the family of MSP i (mspid_blob + (n_msps+1) offsets); each creator signature is hashed with the creator's family, each
 * endorsement signature with the endorser's.  MSPs not listed stay SHA2; n_msps = 0 restores all-SHA2, and so does every
 * fabgpu_msp_configure.  The tx-id check (protoutil/proputils.go:355-364) and the proposal hash (protoutil/txutils.go:431-448)
 * are SHA-256 whatever the family.  FABGPU_E_ARG (with fabgpu_last_error) for a family code other than the two, an MSP id
 * that no identity of the table carries, or one MSP listed twice with different families. */
#define FABGPU_HASH_SHA2 0
#define FABGPU_HASH_SHA3 1
int fabgpu_msp_hash_families(fabgpu_ctx* ctx, const uint8_t* mspid_blob, const uint32_t* mspid_off, const uint8_t* family, int n_msps);
/* flags[i] receives the validation code of transaction i; *n_tx_out the number of transactions. */
int fabgpu_validate_block(fabgpu_ctx* ctx, const uint8_t* block, size_t block_len, uint8_t* flags, size_t flags_cap, size_t* n_tx_out);
/* Same for a caller that already holds Block.Data.Data as separate byte strings (the Go validator does): `blob` is their
 * concatenation, env_off the (n_env+1)-entry offset table.  Saves the serial walk over the length-prefixed envelopes. */
int fabgpu_validate_envelopes(fabgpu_ctx* ctx, const uint8_t* blob, const uint32_t* env_off, size_t n_env, uint8_t* flags, size_t flags_cap,
                              size_t* n_tx_out);
/* Both calls in two halves over the FABGPU_SLOTS slots, for a committer that keeps several blocks in flight: _async enqueues
 * the copy and every kernel of the block on the slot's stream and returns; fabgpu_validate_wait blocks until the slot's
 * block is done, runs the duplicate-tx-id pass and writes the flags.  The block bytes must stay valid and unchanged until
 * the wait returns (they are copied by DMA and read again by the duplicate pass).  While the GPU works on block k, the
 * copy of block k+1 proceeds: the PCIe transfer (the largest single phase of a block) is hidden across blocks.
 * fabgpu_validate_block / _envelopes are _async + _wait on slot 0. */
int fabgpu_validate_block_async(fabgpu_ctx* ctx, int slot, const uint8_t* block, size_t block_len);
int fabgpu_validate_envelopes_async(fabgpu_ctx* ctx, int slot, const uint8_t* blob, const uint32_t* env_off, size_t n_env);
int fabgpu_validate_wait(fabgpu_ctx* ctx, int slot, uint8_t* flags, size_t flags_cap, size_t* n_tx_out);
/* Optional pinned staging buffer for the block bytes (the H2D copy of a pageable buffer is several times slower); one per slot. */
int fabgpu_block_buffer(fabgpu_ctx* ctx, size_t bytes, uint8_t** out);                      /* slot 0 */
int fabgpu_block_buffer_slot(fabgpu_ctx* ctx, int slot, size_t bytes, uint8_t** out);
/* Times of the last completed block, microseconds.  [0..4] host wall clock: enqueue, (unused), wait for the device,
 * duplicate-tx-id pass, total from submit to flags.  [5..9] CUDA-event times of the device stages (FABGPU_BLOCK_EVENTS=1):
 * H2D + walk + creator resolve + SHA-256, (unused), endorsement resolve + SHA-256, verify kernel(s), block_decide_kernel.
 * (With a SHA3 MSP in the table the hash stages include the SHA3-256 launches.) */
int fabgpu_block_timing(const fabgpu_ctx* ctx, double out_us[10]);
/* Device SHA-256 of messages given as up to three byte ranges of `buf` each: jobs = n x {off0,off1,off2,len0,len1,len2}
 * (uint32); digests = n x 32 bytes.  (The hash msp identity.Verify computes first: msp/identities.go:178.) */
int fabgpu_sha256_segments(fabgpu_ctx* ctx, const uint8_t* buf, size_t buf_len, const uint32_t* jobs, size_t n, uint8_t* digests);
/* The same for SHA3-256 (FIPS 202), the digest of identity.Verify for an MSP whose SignatureHashFamily is SHA3. */
int fabgpu_sha3_256_segments(fabgpu_ctx* ctx, const uint8_t* buf, size_t buf_len, const uint32_t* jobs, size_t n, uint8_t* digests);

/* ---- test / bring-up hooks ------------------------------------------------------------------------------ */
/* Device field primitives on arrays (op: 0 fe_mul, 1 fe_add, 2 fe_sub, 3 sc_mul, 4 fe_inv,
 * 5 sc_inv_to_mont by Fermat, 6 the same by division steps, 7 fe_sqr). */
int fabgpu_test_fieldop(fabgpu_ctx* ctx, int op, const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out);
/* Sampled entries of a device window table: out[i] (64 bytes: X then Y, Montgomery form, little-endian 32-bit limbs) =
 * entry (window[i], digit[i]) = digit * 2^(w * window) * P, digit in [1, 2^w).  key_slot < 0: the generator's table
 * (w = g_window_bits of fabgpu_build_info); otherwise the table in that raw key slot (w = key_window_bits). */
int fabgpu_test_table_entries(fabgpu_ctx* ctx, int key_slot, const uint32_t* window, const uint32_t* digit, size_t n, uint8_t* out);
/* Phase times of the last fabgpu_bccsp_verify_batch call, microseconds: [0] key-table lookup/registration,
 * [1] staging copy into pinned memory (host gates + packing on the host-gated path), [2] H2D + kernels + D2H (enqueue to
 * completion), [3] status copy-out.  For metrics export
 * (the reference only has a block-level histogram, gossip/metrics/metrics.go:187-194). */
int fabgpu_last_timing(const fabgpu_ctx* ctx, double out_us[4]);
/* Compile-time table shapes: window bits of the fixed-base table of G and of the per-key tables. */
void fabgpu_build_info(int* g_window_bits, int* key_window_bits);
/* Kernel launches issued by this context so far (bench.py's gpu_launches). */
unsigned long long fabgpu_launch_count(const fabgpu_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* FABGPU_ECDSA_H */
