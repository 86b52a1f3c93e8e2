// C-ABI shim of libfabgpu_ecdsa.so (declared in include/fabgpu_ecdsa.h): context, pinned SoA slots, multi-device
// batch split, kernel launches.  No CPU verification fallback lives here by design: a failure is reported to the
// caller, who falls back to the reference's software provider (SURVEY.md section 5).
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <memory>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <shared_mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../../include/fabgpu_ecdsa.h"
#include "bccsp_host.hpp"
#include "blockval.hpp"
#include "sha256.cuh"
#include "sha3.cuh"
#include "blockdev_kernels.cuh"
#include "ecdsa_kernels.cuh"

#if defined(__SSE2__)
#include <emmintrin.h>
#endif

using namespace fabgpu;

namespace {

std::string g_init_error = "";

struct DevSlot {
    cudaStream_t stream = nullptr;
    uint8_t* d_in[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // qx qy e r s
    uint32_t* d_mask = nullptr;
    uint32_t* d_off = nullptr;
    int32_t* d_key_slot = nullptr;
    uint32_t* d_idx = nullptr;      // dev_cap + 2 words: compaction scratch of mixed batches
};

struct Device {
    int id = 0;
    aff* gtab = nullptr;
    int sms = 148;            // multiprocessors (launch shapes)
    aff* qtab = nullptr;      // key_slots tables of FAB_G_WINDOWS * FAB_G_ENTRIES points (per-key fixed-base tables)
    // small key tables (FAB_S_POINTS points each): the pool, the build scratch (grown on demand) and the build stream.  Every
    // enqueue that may read a small table first makes its stream wait for s_ev (the last build): builds are ordered among
    // themselves by s_stream, so one event covers all earlier ones.
    aff* stab = nullptr;
    aff* s_bases = nullptr; uint8_t* s_keys = nullptr; int32_t* s_slots = nullptr; size_t s_cap = 0;
    cudaStream_t s_stream = nullptr; cudaEvent_t s_ev = nullptr; bool s_ev_set = false;
    DevSlot slot[FABGPU_SLOTS];
    // bitmask exchange over peer memory (fabgpu_peer_mask_*): this rank's receive buffer, the peers' mapped ones
    struct Peer {
        uint32_t* local = nullptr; uint32_t* mapped[FAB_PEER_MAX] = {nullptr}; bool opened[FAB_PEER_MAX] = {false};
        uint32_t* done = nullptr; uint32_t* timeout = nullptr; uint32_t* h_timeout = nullptr;
        int world = 0, rank = 0; size_t words_per_rank = 0; bool ready = false;
    } peer;
};

struct HostSlot {
    uint8_t* h_in[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    uint32_t* h_mask = nullptr;
    uint32_t* h_off = nullptr;
    int32_t* h_key_slot = nullptr;
};

}  // namespace

// Minimal fork-join pool for the host gates (DER parse + packing is ~40 ns/signature single-threaded, which would
// otherwise cap the end-to-end rate near 20 M/s).
class GatePool {
public:
    explicit GatePool(int n) : n_(n < 1 ? 1 : n) {
        for (int t = 1; t < n_; t++) th_.emplace_back([this, t] { loop(t); });
    }
    ~GatePool() {
        { std::lock_guard<std::mutex> lk(mu_); stop_ = true; gen_.fetch_add(1); }
        cv_.notify_all();
        for (auto& t : th_) t.join();
    }
    int size() const { return n_; }
    // runs fn(tid) for tid in [0, size) and returns when all are done
    void run(const std::function<void(int)>& fn) {
        if (n_ == 1) { fn(0); return; }
        { std::lock_guard<std::mutex> lk(mu_); fn_ = &fn; pending_.store(n_ - 1); gen_.fetch_add(1); }
        cv_.notify_all();
        fn(0);
        for (int spin = 0; spin < 20000 && pending_.load(std::memory_order_acquire) != 0; spin++) cpu_relax();
        if (pending_.load(std::memory_order_acquire) == 0) return;
        std::unique_lock<std::mutex> lk(mu_);
        done_.wait(lk, [this] { return pending_.load() == 0; });
    }
private:
    static void cpu_relax() {
#if defined(__SSE2__)
        _mm_pause();
#endif
    }
    // Workers spin briefly for the next job (back-to-back batches arrive within microseconds) before sleeping.
    void loop(int tid) {
        unsigned long long seen = 0;
        for (;;) {
            for (int spin = 0; spin < 20000 && gen_.load(std::memory_order_acquire) == seen; spin++) cpu_relax();
            const std::function<void(int)>* fn;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] { return gen_.load() != seen; });
                seen = gen_.load();
                if (stop_) return;
                fn = fn_;
            }
            (*fn)(tid);
            if (pending_.fetch_sub(1, std::memory_order_acq_rel) == 1) { std::lock_guard<std::mutex> lk(mu_); done_.notify_one(); }
        }
    }
    int n_;
    std::vector<std::thread> th_;
    std::mutex mu_;
    std::condition_variable cv_, done_;
    const std::function<void(int)>* fn_ = nullptr;
    std::atomic<int> pending_{0};
    std::atomic<unsigned long long> gen_{0};
    bool stop_ = false;
};

struct fabgpu_ctx {
    std::vector<Device> devs;
    std::unique_ptr<GatePool> pool;
    HostSlot hslot[FABGPU_SLOTS];
    size_t max_batch = 0;      // per slot, whole context
    size_t dev_cap = 0;        // per device per slot (multiple of 32)
    std::string last_error;
    std::mutex mu;         // guards enqueue and the key-table bookkeeping
    // Key-table slots: whoever turns handles into raw slot numbers and then enqueues kernels that read those slots' tables holds this
    // SHARED from the resolution to the last enqueue; fabgpu_keys_register holds it EXCLUSIVE while it recycles slots (it then drains
    // every stream before rebuilding a table), so a slot cannot change hands between "resolved" and "enqueued".  Order: tab_mu, then mu.
    std::shared_mutex tab_mu;
    std::mutex sync_mu;    // one synchronous fabgpu_bccsp_verify_batch at a time
    std::mutex sync_blk_mu;   // one synchronous fabgpu_validate_block / _envelopes at a time
    std::mutex slot0_mu;   // serialises the composite calls that stage through slot 0's pinned buffers
    std::atomic<unsigned long long> launches{0};
    // per-key table cache (fabgpu_keys_register): 64-byte X||Y -> slot, least-recently-used eviction
    int key_slots = 0;
    std::unordered_map<std::string, int> key_map;
    std::vector<std::string> slot_key;
    std::vector<unsigned long long> slot_tick;
    std::vector<uint32_t> slot_gen;          // bumped whenever a slot is recycled: handles carry the generation they were issued under
    unsigned long long tick = 0;
    int key_min_uses = 256;
    // small-table cache (fabgpu_keys_register_small): same protocol as the big tables (tab_mu / mu), least-recently-used eviction
    // in bulk.  A small handle is -2 - ((generation & 0x3ff) << 20 | slot); on the device the code is -2 - slot.
    int small_slots = 0;
    int small_threads_env = 0;                // FABGPU_SMALL_THREADS: CTA width of ecdsa_verify_small_kernel (0 = by batch size)
    // Cumulative signatures of a key (over all calls) before it earns a small table; < 0: tier off.  A table costs about as much GPU time as 37 generic
    // verifications (1.5 us against 41 ns) and saves 34 ns per later signature: 32 is the rent-or-buy point -- by then the key has cost as much on the
    // generic kernel as its table does, so building is at most twice the optimum whatever the key does next, and a block full of one-off keys is
    // not slowed down by thousands of useless builds.
    int small_min_uses = 32;
    struct Key64 { uint8_t b[64]; bool operator==(const Key64& o) const { return memcmp(b, o.b, 64) == 0; } };
    struct Key64Hash { size_t operator()(const Key64& k) const { uint64_t h; memcpy(&h, k.b + 8, 8); return (size_t)(h * 0x9E3779B97F4A7C15ull); } };
    std::unordered_map<Key64, int, Key64Hash> small_map;
    std::vector<Key64> small_key; std::vector<char> small_used;
    std::vector<unsigned long long> small_tick;
    std::vector<uint32_t> small_gen;
    std::vector<int> small_free;
    unsigned long long small_built = 0, small_recycled = 0;     // fabgpu_key_table_stats
    // Keys without any table: signatures seen so far.  Buckets of four (tag, count) entries indexed by a hash of the key bytes -- no allocation
    // on the batch path; a full bucket gives up its least used entry, which only delays that key's table (resolve_key_tables).
    std::vector<uint64_t> seen_tag; std::vector<uint32_t> seen_cnt;
    // key-table kernel (FABGPU_CACHED_KERNEL): 0 "jac" = Jacobian chain, one signature per thread (ecdsa_verify_cached_kernel) -- the DEFAULT: fastest at
    // every batch size measured on B200 (profiles/r2_kernel_variants.txt); 1 "ba" = batch-affine with CTA-shared inversions, 3 "ba2" = batch-affine, two
    // signatures per thread, 2 / 4 "l2" / "l4" = the Jacobian chain split over 2 / 4 lanes.  The alternatives stay selectable: they are the measurements.
    int cached_kernel = 0;
    double timing[4] = {0, 0, 0, 0};   // last fabgpu_bccsp_verify_batch: key lookup, host gates, device (H2D+kernel+D2H), scatter [us]
    // block validation (fabgpu_msp_configure / fabgpu_validate_block), device 0 of the context
    blockval::MspTable msp;
    std::vector<blockval::PolicyNode> policy;
    std::vector<std::string> principals;
    std::string channel;
    std::vector<int32_t> identity_slot;
    struct BlockBufs {
        uint8_t* d_block = nullptr; size_t block_cap = 0;
        uint8_t* h_block = nullptr; size_t h_block_cap = 0;       // optional pinned staging the caller may fill directly
        size_t job_cap = 0;                                       // signature jobs
        size_t sha_cap = 0;                                       // all digests (signature jobs + 2 per transaction)
        ShaJob* d_sha = nullptr; ShaJob* h_sha = nullptr;
        uint8_t* d_dig = nullptr; uint8_t* h_dig = nullptr;       // h_dig: check digests only
        uint8_t *d_r = nullptr, *d_s = nullptr, *d_qx = nullptr, *d_qy = nullptr;
        uint8_t *h_r = nullptr, *h_s = nullptr, *h_qx = nullptr, *h_qy = nullptr;
        int32_t *d_ks = nullptr, *h_ks = nullptr;
        uint32_t *d_mask = nullptr, *d_off = nullptr, *h_mask = nullptr;
    } bbs[FABGPU_SLOTS];          // [0] also serves the host-thread path (FABGPU_BLOCK_HOST=1)
    double block_timing[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};   // host phases [0..4] (see fabgpu_block_timing), device stages [5..9]
    // device-side copy of the MSP view / policy (block_plan_kernel, block_decide_kernel)
    struct DevMsp {
        uint8_t *id_blob = nullptr, *valid = nullptr, *keys_xy = nullptr, *channel = nullptr;
        uint32_t* id_off = nullptr; int32_t *key_slot = nullptr, *msp_code = nullptr, *ht_idx = nullptr, *nodes = nullptr, *principal_code = nullptr;
        int32_t* group = nullptr;                                     // de-duplication groups (fabgpu_msp_identity_groups), null = identity index
        uint8_t* ns_blob = nullptr; uint32_t* ns_off = nullptr; int32_t* ns_root = nullptr; int32_t n_ns = 0;    // fabgpu_namespace_policies
        uint64_t* ht_hash = nullptr; uint32_t ht_size = 0; int32_t n_ids = 0, n_nodes = 0, n_principals = 0; uint32_t channel_len = 0;
        bool all_slots = true; int classes = 0;                    // which non-big classes the identities' keys fall in (CLASS_*)
        uint8_t* hash_kind = nullptr; bool any_sha3 = false;        // per identity: SHA_KIND_* of its MSP (fabgpu_msp_hash_families)
    } dm;
    struct GateBufs {                          // fabgpu_bccsp_verify_batch with device-side gates
        size_t n_cap = 0, sig_cap = 0, dig_cap = 0, k_cap = 0;
        uint8_t *h_sigs = nullptr, *h_digs = nullptr, *h_keys = nullptr, *h_status = nullptr; uint32_t *h_sig_off = nullptr, *h_dig_off = nullptr;
        int32_t *h_kidx = nullptr, *h_slot_of = nullptr;
        uint8_t *d_sigs = nullptr, *d_digs = nullptr, *d_keys = nullptr, *d_status = nullptr, *d_pre = nullptr, *d_r = nullptr, *d_s = nullptr, *d_e = nullptr,
        *d_qx = nullptr, *d_qy = nullptr; uint32_t *d_sig_off = nullptr, *d_dig_off = nullptr, *d_mask = nullptr, *d_off = nullptr;
        int32_t *d_kidx = nullptr, *d_slot_of = nullptr, *d_ks = nullptr; uint32_t* d_idx = nullptr;
        // fabgpu_bccsp_verify_batch_async .. _wait: what is in flight on this slot
        bool busy = false; bool on_device = false; size_t n = 0;
        std::vector<uint8_t> done_status;       // statuses of a batch that could not take the device-gate path (finished at submit time)
        std::chrono::steady_clock::time_point t_submit;
    } gb[FABGPU_SLOTS];
    std::mutex gb_mu[FABGPU_SLOTS];
    struct DevBlock {
        size_t tx_cap = 0, j_cap = 0;
        uint32_t* d_env_off = nullptr; bdev::TxDev* d_txs = nullptr; bdev::RawJob* d_raw = nullptr; bdev::ShaJobD* d_sha = nullptr; uint8_t *d_r = nullptr, *d_s = nullptr, *d_qx = nullptr,
        *d_qy = nullptr, *d_gate = nullptr, *d_dig = nullptr, *d_flags = nullptr; int32_t *d_ks = nullptr, *d_ident = nullptr; uint32_t *d_mask = nullptr,
        *d_off = nullptr, *d_counter = nullptr, *d_idx = nullptr; uint64_t* d_hash = nullptr; bdev::Seg* d_seg = nullptr;
        uint8_t* d_kind = nullptr;               // per signature job: SHA_KIND_* (written only when the MSP table holds a SHA3 identity)
        uint8_t* h_flags = nullptr; uint64_t* h_hash = nullptr; bdev::Seg* h_seg = nullptr; uint32_t* h_counter = nullptr; uint32_t* h_env_off = nullptr;
        // the block in flight on this slot (fabgpu_validate_*_async .. fabgpu_validate_wait)
        bool busy = false, on_device = false, use_ev = false; size_t T = 0; const uint8_t* block = nullptr;
        std::vector<uint8_t> done_flags;         // host-thread path: finished at submit time
        std::vector<uint64_t> dup_keys; std::vector<uint32_t> dup_idx;   // scratch of the duplicate-tx-id pass (per slot: waits may run concurrently)
        std::chrono::steady_clock::time_point t0, t1;
        cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    } dbs[FABGPU_SLOTS];
    std::mutex blk_mu[FABGPU_SLOTS];
};

namespace {

#define CK(ctx, call)                                                                                       \
    do {                                                                                                    \
        cudaError_t e_ = (call);                                                                            \
        if (e_ != cudaSuccess) {                                                                            \
            char buf_[512];                                                                                 \
            snprintf(buf_, sizeof buf_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            if (ctx) (ctx)->last_error = buf_; else g_init_error = buf_;                                    \
            return FABGPU_E_CUDA;                                                                           \
        }                                                                                                   \
    } while (0)

bool fault_injected()
{
    const char* v = getenv("FABGPU_FAULT_INJECT");
    return v && v[0] == '1';
}

size_t round_up32(size_t x) { return (x + 31) / 32 * 32; }

// 32-byte copy into a pinned staging buffer with streaming stores: the lines never become dirty in this core's cache,
// so the H2D DMA that follows does not have to snoop 16+ cores across two sockets (measured: that snooping more than
// doubled the copy phase when the gates ran multi-threaded).
inline void stage32(uint8_t* dst, const uint8_t* src)
{
#if defined(__SSE2__)
    const __m128i a = _mm_loadu_si128((const __m128i*)src), b = _mm_loadu_si128((const __m128i*)(src + 16));
    _mm_stream_si128((__m128i*)dst, a);
    _mm_stream_si128((__m128i*)(dst + 16), b);
#else
    memcpy(dst, src, 32);
#endif
}
inline void stage_i32(int32_t* dst, int32_t v)
{
#if defined(__SSE2__)
    _mm_stream_si32((int*)dst, v);
#else
    *dst = v;
#endif
}
// bytes -> pinned staging with streaming stores (16-byte aligned body), see stage32
inline void stage_copy(uint8_t* dst, const uint8_t* src, size_t n)
{
#if defined(__SSE2__)
    size_t i = 0;
    while (i < n && ((uintptr_t)(dst + i) & 15u)) { dst[i] = src[i]; i++; }
    for (; i + 16 <= n; i += 16) _mm_stream_si128((__m128i*)(dst + i), _mm_loadu_si128((const __m128i*)(src + i)));
    for (; i < n; i++) dst[i] = src[i];
#else
    memcpy(dst, src, n);
#endif
}
inline void stage_fence()
{
#if defined(__SSE2__)
    _mm_sfence();
#endif
}

// mode: 0 = no signature has a key table (generic kernel only), 1 = all have one (cached kernel only),
//       2 = mixed (cached kernel, then the generic kernel fills in the rest)
//       3 = all have a SMALL table (key_slot codes <= -2 throughout)
// In mode 2 key_slot codes decide per signature: >= 0 big table, -1 none, <= -2 small table (see compact_classes_kernel).
enum { MODE_GENERIC = 0, MODE_CACHED = 1, MODE_MIXED = 2, MODE_SMALL = 3 };

// CTA width of the small-table kernel: as for the key-table kernel, a batch that fits one wave of 512-thread CTAs runs best as such; when
// the count is only an upper bound (compacted list) small CTAs spread the unknown number of live warps over all SMs.  FABGPU_SMALL_THREADS
// overrides (measurements).
unsigned small_threads(const fabgpu_ctx* ctx, const Device& dv, size_t n, bool bound_only)
{
    if (ctx->small_threads_env) return (unsigned)ctx->small_threads_env;
    if (bound_only) return 128;
    const size_t sms = (size_t)dv.sms;
    if (n > sms * 384) return (n <= sms * FAB_SMALL_THREADS) ? FAB_SMALL_THREADS : 256;
    return 128;
}
// classes (mode 2 with scratch): which of the non-big classes the batch may contain -- a class the caller knows to be absent is not launched.
enum { CLASS_SMALL = 1, CLASS_GENERIC = 2 };
// n_dev / n_base (block path): the batch is [0, min(n, n_base + *n_dev)) with *n_dev written by an earlier kernel of the stream.
int launch_verify(fabgpu_ctx* ctx, const Device& dv, int mode, const int32_t* key_slot, const uint8_t* qx, const uint8_t* qy,
                  const uint8_t* e, const uint8_t* r, const uint8_t* s, size_t n, uint32_t* mask, uint32_t* off, cudaStream_t st,
                  const uint32_t* n_dev = nullptr, uint32_t n_base = 0, const PeerOut* peer = nullptr, uint32_t* scratch_idx = nullptr,
                  int classes = CLASS_SMALL | CLASS_GENERIC)
{
    PeerOut po; memset(&po, 0, sizeof po);
    const bool fused_peer = peer && mode == MODE_CACHED && (ctx->cached_kernel == 0 || ctx->cached_kernel == 1 || ctx->cached_kernel == 3) && n > 0 && !n_dev;
    if (fused_peer) po = *peer;
    if (peer && !fused_peer) {                            // several kernels write the mask: scatter it afterwards (below)
        if (n_dev) { ctx->last_error = "peer exchange needs a host-known batch size"; return FABGPU_E_ARG; }
    }
    if (n == 0 && !peer) return FABGPU_OK;
    if ((mode == MODE_MIXED || mode == MODE_SMALL) && dv.s_ev_set) CK(ctx, cudaStreamWaitEvent(st, dv.s_ev, 0));   // small tables still being built
    if (mode == MODE_SMALL && n > 0) {
        const unsigned sthreads = small_threads(ctx, dv, n, false);
        ecdsa_verify_small_kernel<<<(unsigned)((n + sthreads - 1) / sthreads), sthreads, 0, st>>>(
            nullptr, nullptr, 0u, key_slot, e, r, s, (uint32_t)n, dv.gtab, dv.stab, mask, off);
        ctx->launches++;
        CK(ctx, cudaGetLastError());
    }
    if (mode != MODE_GENERIC && mode != MODE_SMALL && n > 0) {
        // CTA shape (the kernel allows up to FAB_CACHED_THREADS = 512 threads at 128 registers, i.e. one such CTA per SM).
        // Measured on B200 (profiles/r1_kbench_table_widths.txt): a batch that fits one wave of 512-thread CTAs (64k: 128 CTAs)
        // finishes in 0.315 ms against 0.346 ms as 512 CTAs of 128 threads; beyond one wave 256-thread CTAs quantise best
        // (256k: 231 M/s against 223 / 212 for 128 / 512); below ~12 warps per SM small CTAs spread over all SMs win
        // (fewer warps per scheduler = lower latency per warp), and so they do when the batch size is only an upper bound.
        if (ctx->cached_kernel == 2 || ctx->cached_kernel == 4) {
            // lane-split Jacobian chain (measurement variant): 2 or 4 lanes per signature
            const unsigned sigs = FAB_LANES_THREADS / (unsigned)ctx->cached_kernel, blocks = (unsigned)((n + sigs - 1) / sigs);
            uint32_t nn = (uint32_t)n;
            if (n_dev) { ctx->last_error = "the lane-split kernel has no device-side batch size"; return FABGPU_E_ARG; }
            if (ctx->cached_kernel == 2) ecdsa_verify_lanes_kernel<2><<<blocks, FAB_LANES_THREADS, 0, st>>>(key_slot, e, r, s, nn, dv.gtab, dv.qtab, mask, off);
            else ecdsa_verify_lanes_kernel<4><<<blocks, FAB_LANES_THREADS, 0, st>>>(key_slot, e, r, s, nn, dv.gtab, dv.qtab, mask, off);
        } else if (ctx->cached_kernel == 3 && !n_dev && !fused_peer) {
            // batch-affine, two signatures per thread, no CTA exchange
            const unsigned per = 2 * FAB_BA2_THREADS, blocks = (unsigned)((n + per - 1) / per);
            ecdsa_verify_ba2_kernel<<<blocks, FAB_BA2_THREADS, 0, st>>>(key_slot, e, r, s, (uint32_t)n, dv.gtab, dv.qtab, mask, off);
        } else if (ctx->cached_kernel == 1 || ctx->cached_kernel == 3) {
            // batch-affine accumulation with CTA-shared inversions (ecdsa_batchaffine.cuh): fixed CTA width
            const unsigned blocks = (unsigned)((n + FAB_BA_THREADS - 1) / FAB_BA_THREADS);
            ecdsa_verify_ba_kernel<<<blocks, FAB_BA_THREADS, 0, st>>>(key_slot, e, r, s, (uint32_t)n, dv.gtab, dv.qtab, mask, off, n_dev, n_base, po);
        } else {
        unsigned threads = 128;
        const size_t sms = (size_t)dv.sms;
        if (!n_dev && n > sms * 384) threads = (n <= sms * FAB_CACHED_THREADS) ? FAB_CACHED_THREADS : 256;
        const unsigned blocks = (unsigned)((n + threads - 1) / threads);
        ecdsa_verify_cached_kernel<<<blocks, threads, 0, st>>>(key_slot, e, r, s, (uint32_t)n, dv.gtab, dv.qtab, mask, off, n_dev, n_base, po);
        }
        ctx->launches++;
        CK(ctx, cudaGetLastError());
    }
    if (mode == MODE_MIXED && n > 0 && scratch_idx) {
        // signatures without a big table: compact their indices by class, then whole warps of small-table / generic arithmetic
        // (see compact_classes_kernel).  scratch_idx: n + 2 words owned by the caller's slot (indices, then the two counters).
        CK(ctx, cudaMemsetAsync(scratch_idx + n, 0, 8, st));
        compact_classes_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(key_slot, (uint32_t)n, scratch_idx, scratch_idx + n, n_dev, n_base);
        if (classes & CLASS_SMALL) {
            const unsigned sthreads = small_threads(ctx, dv, n, true);
            ecdsa_verify_small_kernel<<<(unsigned)((n + sthreads - 1) / sthreads), sthreads, 0, st>>>(
                scratch_idx, scratch_idx + n + 1, (uint32_t)n, key_slot, e, r, s, (uint32_t)n, dv.gtab, dv.stab, mask, off);
        }
        if (classes & CLASS_GENERIC)
            ecdsa_verify_indexed_kernel<<<(unsigned)((n + FAB_INDEXED_THREADS - 1) / FAB_INDEXED_THREADS), FAB_INDEXED_THREADS, 0, st>>>(
                scratch_idx, scratch_idx + n, qx, qy, e, r, s, dv.gtab, mask, off);
        ctx->launches += 1 + ((classes & CLASS_SMALL) ? 1 : 0) + ((classes & CLASS_GENERIC) ? 1 : 0);
        CK(ctx, cudaGetLastError());
    } else if (mode == MODE_MIXED && n > 0) {
        // no scratch (launches on a caller's stream): the generic kernel filters on key_slot itself
        const unsigned gthreads = 128, blocks = (unsigned)((n + gthreads - 1) / gthreads);
        ecdsa_verify_kernel<<<blocks, gthreads, 0, st>>>(key_slot, qx, qy, e, r, s, (uint32_t)n, dv.gtab, mask, off, n_dev, n_base);
        ctx->launches++;
        CK(ctx, cudaGetLastError());
    }
    if (mode == MODE_GENERIC && n > 0) {
        // same reasoning for the generic kernel (measured: 64k as 147 CTAs of 448 threads 24.1 M/s, as 1024 CTAs of 64 threads 22.6;
        // 256k as CTAs of 256 threads 27.6 M/s, of 448 threads 24.3)
        unsigned gthreads = 64;
        if (!n_dev && n > (size_t)dv.sms * 192) gthreads = (n <= (size_t)dv.sms * FAB_VERIFY_THREADS) ? FAB_VERIFY_THREADS : 256;
        const unsigned blocks = (unsigned)((n + gthreads - 1) / gthreads);
        ecdsa_verify_kernel<<<blocks, gthreads, 0, st>>>(nullptr, qx, qy, e, r, s, (uint32_t)n, dv.gtab, mask, off, n_dev, n_base);
        ctx->launches++;
        CK(ctx, cudaGetLastError());
    }
    if (peer && !fused_peer) {
        const uint32_t words = (uint32_t)((n + 31) / 32);
        peer_scatter_kernel<<<words ? (words + 127) / 128 : 1, 128, 0, st>>>(mask, words, *peer);
        ctx->launches++;
        CK(ctx, cudaGetLastError());
    }
    return FABGPU_OK;
}

// (The generation field is 19 bits: a handle kept across 524 288 recyclings of ITS slot would match again.  At one recycling per registration
// call that is days of continuous eviction of one slot while a caller sits on a stale handle; the Go provider re-reads the handle from the key
// object on every batch, so it never holds one that long.)
// A key handle is (generation << 12) | slot.  A handle issued before its slot was recycled no longer matches the slot's
// generation and silently degrades to "no table" (-1): the generic kernel then verifies against the Qx/Qy the caller
// supplied, so a stale handle can cost speed but never correctness.
inline int32_t make_handle(const fabgpu_ctx* ctx, int sl) { return (int32_t)(((ctx->slot_gen[sl] & 0x7ffffu) << 12) | (uint32_t)sl); }
inline int32_t make_small_handle(const fabgpu_ctx* ctx, int sl) { return -2 - (int32_t)(((ctx->small_gen[sl] & 0x3ffu) << 20) | (uint32_t)sl); }
// handle -> device code: >= 0 big-table slot, -2 - slot for a live small table, -1 otherwise (no table, stale handle)
inline int32_t handle_to_slot(const fabgpu_ctx* ctx, int32_t h)
{
    if (h <= -2) {
        const uint32_t v = (uint32_t)(-2 - h);
        const int sl = (int)(v & 0xfffffu);
        if (sl >= ctx->small_slots || (v >> 20) != (ctx->small_gen[sl] & 0x3ffu) || !ctx->small_used[sl]) return -1;
        return -2 - sl;
    }
    if (h < 0) return -1;
    const int sl = h & 0xfff;
    if (sl >= ctx->key_slots || ((uint32_t)h >> 12) != (ctx->slot_gen[sl] & 0x7ffffu) || ctx->slot_key[sl].empty()) return -1;
    return sl;
}

int slots_mode(const int32_t* ks, size_t n, int* classes)
{
    bool any_c = false, any_g = false, any_s = false;
    for (size_t i = 0; i < n; i++) { if (ks[i] >= 0) any_c = true; else if (ks[i] == -1) any_g = true; else any_s = true; }
    *classes = (any_s ? CLASS_SMALL : 0) | (any_g ? CLASS_GENERIC : 0);
    if (!any_c && !any_g && any_s) return MODE_SMALL;
    if (!any_c && !any_s) return MODE_GENERIC;
    return (any_g || any_s) ? MODE_MIXED : MODE_CACHED;
}

int enqueue_slot(fabgpu_ctx* ctx, int slot, size_t n, bool keyed)
{
    // contiguous 32-aligned ranges per device
    const size_t ndev = ctx->devs.size();
    const size_t per = round_up32((n + ndev - 1) / ndev);
    for (size_t d = 0; d < ndev; d++) {
        const size_t begin = std::min(n, d * per), end = std::min(n, (d + 1) * per);
        const size_t cnt = end - begin;
        if (cnt == 0) continue;
        Device& dv = ctx->devs[d];
        DevSlot& ds = dv.slot[slot];
        HostSlot& hs = ctx->hslot[slot];
        CK(ctx, cudaSetDevice(dv.id));
        if (keyed) for (size_t i = begin; i < end; i++) hs.h_key_slot[i] = handle_to_slot(ctx, hs.h_key_slot[i]);   // handles -> live slots
        int classes = CLASS_GENERIC;
        const int mode = keyed ? slots_mode(hs.h_key_slot + begin, cnt, &classes) : MODE_GENERIC;
        for (int a = ((mode == MODE_CACHED || mode == MODE_SMALL) ? 2 : 0); a < 5; a++)     // a range where every key has a table needs no Qx/Qy on the device
            CK(ctx, cudaMemcpyAsync(ds.d_in[a], hs.h_in[a] + 32 * begin, 32 * cnt, cudaMemcpyHostToDevice, ds.stream));
        if (mode != MODE_GENERIC)
            CK(ctx, cudaMemcpyAsync(ds.d_key_slot, hs.h_key_slot + begin, 4 * cnt, cudaMemcpyHostToDevice, ds.stream));
        int rc = launch_verify(ctx, dv, mode, ds.d_key_slot, ds.d_in[0], ds.d_in[1], ds.d_in[2], ds.d_in[3], ds.d_in[4], cnt, ds.d_mask,
                               ds.d_off, ds.stream, nullptr, 0, nullptr, ds.d_idx, classes);
        if (rc) return rc;
        const size_t words = (cnt + 31) / 32;
        CK(ctx, cudaMemcpyAsync(hs.h_mask + begin / 32, ds.d_mask, 4 * words, cudaMemcpyDeviceToHost, ds.stream));
        CK(ctx, cudaMemcpyAsync(hs.h_off + begin / 32, ds.d_off, 4 * words, cudaMemcpyDeviceToHost, ds.stream));
    }
    return FABGPU_OK;
}

int wait_slot(fabgpu_ctx* ctx, int slot)
{
    for (auto& dv : ctx->devs) {
        CK(ctx, cudaSetDevice(dv.id));
        CK(ctx, cudaStreamSynchronize(dv.slot[slot].stream));
    }
    return FABGPU_OK;
}

void free_all(fabgpu_ctx* ctx)
{
    {
        if (!ctx->devs.empty()) cudaSetDevice(ctx->devs[0].id);
        for (auto& bb : ctx->bbs) {
            void* dev_ptrs[] = {bb.d_block, bb.d_sha, bb.d_dig, bb.d_r, bb.d_s, bb.d_qx, bb.d_qy, bb.d_ks, bb.d_mask, bb.d_off};
            for (void* p : dev_ptrs) if (p) cudaFree(p);
            void* host_ptrs[] = {bb.h_block, bb.h_sha, bb.h_dig, bb.h_r, bb.h_s, bb.h_qx, bb.h_qy, bb.h_ks, bb.h_mask};
            for (void* p : host_ptrs) if (p) cudaFreeHost(p);
        }
        auto& dm = ctx->dm;
        void* dev2[] = {dm.id_blob, dm.valid, dm.keys_xy, dm.channel, dm.id_off, dm.key_slot, dm.msp_code, dm.ht_idx, dm.nodes, dm.principal_code, dm.ht_hash,
                        dm.group, dm.ns_blob, dm.ns_off, dm.ns_root, dm.hash_kind};
        for (void* p : dev2) if (p) cudaFree(p);
        for (auto& db : ctx->dbs) {
            void* dev4[] = {db.d_env_off, db.d_txs, db.d_raw, db.d_sha, db.d_r, db.d_s, db.d_qx, db.d_qy, db.d_gate, db.d_dig, db.d_flags, db.d_ks, db.d_ident, db.d_mask, db.d_off,
                            db.d_counter, db.d_hash, db.d_seg, db.d_idx, db.d_kind};
            for (void* p : dev4) if (p) cudaFree(p);
            void* host2[] = {db.h_flags, db.h_hash, db.h_seg, db.h_counter, db.h_env_off};
            for (void* p : host2) if (p) cudaFreeHost(p);
            for (auto& e : db.ev) if (e) cudaEventDestroy(e);
        }
        for (auto& gb : ctx->gb) {
        void* dev3[] = {gb.d_sigs, gb.d_digs, gb.d_keys, gb.d_status, gb.d_pre, gb.d_r, gb.d_s, gb.d_e, gb.d_qx, gb.d_qy, gb.d_sig_off, gb.d_dig_off, gb.d_mask, gb.d_off,
                        gb.d_kidx, gb.d_slot_of, gb.d_ks, gb.d_idx};
        for (void* p : dev3) if (p) cudaFree(p);
        void* host3[] = {gb.h_sigs, gb.h_digs, gb.h_keys, gb.h_status, gb.h_sig_off, gb.h_dig_off, gb.h_kidx, gb.h_slot_of};
        for (void* p : host3) if (p) cudaFreeHost(p);
        }
    }
    for (auto& dv : ctx->devs) {
        cudaSetDevice(dv.id);
        {   // peer-memory bitmask exchange (fabgpu_peer_mask_*)
            auto& pr = dv.peer;
            for (int p = 0; p < FAB_PEER_MAX; p++) if (pr.opened[p]) cudaIpcCloseMemHandle(pr.mapped[p]);
            if (pr.local) cudaFree(pr.local);
            if (pr.done) cudaFree(pr.done);
            if (pr.h_timeout) cudaFreeHost(pr.h_timeout);
            pr = Device::Peer();
        }
        if (dv.gtab) cudaFree(dv.gtab);
        if (dv.qtab) cudaFree(dv.qtab);
        void* sm[] = {dv.stab, dv.s_bases, dv.s_keys, dv.s_slots};
        for (void* q : sm) if (q) cudaFree(q);
        if (dv.s_ev) cudaEventDestroy(dv.s_ev);
        if (dv.s_stream) cudaStreamDestroy(dv.s_stream);
        for (auto& ds : dv.slot) {
            if (ds.d_key_slot) cudaFree(ds.d_key_slot);
            if (ds.d_idx) cudaFree(ds.d_idx);
            for (auto& p : ds.d_in) if (p) cudaFree(p);
            if (ds.d_mask) cudaFree(ds.d_mask);
            if (ds.d_off) cudaFree(ds.d_off);
            if (ds.stream) cudaStreamDestroy(ds.stream);
        }
    }
    for (auto& hs : ctx->hslot) {
        for (auto& p : hs.h_in) if (p) cudaFreeHost(p);
        if (hs.h_mask) cudaFreeHost(hs.h_mask);
        if (hs.h_off) cudaFreeHost(hs.h_off);
        if (hs.h_key_slot) cudaFreeHost(hs.h_key_slot);
    }
}

int init_impl(fabgpu_ctx* ctx, const int* device_ids, int n_dev, size_t max_batch)
{
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        ctx->last_error = std::string("no usable CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                          " (libfabgpu_ecdsa has no CPU fallback; use the software provider)";
        return FABGPU_E_NO_DEVICE;
    }
    std::vector<int> ids;
    if (device_ids == nullptr || n_dev <= 0) ids.push_back(0);
    else ids.assign(device_ids, device_ids + n_dev);
    for (int id : ids)
        if (id < 0 || id >= count) { ctx->last_error = "device id out of range"; return FABGPU_E_NO_DEVICE; }
    if (max_batch == 0) { ctx->last_error = "max_batch must be > 0"; return FABGPU_E_ARG; }
    ctx->max_batch = max_batch;
    {
        int hw = (int)std::thread::hardware_concurrency();
        const char* ev = getenv("FABGPU_GATE_THREADS");
        int want = ev ? atoi(ev) : std::max(1, std::min(hw > 0 ? hw / 2 : 1, 32));   // gates and block parsing are latency-bound
        ctx->pool.reset(new GatePool(want));
        // Per-key tables are 64 MiB each (FAB_WQ = 16), per device.  The request (default 256 = 16 GiB of a B200's 180 GB) is
        // capped so that the tables never take more than half of the smallest device's free memory.
        const char* ks = getenv("FABGPU_KEY_SLOTS");
        ctx->key_slots = ks ? std::max(1, atoi(ks)) : 256;
        if (ctx->key_slots > 4096) ctx->key_slots = 4096;     // a handle keeps 12 bits for the slot
        const size_t per_key = (size_t)FAB_Q_WINDOWS * FAB_Q_ENTRIES * sizeof(aff);
        for (int id : ids) {
            size_t free_b = 0, total_b = 0;
            CK(ctx, cudaSetDevice(id));
            CK(ctx, cudaMemGetInfo(&free_b, &total_b));
            const size_t g_bytes = (size_t)FAB_G_WINDOWS * FAB_G_ENTRIES * sizeof(aff);
            const size_t room = free_b > 2 * g_bytes ? (free_b - 2 * g_bytes) / 2 : 0;
            ctx->key_slots = (int)std::max<size_t>(1, std::min<size_t>((size_t)ctx->key_slots, room / per_key));
        }
        ctx->slot_key.assign(ctx->key_slots, std::string());
        ctx->slot_tick.assign(ctx->key_slots, 0ull);
        ctx->slot_gen.assign(ctx->key_slots, 0u);
        // Small tables (FAB_S_POINTS * 64 bytes = 264 KiB each): default 16 384 of them (4.4 GB); FABGPU_SMALL_SLOTS = 0 turns the tier off.
        const char* ss = getenv("FABGPU_SMALL_SLOTS");
        ctx->small_slots = ss ? std::max(0, atoi(ss)) : 16384;
        if (ctx->small_slots > (1 << 20)) ctx->small_slots = 1 << 20;       // a handle keeps 20 bits for the slot
        for (int id : ids) {
            size_t free_b = 0, total_b = 0;
            CK(ctx, cudaSetDevice(id));
            CK(ctx, cudaMemGetInfo(&free_b, &total_b));
            const size_t per_small = (size_t)FAB_S_POINTS * sizeof(aff);
            ctx->small_slots = (int)std::min<size_t>((size_t)ctx->small_slots, free_b / 8 / per_small);
        }
        ctx->small_key.assign(ctx->small_slots, fabgpu_ctx::Key64());
        ctx->small_used.assign(ctx->small_slots, 0);
        ctx->small_tick.assign(ctx->small_slots, 0ull);
        ctx->small_gen.assign(ctx->small_slots, 0u);
        ctx->small_free.clear();
        for (int sl = ctx->small_slots - 1; sl >= 0; sl--) ctx->small_free.push_back(sl);
        ctx->seen_tag.assign((size_t)1 << 18, 0ull); ctx->seen_cnt.assign((size_t)1 << 18, 0u);
        const char* sth = getenv("FABGPU_SMALL_THREADS");
        if (sth) { const int v = atoi(sth); if (v == 64 || v == 128 || v == 256 || v == 512) ctx->small_threads_env = v; }
        const char* smu = getenv("FABGPU_SMALL_MIN_USES");
        ctx->small_min_uses = smu ? atoi(smu) : 32;
        if (ctx->small_slots == 0) ctx->small_min_uses = -1;
        const char* mu = getenv("FABGPU_KEY_MIN_USES");
        ctx->key_min_uses = mu ? atoi(mu) : 256;           // a table costs about 300 generic verifications to build
        const char* ck = getenv("FABGPU_CACHED_KERNEL");
        if (ck) ctx->cached_kernel = (ck[0] == 'j' || ck[0] == '0') ? 0 : (ck[0] == 'l' ? (ck[1] == '4' ? 4 : 2) : (ck[0] == 'b' && ck[1] == 'a' && ck[2] == '2' ? 3 : 1));   // "jac" / "0": the Jacobian-chain kernel; "l2" / "l4": its lane-split variant
    }
    ctx->dev_cap = round_up32((max_batch + ids.size() - 1) / ids.size());
    ctx->devs.resize(ids.size());
    const size_t words = ctx->dev_cap / 32;
    const size_t tab_entries = (size_t)FAB_G_WINDOWS * FAB_G_ENTRIES;
    for (size_t d = 0; d < ids.size(); d++) {
        Device& dv = ctx->devs[d];
        dv.id = ids[d];
        CK(ctx, cudaSetDevice(dv.id));
        CK(ctx, cudaDeviceGetAttribute(&dv.sms, cudaDevAttrMultiProcessorCount, dv.id));
        {   // Table gathers read 64-byte points at random addresses: by default the L2 fetches 128 bytes around a miss (two sectors'
            // worth of DRAM traffic per point).  FABGPU_L2_FETCH = 32 / 64 / 128 sets cudaLimitMaxL2FetchGranularity; default 64.
            const char* fg = getenv("FABGPU_L2_FETCH");
            const size_t want = fg ? (size_t)atoi(fg) : 64;
            if (want == 32 || want == 64 || want == 128) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, want);   // a hint: failure is not an error
            (void)cudaGetLastError();
        }
        CK(ctx, cudaMalloc(&dv.gtab, tab_entries * sizeof(aff)));
        CK(ctx, cudaMalloc(&dv.qtab, (size_t)ctx->key_slots * FAB_Q_WINDOWS * FAB_Q_ENTRIES * sizeof(aff)));
        if (ctx->small_slots > 0) {
            CK(ctx, cudaMalloc(&dv.stab, (size_t)ctx->small_slots * FAB_S_POINTS * sizeof(aff)));
            // build scratch for up to 16 384 keys per registration, allocated once: growing it later costs a cudaFree + cudaMalloc pair in the
            // middle of traffic (measured 86 ms on B200 with work in flight; profiles/r2_small_tables_shapes.txt)
            const size_t c = (size_t)std::min(ctx->small_slots, 16384);
            CK(ctx, cudaMalloc(&dv.s_bases, c * FAB_S_WINDOWS * sizeof(aff)));
            CK(ctx, cudaMalloc(&dv.s_keys, 64 * c));
            CK(ctx, cudaMalloc(&dv.s_slots, 4 * c));
            dv.s_cap = c;
        }
        CK(ctx, cudaStreamCreateWithFlags(&dv.s_stream, cudaStreamNonBlocking));
        CK(ctx, cudaEventCreateWithFlags(&dv.s_ev, cudaEventDisableTiming));
        for (auto& ds : dv.slot) {
            CK(ctx, cudaStreamCreateWithFlags(&ds.stream, cudaStreamNonBlocking));
            for (auto& p : ds.d_in) CK(ctx, cudaMalloc(&p, 32 * ctx->dev_cap));
            CK(ctx, cudaMalloc(&ds.d_mask, 4 * words));
            CK(ctx, cudaMalloc(&ds.d_off, 4 * words));
            CK(ctx, cudaMalloc(&ds.d_key_slot, 4 * ctx->dev_cap));
            CK(ctx, cudaMalloc(&ds.d_idx, 4 * (ctx->dev_cap + 2)));
        }
#if FAB_G_TWO_LEVEL
        {
            aff* d_small = nullptr; u256* d_scratch = nullptr;
            const size_t nsmall = ((size_t)1 << (FAB_WG / 2)) - 1;
            const size_t threads = (size_t)FAB_G_WINDOWS * 2;
            CK(ctx, cudaMalloc(&d_scratch, threads * 2 * nsmall * sizeof(u256)));
            CK(ctx, cudaMalloc(&d_small, threads * nsmall * sizeof(aff)));
            small_tables_kernel<<<(unsigned)((threads + 31) / 32), 32, 0, dv.slot[0].stream>>>(nullptr, 1, FAB_WG, FAB_G_WINDOWS, d_small, d_scratch, nullptr);
            const size_t threads2 = (size_t)FAB_G_WINDOWS * ((FAB_G_ENTRIES + FAB_TAB_CHUNK - 1) / FAB_TAB_CHUNK);
            full_tables_kernel<<<(unsigned)((threads2 + 127) / 128), 128, 0, dv.slot[0].stream>>>(d_small, nullptr, nullptr, 1, FAB_WG, FAB_G_WINDOWS, dv.gtab);
            ctx->launches += 2;
            CK(ctx, cudaGetLastError());
            CK(ctx, cudaStreamSynchronize(dv.slot[0].stream));
            cudaFree(d_small); cudaFree(d_scratch);
        }
#else
        build_g_table_kernel<<<(unsigned)((tab_entries + 127) / 128), 128, 0, dv.slot[0].stream>>>(dv.gtab);
        ctx->launches++;
        CK(ctx, cudaGetLastError());
#endif
    }
    const size_t hwords = (round_up32(max_batch) / 32) + ids.size();
    for (auto& hs : ctx->hslot) {
        for (auto& p : hs.h_in) CK(ctx, cudaHostAlloc(&p, 32 * round_up32(max_batch), cudaHostAllocPortable));
        CK(ctx, cudaHostAlloc(&hs.h_mask, 4 * hwords, cudaHostAllocPortable));
        CK(ctx, cudaHostAlloc(&hs.h_off, 4 * hwords, cudaHostAllocPortable));
        CK(ctx, cudaHostAlloc(&hs.h_key_slot, 4 * round_up32(max_batch), cudaHostAllocPortable));
        for (size_t i = 0; i < round_up32(max_batch); i++) hs.h_key_slot[i] = -1;
    }
    for (auto& dv : ctx->devs) {
        CK(ctx, cudaSetDevice(dv.id));
        CK(ctx, cudaStreamSynchronize(dv.slot[0].stream));
    }
    return FABGPU_OK;
}

// device temporaries released on every path (fabgpu_keys_register)
struct DevTmp {
    std::vector<void*> p;
    ~DevTmp() { for (void* q : p) if (q) cudaFree(q); }
    template <typename T> cudaError_t alloc(T*& out, size_t bytes) { void* q = nullptr; cudaError_t e = cudaMalloc(&q, bytes); out = (T*)q; if (e == cudaSuccess) p.push_back(q); return e; }
};

template <typename T> int grow_dev(fabgpu_ctx* ctx, T*& p, size_t bytes) { if (p) cudaFree(p); p = nullptr; CK(ctx, cudaMalloc(&p, bytes)); return FABGPU_OK; }
template <typename T> int grow_host(fabgpu_ctx* ctx, T*& p, size_t bytes) { if (p) cudaFreeHost(p); p = nullptr; CK(ctx, cudaHostAlloc(&p, bytes, cudaHostAllocPortable)); return FABGPU_OK; }

}  // namespace

extern "C" {

int fabgpu_init(const int* device_ids, int n_dev, size_t max_batch, fabgpu_ctx** out)
{
    if (!out) return FABGPU_E_ARG;
    *out = nullptr;
    fabgpu_ctx* ctx = new fabgpu_ctx();
    int rc = init_impl(ctx, device_ids, n_dev, max_batch);
    if (rc != FABGPU_OK) {
        g_init_error = ctx->last_error;
        free_all(ctx);
        delete ctx;
        return rc;
    }
    *out = ctx;
    return FABGPU_OK;
}

void fabgpu_destroy(fabgpu_ctx* ctx)
{
    if (!ctx) return;
    for (int s = 0; s < FABGPU_SLOTS; s++) wait_slot(ctx, s);
    free_all(ctx);
    delete ctx;
}

const char* fabgpu_last_error(const fabgpu_ctx* ctx) { return ctx ? ctx->last_error.c_str() : g_init_error.c_str(); }
int fabgpu_device_count(const fabgpu_ctx* ctx) { return ctx ? (int)ctx->devs.size() : 0; }
size_t fabgpu_max_batch(const fabgpu_ctx* ctx) { return ctx ? ctx->max_batch : 0; }
unsigned long long fabgpu_launch_count(const fabgpu_ctx* ctx) { return ctx ? ctx->launches.load() : 0ull; }

int fabgpu_host_buffers(fabgpu_ctx* ctx, int slot, uint8_t** qx, uint8_t** qy, uint8_t** e, uint8_t** r, uint8_t** s,
                        uint32_t** mask, uint32_t** offcurve)
{
    if (!ctx || slot < 0 || slot >= FABGPU_SLOTS) return FABGPU_E_ARG;
    HostSlot& hs = ctx->hslot[slot];
    if (qx) *qx = hs.h_in[0];
    if (qy) *qy = hs.h_in[1];
    if (e) *e = hs.h_in[2];
    if (r) *r = hs.h_in[3];
    if (s) *s = hs.h_in[4];
    if (mask) *mask = hs.h_mask;
    if (offcurve) *offcurve = hs.h_off;
    return FABGPU_OK;
}

static int verify_async_impl(fabgpu_ctx* ctx, int slot, size_t n, bool keyed)
{
    if (!ctx || slot < 0 || slot >= FABGPU_SLOTS) return FABGPU_E_ARG;
    std::shared_lock<std::shared_mutex> rl(ctx->tab_mu);     // handles -> slots -> enqueue, see fabgpu_ctx::tab_mu
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (n > ctx->max_batch) { ctx->last_error = "n exceeds max_batch"; return FABGPU_E_ARG; }
    if (fault_injected()) { ctx->last_error = "fault injected (FABGPU_FAULT_INJECT=1)"; return FABGPU_E_INJECTED; }
    return enqueue_slot(ctx, slot, n, keyed);
}

int fabgpu_verify_p256_async(fabgpu_ctx* ctx, int slot, size_t n) { return verify_async_impl(ctx, slot, n, false); }
int fabgpu_verify_p256_keyed_async(fabgpu_ctx* ctx, int slot, size_t n) { return verify_async_impl(ctx, slot, n, true); }

int fabgpu_verify_p256_keyed(fabgpu_ctx* ctx, int slot, size_t n)
{
    int rc = fabgpu_verify_p256_keyed_async(ctx, slot, n);
    if (rc) return rc;
    return fabgpu_wait(ctx, slot);
}

int fabgpu_host_key_slots(fabgpu_ctx* ctx, int slot, int32_t** key_slot)
{
    if (!ctx || slot < 0 || slot >= FABGPU_SLOTS || !key_slot) return FABGPU_E_ARG;
    *key_slot = ctx->hslot[slot].h_key_slot;
    return FABGPU_OK;
}

int fabgpu_key_slot_capacity(const fabgpu_ctx* ctx) { return ctx ? ctx->key_slots : 0; }

// Looks the keys up in the table cache and builds tables for the missing ones (one launch per device for the whole set).
int fabgpu_keys_register(fabgpu_ctx* ctx, const uint8_t* keys_xy, int K, int32_t* slots_out)
{
    if (!ctx || K < 0 || (K && (!keys_xy || !slots_out))) return FABGPU_E_ARG;
    // Fast path under the shared lock: every key already owns a table (the steady state of KeyImport / resolve_key_tables).
    {
        std::shared_lock<std::shared_mutex> rl(ctx->tab_mu);
        std::lock_guard<std::mutex> lk(ctx->mu);
        bool all = true;
        for (int k = 0; k < K && all; k++) all = ctx->key_map.count(std::string((const char*)keys_xy + 64 * (size_t)k, 64)) != 0;
        if (all) {
            ctx->tick++;
            for (int k = 0; k < K; k++) {
                const int sl = ctx->key_map[std::string((const char*)keys_xy + 64 * (size_t)k, 64)];
                slots_out[k] = make_handle(ctx, sl); ctx->slot_tick[sl] = ctx->tick;
            }
            return FABGPU_OK;
        }
    }
    std::unique_lock<std::shared_mutex> wl(ctx->tab_mu);
    std::lock_guard<std::mutex> lk(ctx->mu);
    std::vector<int> fresh;                      // indices into keys_xy that need a table
    std::vector<int32_t> fresh_slot;
    std::vector<char> slot_taken(ctx->key_slots, 0);
    ctx->tick++;
    for (int k = 0; k < K; k++) {
        std::string key((const char*)keys_xy + 64 * (size_t)k, 64);
        auto it = ctx->key_map.find(key);
        if (it != ctx->key_map.end()) { slots_out[k] = make_handle(ctx, it->second); ctx->slot_tick[it->second] = ctx->tick; slot_taken[it->second] = 1; continue; }
        // least recently used slot that this call has not touched
        int best = -1;
        for (int sl = 0; sl < ctx->key_slots; sl++)
            if (!slot_taken[sl] && (best < 0 || ctx->slot_tick[sl] < ctx->slot_tick[best])) best = sl;
        if (best < 0) { slots_out[k] = -1; continue; }            // more distinct keys in one call than slots: stays generic
        // The slot's old owner loses it NOW (its handles die with the generation bump), but the new key is mapped only after
        // its table exists on every device: a failure below leaves the slot empty, never pointing at another key's table.
        if (!ctx->slot_key[best].empty()) { ctx->key_map.erase(ctx->slot_key[best]); ctx->slot_key[best].clear(); ctx->slot_gen[best]++; }
        ctx->slot_tick[best] = ctx->tick; slot_taken[best] = 1;
        slots_out[k] = -1;
        fresh.push_back(k); fresh_slot.push_back(best);
    }
    if (fresh.empty()) return FABGPU_OK;
    const int F = (int)fresh.size();
    std::vector<uint8_t> fk(64 * (size_t)F);
    for (int i = 0; i < F; i++) memcpy(fk.data() + 64 * (size_t)i, keys_xy + 64 * (size_t)fresh[i], 64);
    std::vector<uint32_t> flags(F, 0);
    auto build_on = [&](Device& dv) -> int {
        DevTmp tmp;
        CK(ctx, cudaSetDevice(dv.id));
        // an evicted slot's table may still be read by a batch in flight: drain this device first (registration is rare)
        for (auto& ds : dv.slot) CK(ctx, cudaStreamSynchronize(ds.stream));
        CK(ctx, cudaDeviceSynchronize());            // launches on caller streams (fabgpu_verify_p256_device_keyed) as well
        uint8_t* d_keys = nullptr; int32_t* d_slots = nullptr; uint32_t* d_flags = nullptr; u256* d_scratch = nullptr;
        CK(ctx, tmp.alloc(d_keys, fk.size()));
        CK(ctx, tmp.alloc(d_slots, 4 * (size_t)F));
        CK(ctx, tmp.alloc(d_flags, 4 * (size_t)F));
        CK(ctx, cudaMemcpy(d_keys, fk.data(), fk.size(), cudaMemcpyHostToDevice));
        CK(ctx, cudaMemcpy(d_slots, fresh_slot.data(), 4 * (size_t)F, cudaMemcpyHostToDevice));
#if FAB_Q_TWO_LEVEL
        aff* d_small = nullptr;
        const size_t nsmall = ((size_t)1 << (FAB_WQ / 2)) - 1;
        const size_t threads = (size_t)F * FAB_Q_WINDOWS * 2;
        CK(ctx, tmp.alloc(d_scratch, threads * 2 * nsmall * sizeof(u256)));
        CK(ctx, tmp.alloc(d_small, threads * nsmall * sizeof(aff)));
        small_tables_kernel<<<(unsigned)((threads + 31) / 32), 32, 0, dv.slot[0].stream>>>(d_keys, F, FAB_WQ, FAB_Q_WINDOWS, d_small, d_scratch, d_flags);
        const size_t threads2 = (size_t)F * FAB_Q_WINDOWS * ((FAB_Q_ENTRIES + FAB_TAB_CHUNK - 1) / FAB_TAB_CHUNK);
        full_tables_kernel<<<(unsigned)((threads2 + 127) / 128), 128, 0, dv.slot[0].stream>>>(d_small, d_slots, d_flags, F, FAB_WQ, FAB_Q_WINDOWS, dv.qtab);
        ctx->launches += 2;
#else
        const size_t threads = (size_t)F * FAB_Q_WINDOWS;
        CK(ctx, tmp.alloc(d_scratch, threads * 2 * FAB_Q_ENTRIES * sizeof(u256)));
        build_key_tables_kernel<<<(unsigned)((threads + 31) / 32), 32, 0, dv.slot[0].stream>>>(d_keys, d_slots, F, dv.qtab, d_scratch, d_flags);
        ctx->launches++;
#endif
        CK(ctx, cudaGetLastError());
        CK(ctx, cudaStreamSynchronize(dv.slot[0].stream));
        CK(ctx, cudaMemcpy(flags.data(), d_flags, 4 * (size_t)F, cudaMemcpyDeviceToHost));
        return FABGPU_OK;
    };
    for (auto& dv : ctx->devs) {
        const int rc = build_on(dv);
        if (rc) return rc;                        // nothing was committed: the recycled slots stay empty (handles -1), the keys stay generic
    }
    for (int i = 0; i < F; i++) {
        if (!flags[i]) continue;                  // not a curve point: no table; the generic kernel reports it as off-curve
        const int sl = fresh_slot[i];
        std::string key((const char*)fk.data() + 64 * (size_t)i, 64);
        ctx->slot_key[sl] = key; ctx->key_map[key] = sl;
        slots_out[fresh[i]] = make_handle(ctx, sl);
    }
    return FABGPU_OK;
}

// Small tables for the keys that have none yet; handles_out[k] = small handle, or -1 when no slot could be had.  The builds are
// enqueued on every device's build stream and NOT waited for: consumers order themselves behind Device::s_ev (launch_verify).
// Caller holds neither tab_mu nor mu.
static int small_register(fabgpu_ctx* ctx, const uint8_t* keys_xy, int K, int32_t* handles_out)
{
    if (ctx->small_slots <= 0) { for (int k = 0; k < K; k++) handles_out[k] = -1; return FABGPU_OK; }
    {   // fast path under the shared lock: every key already owns a small table
        std::shared_lock<std::shared_mutex> rl(ctx->tab_mu);
        std::lock_guard<std::mutex> lk(ctx->mu);
        bool all = true;
        fabgpu_ctx::Key64 kk;
        for (int k = 0; k < K && all; k++) { memcpy(kk.b, keys_xy + 64 * (size_t)k, 64); all = ctx->small_map.count(kk) != 0; }
        if (all) {
            ctx->tick++;
            for (int k = 0; k < K; k++) {
                memcpy(kk.b, keys_xy + 64 * (size_t)k, 64);
                const int sl = ctx->small_map[kk];
                handles_out[k] = make_small_handle(ctx, sl); ctx->small_tick[sl] = ctx->tick;
            }
            return FABGPU_OK;
        }
    }
    const bool trace = getenv("FABGPU_TRACE") != nullptr;
    auto tnow = [] { return std::chrono::steady_clock::now(); };
    auto tus = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double, std::micro>(b - a).count(); };
    auto tr0 = tnow();
    std::unique_lock<std::shared_mutex> wl(ctx->tab_mu);
    std::lock_guard<std::mutex> lk(ctx->mu);
    auto tr1 = tnow();
    ctx->tick++;
    std::vector<int> fresh; std::vector<int32_t> fresh_slot;
    fabgpu_ctx::Key64 kk;
    int need = 0;
    for (int k = 0; k < K; k++) { memcpy(kk.b, keys_xy + 64 * (size_t)k, 64); if (!ctx->small_map.count(kk)) need++; }
    if (need > (int)ctx->small_free.size()) {
        // Out of free slots: recycle the least recently used ones in bulk (an eighth of the pool at least), after draining every device --
        // a batch in flight may still read them.  Rare by construction: the pool holds thousands of keys.
        for (auto& dv : ctx->devs) { CK(ctx, cudaSetDevice(dv.id)); CK(ctx, cudaDeviceSynchronize()); }
        std::vector<int> order;
        for (int sl = 0; sl < ctx->small_slots; sl++) if (ctx->small_used[sl]) order.push_back(sl);
        // keys of THIS call keep their tables
        for (int k = 0; k < K; k++) { memcpy(kk.b, keys_xy + 64 * (size_t)k, 64); auto it = ctx->small_map.find(kk); if (it != ctx->small_map.end()) ctx->small_tick[it->second] = ctx->tick; }
        std::sort(order.begin(), order.end(), [&](int a, int b) { return ctx->small_tick[a] < ctx->small_tick[b]; });
        const size_t want = std::max<size_t>((size_t)need - ctx->small_free.size(), (size_t)ctx->small_slots / 8);
        for (size_t i = 0; i < order.size() && i < want; i++) {
            const int sl = order[i];
            if (ctx->small_tick[sl] == ctx->tick) break;
            ctx->small_map.erase(ctx->small_key[sl]); ctx->small_used[sl] = 0; ctx->small_gen[sl]++;
            ctx->small_free.push_back(sl); ctx->small_recycled++;
        }
    }
    for (int k = 0; k < K; k++) {
        memcpy(kk.b, keys_xy + 64 * (size_t)k, 64);
        auto it = ctx->small_map.find(kk);
        if (it != ctx->small_map.end()) { handles_out[k] = make_small_handle(ctx, it->second); ctx->small_tick[it->second] = ctx->tick; continue; }
        handles_out[k] = -1;
        if (ctx->small_free.empty()) continue;                      // more distinct keys in one call than the pool holds: stays generic
        const int sl = ctx->small_free.back(); ctx->small_free.pop_back();
        // mapped at once (a duplicate later in this call finds it); un-mapped again below if the enqueue fails
        ctx->small_map[kk] = sl; ctx->small_key[sl] = kk; ctx->small_used[sl] = 1; ctx->small_tick[sl] = ctx->tick;
        fresh.push_back(k); fresh_slot.push_back(sl);
        handles_out[k] = make_small_handle(ctx, sl);
    }
    if (fresh.empty()) return FABGPU_OK;
    const int F = (int)fresh.size();
    ctx->small_built += (unsigned long long)F;
    std::vector<uint8_t> fk(64 * (size_t)F);
    for (int i = 0; i < F; i++) memcpy(fk.data() + 64 * (size_t)i, keys_xy + 64 * (size_t)fresh[i], 64);
    auto tr2 = tnow();
    auto build_on = [&](Device& dv) -> int {
        CK(ctx, cudaSetDevice(dv.id));
        auto b0 = tnow();
        if ((size_t)F > dv.s_cap) {
            CK(ctx, cudaStreamSynchronize(dv.s_stream));            // an earlier build may still use the scratch
            const size_t c = (size_t)F + (size_t)F / 2 + 256;
            void* old[] = {dv.s_bases, dv.s_keys, dv.s_slots};
            for (void* q : old) if (q) cudaFree(q);
            dv.s_bases = nullptr; dv.s_keys = nullptr; dv.s_slots = nullptr; dv.s_cap = 0;
            CK(ctx, cudaMalloc(&dv.s_bases, c * FAB_S_WINDOWS * sizeof(aff)));
            CK(ctx, cudaMalloc(&dv.s_keys, 64 * c));
            CK(ctx, cudaMalloc(&dv.s_slots, 4 * c));
            dv.s_cap = c;
        }
        auto b1 = tnow();
        CK(ctx, cudaMemcpyAsync(dv.s_keys, fk.data(), fk.size(), cudaMemcpyHostToDevice, dv.s_stream));
        CK(ctx, cudaMemcpyAsync(dv.s_slots, fresh_slot.data(), 4 * (size_t)F, cudaMemcpyHostToDevice, dv.s_stream));
        CK(ctx, cudaStreamSynchronize(dv.s_stream));                // the sources are local vectors
        auto b2 = tnow();
        small_bases_kernel<<<(unsigned)((F + 31) / 32), 32, 0, dv.s_stream>>>(dv.s_keys, dv.s_slots, F, dv.s_bases, dv.stab);
        small_windows_kernel<<<(unsigned)(((size_t)F * FAB_S_WINDOWS + 127) / 128), 128, 0, dv.s_stream>>>(dv.s_bases, dv.s_slots, F, dv.stab);
        ctx->launches += 2;
        CK(ctx, cudaGetLastError());
        CK(ctx, cudaEventRecord(dv.s_ev, dv.s_stream));
        dv.s_ev_set = true;
        if (trace) fprintf(stderr, "[fabgpu] small_register F=%d: lock %.0f us, bookkeeping %.0f us, scratch %.0f us, copies %.0f us, launches %.0f us\n", F, tus(tr0, tr1),
                           tus(tr1, tr2), tus(b0, b1), tus(b1, b2), tus(b2, tnow()));
        return FABGPU_OK;
    };
    for (auto& dv : ctx->devs) {
        const int rc = build_on(dv);
        if (rc) {                                                   // nothing usable was built: give the slots back, the keys stay generic
            for (int i = 0; i < F; i++) {
                const int sl = fresh_slot[i];
                ctx->small_map.erase(ctx->small_key[sl]); ctx->small_used[sl] = 0; ctx->small_gen[sl]++; ctx->small_free.push_back(sl);
                handles_out[fresh[i]] = -1;
            }
            return rc;
        }
    }
    return FABGPU_OK;
}

int fabgpu_keys_register_small(fabgpu_ctx* ctx, const uint8_t* keys_xy, int K, int32_t* handles_out)
{
    if (!ctx || K < 0 || (K && (!keys_xy || !handles_out))) return FABGPU_E_ARG;
    return small_register(ctx, keys_xy, K, handles_out);
}
int fabgpu_small_slot_capacity(const fabgpu_ctx* ctx) { return ctx ? ctx->small_slots : 0; }
void fabgpu_small_table_info(int* window_bits, int* windows, size_t* table_bytes)
{
    if (window_bits) *window_bits = FAB_WS;
    if (windows) *windows = FAB_S_WINDOWS;
    if (table_bytes) *table_bytes = (size_t)FAB_S_POINTS * sizeof(aff);
}
int fabgpu_key_table_stats(fabgpu_ctx* ctx, unsigned long long out[4])
{
    if (!ctx || !out) return FABGPU_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    out[0] = ctx->key_map.size(); out[1] = ctx->small_map.size(); out[2] = ctx->small_built; out[3] = ctx->small_recycled;
    return FABGPU_OK;
}

int fabgpu_wait(fabgpu_ctx* ctx, int slot)
{
    if (!ctx || slot < 0 || slot >= FABGPU_SLOTS) return FABGPU_E_ARG;
    // No context lock: waiting on one slot's streams must not block the enqueue of another slot (the provider's aggregator
    // fills slot k+1 while slot k runs).  Stream handles are immutable after fabgpu_init; errors go to a local string first.
    for (auto& dv : ctx->devs) {
        cudaError_t e = cudaSetDevice(dv.id);
        if (e == cudaSuccess) e = cudaStreamSynchronize(dv.slot[slot].stream);
        if (e != cudaSuccess) {
            std::lock_guard<std::mutex> lk(ctx->mu);
            ctx->last_error = std::string("cudaStreamSynchronize failed: ") + cudaGetErrorString(e);
            return FABGPU_E_CUDA;
        }
    }
    return FABGPU_OK;
}

int fabgpu_verify_p256(fabgpu_ctx* ctx, int slot, size_t n)
{
    int rc = fabgpu_verify_p256_async(ctx, slot, n);
    if (rc) return rc;
    return fabgpu_wait(ctx, slot);
}

int fabgpu_verify_p256_host(fabgpu_ctx* ctx, const uint8_t* qx, const uint8_t* qy, const uint8_t* e, const uint8_t* r,
                            const uint8_t* s, size_t n, uint32_t* mask, uint32_t* offcurve)
{
    if (!ctx || (n && (!qx || !qy || !e || !r || !s || !mask))) return FABGPU_E_ARG;
    if (n > ctx->max_batch) { ctx->last_error = "n exceeds max_batch"; return FABGPU_E_ARG; }
    std::lock_guard<std::mutex> lk0(ctx->slot0_mu);
    HostSlot& hs = ctx->hslot[0];
    const uint8_t* src[5] = {qx, qy, e, r, s};
    for (int a = 0; a < 5; a++) memcpy(hs.h_in[a], src[a], 32 * n);
    int rc = fabgpu_verify_p256(ctx, 0, n);
    if (rc) return rc;
    const size_t words = (n + 31) / 32;
    memcpy(mask, hs.h_mask, 4 * words);
    if (offcurve) memcpy(offcurve, hs.h_off, 4 * words);
    return FABGPU_OK;
}

int fabgpu_verify_p256_device(fabgpu_ctx* ctx, int dev_index, const void* d_qx, const void* d_qy, const void* d_e,
                              const void* d_r, const void* d_s, size_t n, void* d_mask, void* d_offcurve, void* cuda_stream)
{
    if (!ctx || dev_index < 0 || dev_index >= (int)ctx->devs.size()) return FABGPU_E_ARG;
    if (n && (!d_qx || !d_qy || !d_e || !d_r || !d_s || !d_mask)) return FABGPU_E_ARG;
    if (fault_injected()) { ctx->last_error = "fault injected (FABGPU_FAULT_INJECT=1)"; return FABGPU_E_INJECTED; }
    Device& dv = ctx->devs[dev_index];
    CK(ctx, cudaSetDevice(dv.id));
    cudaStream_t st = (cudaStream_t)cuda_stream;   // NULL is CUDA's default stream, exactly as in the runtime API
    return launch_verify(ctx, dv, MODE_GENERIC, nullptr, (const uint8_t*)d_qx, (const uint8_t*)d_qy, (const uint8_t*)d_e,
                         (const uint8_t*)d_r, (const uint8_t*)d_s, n, (uint32_t*)d_mask, (uint32_t*)d_offcurve, st);
}

int fabgpu_verify_p256_device_keyed(fabgpu_ctx* ctx, int dev_index, int all_cached, const void* d_key_slot, const void* d_qx,
                                    const void* d_qy, const void* d_e, const void* d_r, const void* d_s, size_t n, void* d_mask,
                                    void* d_offcurve, void* cuda_stream)
{
    if (!ctx || dev_index < 0 || dev_index >= (int)ctx->devs.size()) return FABGPU_E_ARG;
    if (n && (!d_key_slot || !d_e || !d_r || !d_s || !d_mask)) return FABGPU_E_ARG;
    if (n && !all_cached && (!d_qx || !d_qy)) return FABGPU_E_ARG;
    if (fault_injected()) { ctx->last_error = "fault injected (FABGPU_FAULT_INJECT=1)"; return FABGPU_E_INJECTED; }
    Device& dv = ctx->devs[dev_index];
    CK(ctx, cudaSetDevice(dv.id));
    return launch_verify(ctx, dv, all_cached == 2 ? MODE_SMALL : (all_cached ? MODE_CACHED : MODE_MIXED), (const int32_t*)d_key_slot, (const uint8_t*)d_qx,
                         (const uint8_t*)d_qy, (const uint8_t*)d_e, (const uint8_t*)d_r, (const uint8_t*)d_s, n, (uint32_t*)d_mask,
                         (uint32_t*)d_offcurve, (cudaStream_t)cuda_stream);
}

// ---- bitmask exchange over peer memory -------------------------------------------------------------------------------------
static const int kPeerGens = 2;
static size_t peer_buf_words(int world, size_t wpr) { return (size_t)kPeerGens * world * wpr + FAB_PEER_MAX; }

int fabgpu_peer_mask_create(fabgpu_ctx* ctx, int dev_index, int world, int rank, size_t words_per_rank, uint8_t handle_out[FABGPU_IPC_HANDLE_BYTES])
{
    if (!ctx || dev_index < 0 || dev_index >= (int)ctx->devs.size() || world < 1 || world > FAB_PEER_MAX || rank < 0 || rank >= world || !words_per_rank || !handle_out)
        return FABGPU_E_ARG;
    static_assert(sizeof(cudaIpcMemHandle_t) <= FABGPU_IPC_HANDLE_BYTES, "IPC handle size");
    Device& dv = ctx->devs[dev_index];
    auto& pr = dv.peer;
    if (pr.local) { ctx->last_error = "peer mask already created on this device"; return FABGPU_E_ARG; }
    CK(ctx, cudaSetDevice(dv.id));
    const size_t bytes = 4 * peer_buf_words(world, words_per_rank);
    CK(ctx, cudaMalloc(&pr.local, bytes));
    CK(ctx, cudaMemset(pr.local, 0, bytes));
    CK(ctx, cudaMalloc(&pr.done, 8));
    CK(ctx, cudaMemset(pr.done, 0, 8));
    pr.timeout = pr.done + 1;
    CK(ctx, cudaHostAlloc(&pr.h_timeout, 4, cudaHostAllocPortable));
    *pr.h_timeout = 0;
    cudaIpcMemHandle_t h;
    CK(ctx, cudaIpcGetMemHandle(&h, pr.local));
    memset(handle_out, 0, FABGPU_IPC_HANDLE_BYTES);
    memcpy(handle_out, &h, sizeof h);
    pr.world = world; pr.rank = rank; pr.words_per_rank = words_per_rank;
    for (int p = 0; p < FAB_PEER_MAX; p++) { pr.mapped[p] = nullptr; pr.opened[p] = false; }
    pr.mapped[rank] = pr.local;
    pr.ready = world == 1;
    return FABGPU_OK;
}

int fabgpu_peer_mask_open(fabgpu_ctx* ctx, int dev_index, const uint8_t* handles)
{
    if (!ctx || dev_index < 0 || dev_index >= (int)ctx->devs.size() || !handles) return FABGPU_E_ARG;
    Device& dv = ctx->devs[dev_index];
    auto& pr = dv.peer;
    if (!pr.local) { ctx->last_error = "fabgpu_peer_mask_create first"; return FABGPU_E_ARG; }
    CK(ctx, cudaSetDevice(dv.id));
    for (int p = 0; p < pr.world; p++) {
        if (p == pr.rank || pr.opened[p]) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, handles + (size_t)p * FABGPU_IPC_HANDLE_BYTES, sizeof h);
        void* m = nullptr;
        CK(ctx, cudaIpcOpenMemHandle(&m, h, cudaIpcMemLazyEnablePeerAccess));
        pr.mapped[p] = (uint32_t*)m; pr.opened[p] = true;
    }
    pr.ready = true;
    return FABGPU_OK;
}

int fabgpu_peer_mask_close(fabgpu_ctx* ctx, int dev_index)
{
    if (!ctx || dev_index < 0 || dev_index >= (int)ctx->devs.size()) return FABGPU_E_ARG;
    Device& dv = ctx->devs[dev_index];
    auto& pr = dv.peer;
    cudaSetDevice(dv.id);
    cudaDeviceSynchronize();
    for (int p = 0; p < FAB_PEER_MAX; p++) if (pr.opened[p]) { cudaIpcCloseMemHandle(pr.mapped[p]); pr.opened[p] = false; pr.mapped[p] = nullptr; }
    if (pr.local) cudaFree(pr.local);
    if (pr.done) cudaFree(pr.done);
    if (pr.h_timeout) cudaFreeHost(pr.h_timeout);
    pr = Device::Peer();
    return FABGPU_OK;
}

int fabgpu_verify_p256_device_keyed_allgather(fabgpu_ctx* ctx, int dev_index, int all_cached, const void* d_key_slot, const void* d_qx,
                                              const void* d_qy, const void* d_e, const void* d_r, const void* d_s, size_t n, uint32_t step,
                                              void** d_full_mask, void* cuda_stream)
{
    if (!ctx || dev_index < 0 || dev_index >= (int)ctx->devs.size() || !d_full_mask || step == 0) return FABGPU_E_ARG;
    if (n && (!d_key_slot || !d_e || !d_r || !d_s)) return FABGPU_E_ARG;
    if (n && !all_cached && (!d_qx || !d_qy)) return FABGPU_E_ARG;
    Device& dv = ctx->devs[dev_index];
    auto& pr = dv.peer;
    if (!pr.ready) { ctx->last_error = "peer masks are not set up (fabgpu_peer_mask_create / _open)"; return FABGPU_E_ARG; }
    if ((n + 31) / 32 > pr.words_per_rank) { ctx->last_error = "batch exceeds words_per_rank"; return FABGPU_E_ARG; }
    if (fault_injected()) { ctx->last_error = "fault injected (FABGPU_FAULT_INJECT=1)"; return FABGPU_E_INJECTED; }
    if (*pr.h_timeout) { ctx->last_error = "a peer did not publish its bitmask in time"; return FABGPU_E_CUDA; }
    CK(ctx, cudaSetDevice(dv.id));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    PeerOut po; memset(&po, 0, sizeof po);
    for (int p = 0; p < pr.world; p++) po.buf[p] = pr.mapped[p];
    po.done = pr.done; po.world = (uint32_t)pr.world; po.rank = (uint32_t)pr.rank; po.words_per_rank = (uint32_t)pr.words_per_rank;
    po.gen_off = (uint32_t)((step % kPeerGens) * pr.world * pr.words_per_rank);
    po.flag_off = (uint32_t)((size_t)kPeerGens * pr.world * pr.words_per_rank);
    po.step = step;
    // the rank's own words also land in its local segment (buf[rank] is the local buffer): `mask` for the kernels is that segment
    uint32_t* local_seg = pr.local + po.gen_off + (size_t)pr.rank * pr.words_per_rank;
    int rc = launch_verify(ctx, dv, all_cached == 2 ? MODE_SMALL : (all_cached ? MODE_CACHED : MODE_MIXED), (const int32_t*)d_key_slot, (const uint8_t*)d_qx, (const uint8_t*)d_qy,
                           (const uint8_t*)d_e, (const uint8_t*)d_r, (const uint8_t*)d_s, n, local_seg, nullptr, st, nullptr, 0, &po);
    if (rc) return rc;
    peer_wait_kernel<<<1, 32, 0, st>>>(pr.local + po.flag_off, po.world, step, pr.timeout);
    ctx->launches++;
    CK(ctx, cudaGetLastError());
    CK(ctx, cudaMemcpyAsync(pr.h_timeout, pr.timeout, 4, cudaMemcpyDeviceToHost, st));
    *d_full_mask = pr.local + po.gen_off;
    return FABGPU_OK;
}

int fabgpu_gate_signature(const uint8_t* sig, size_t sig_len, uint8_t r_out[32], uint8_t s_out[32])
{
    host::Gate g;
    host::gate_signature(sig, sig_len, g, false);
    if (g.status == FABGPU_ST_VALID) { memcpy(r_out, g.r, 32); memcpy(s_out, g.s, 32); }
    return g.status;
}


// fabgpu_bccsp_verify_batch with the gates on the device: the host only stages the raw blobs into pinned memory
// (parallel streaming copies) and reads one status byte per signature back.  Device 0 of the context.
// Device-gated batch, first half: stage into the slot's pinned buffers and enqueue copies + three kernels + the status
// read-back on the slot's stream.  Returns without waiting; the caller's buffers are no longer referenced.
// Grows the slot's pinned + device buffers of the device-gated batch path to the given capacities.
static int gate_bufs_reserve(fabgpu_ctx* ctx, int slot, size_t n, size_t sig_bytes, size_t dig_bytes, size_t K)
{
    auto& gb = ctx->gb[slot];
    int rc = 0;
    if (n > gb.n_cap) {
        const size_t c = round_up32(n + (n >> 2) + 1024);
        gb.n_cap = 0;
        rc |= grow_host(ctx, gb.h_sig_off, 4 * (c + 1)); rc |= grow_host(ctx, gb.h_dig_off, 4 * (c + 1)); rc |= grow_host(ctx, gb.h_kidx, 4 * c);
        rc |= grow_host(ctx, gb.h_status, c);
        rc |= grow_dev(ctx, gb.d_sig_off, 4 * (c + 1)); rc |= grow_dev(ctx, gb.d_dig_off, 4 * (c + 1)); rc |= grow_dev(ctx, gb.d_kidx, 4 * c);
        rc |= grow_dev(ctx, gb.d_status, c); rc |= grow_dev(ctx, gb.d_pre, c); rc |= grow_dev(ctx, gb.d_r, 32 * c); rc |= grow_dev(ctx, gb.d_s, 32 * c);
        rc |= grow_dev(ctx, gb.d_e, 32 * c); rc |= grow_dev(ctx, gb.d_qx, 32 * c); rc |= grow_dev(ctx, gb.d_qy, 32 * c); rc |= grow_dev(ctx, gb.d_ks, 4 * c);
        rc |= grow_dev(ctx, gb.d_mask, c / 8 + 8); rc |= grow_dev(ctx, gb.d_off, c / 8 + 8); rc |= grow_dev(ctx, gb.d_idx, 4 * (c + 2));
        if (rc) return FABGPU_E_CUDA;
        gb.n_cap = c;
    }
    if (sig_bytes > gb.sig_cap) { const size_t c = sig_bytes + (sig_bytes >> 2) + 4096; gb.sig_cap = 0; rc |= grow_host(ctx, gb.h_sigs, c); rc |= grow_dev(ctx, gb.d_sigs, c); if (rc) return FABGPU_E_CUDA; gb.sig_cap = c; }
    if (dig_bytes > gb.dig_cap) { const size_t c = dig_bytes + (dig_bytes >> 2) + 4096; gb.dig_cap = 0; rc |= grow_host(ctx, gb.h_digs, c); rc |= grow_dev(ctx, gb.d_digs, c); if (rc) return FABGPU_E_CUDA; gb.dig_cap = c; }
    if (K > gb.k_cap) {
        const size_t c = K + 64;
        gb.k_cap = 0;
        rc |= grow_host(ctx, gb.h_keys, 64 * c); rc |= grow_host(ctx, gb.h_slot_of, 4 * c); rc |= grow_dev(ctx, gb.d_keys, 64 * c); rc |= grow_dev(ctx, gb.d_slot_of, 4 * c);
        if (rc) return FABGPU_E_CUDA;
        gb.k_cap = c;
    }
    return FABGPU_OK;
}

// inplace: the batch already lies in the slot's pinned buffers (fabgpu_bccsp_batch_buffers): nothing is staged.
static int bccsp_device_submit(fabgpu_ctx* ctx, int slot, const uint8_t* keys_xy, int K, const int32_t* key_idx, const uint8_t* digests,
                               const uint32_t* dig_off, const uint8_t* sigs, const uint32_t* sig_off, size_t n,
                               const std::vector<int32_t>& slot_of, bool inplace = false)
{
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto us = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
        return std::chrono::duration<double, std::micro>(b - a).count();
    };
    auto t0 = now();
    Device& dv = ctx->devs[0];
    DevSlot& ds = dv.slot[slot];
    auto& gb = ctx->gb[slot];
    CK(ctx, cudaSetDevice(dv.id));
    // sig_off / dig_off may be a window of a longer table (a chunk of a call): bytes [off[0], off[n]) of the blobs belong to it
    const uint32_t sig_base = sig_off[0], dig_base = dig_off[0];
    const size_t sig_bytes = sig_off[n] - sig_base, dig_bytes = dig_off[n] - dig_base;
    int rc = gate_bufs_reserve(ctx, slot, n, sig_bytes, dig_bytes, (size_t)(K > 0 ? K : 0));
    if (rc) return rc;
    // stage: every host thread copies its slice of each array
    const int T = ctx->pool->size();
    bool all_slots = K > 0;
    int classes = K > 0 ? 0 : CLASS_GENERIC;                  // which non-big classes the batch holds (signatures with a bad key index are decided by the gates)
    std::shared_lock<std::shared_mutex> rl(ctx->tab_mu);      // held until the verify kernel is enqueued: the slots cannot be recycled in between
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        for (int k = 0; k < K; k++) {
            gb.h_slot_of[k] = handle_to_slot(ctx, slot_of[k]);
            if (gb.h_slot_of[k] < 0) all_slots = false;
            if (gb.h_slot_of[k] == -1) classes |= CLASS_GENERIC; else if (gb.h_slot_of[k] <= -2) classes |= CLASS_SMALL;
        }
    }
    if (K > 0 && !inplace) memcpy(gb.h_keys, keys_xy, 64 * (size_t)K);
    if (!inplace) ctx->pool->run([&](int tid) {
        auto slice = [&](size_t total, size_t& lo, size_t& hi) { lo = total * (size_t)tid / T; hi = total * (size_t)(tid + 1) / T; };
        size_t lo, hi;
        slice(sig_bytes, lo, hi); stage_copy(gb.h_sigs + lo, sigs + sig_base + lo, hi - lo);
        slice(dig_bytes, lo, hi); stage_copy(gb.h_digs + lo, digests + dig_base + lo, hi - lo);
        slice(4 * (n + 1), lo, hi); stage_copy((uint8_t*)gb.h_sig_off + lo, (const uint8_t*)sig_off + lo, hi - lo);
        slice(4 * (n + 1), lo, hi); stage_copy((uint8_t*)gb.h_dig_off + lo, (const uint8_t*)dig_off + lo, hi - lo);
        slice(4 * n, lo, hi); stage_copy((uint8_t*)gb.h_kidx + lo, (const uint8_t*)key_idx + lo, hi - lo);
        stage_fence();
    });
    auto t1 = now();
    cudaStream_t st = ds.stream;
    CK(ctx, cudaMemcpyAsync(gb.d_sigs, gb.h_sigs, sig_bytes, cudaMemcpyHostToDevice, st));
    CK(ctx, cudaMemcpyAsync(gb.d_digs, gb.h_digs, dig_bytes, cudaMemcpyHostToDevice, st));
    CK(ctx, cudaMemcpyAsync(gb.d_sig_off, gb.h_sig_off, 4 * (n + 1), cudaMemcpyHostToDevice, st));
    CK(ctx, cudaMemcpyAsync(gb.d_dig_off, gb.h_dig_off, 4 * (n + 1), cudaMemcpyHostToDevice, st));
    CK(ctx, cudaMemcpyAsync(gb.d_kidx, gb.h_kidx, 4 * n, cudaMemcpyHostToDevice, st));
    if (K > 0) {
        CK(ctx, cudaMemcpyAsync(gb.d_keys, gb.h_keys, 64 * (size_t)K, cudaMemcpyHostToDevice, st));
        CK(ctx, cudaMemcpyAsync(gb.d_slot_of, gb.h_slot_of, 4 * (size_t)K, cudaMemcpyHostToDevice, st));
    }
    bdev::bccsp_gate_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(gb.d_sigs, gb.d_sig_off, gb.d_digs, gb.d_dig_off, gb.d_kidx, gb.d_slot_of, gb.d_keys, K,
                                                                        (uint32_t)n, gb.d_r, gb.d_s, gb.d_e, gb.d_ks, (classes & CLASS_GENERIC) ? gb.d_qx : nullptr,
                                                                        (classes & CLASS_GENERIC) ? gb.d_qy : nullptr, gb.d_pre, sig_base, dig_base);
    ctx->launches++;
    CK(ctx, cudaGetLastError());
    rc = launch_verify(ctx, dv, all_slots ? MODE_CACHED : MODE_MIXED, gb.d_ks, gb.d_qx, gb.d_qy, gb.d_e, gb.d_r, gb.d_s, n, gb.d_mask, gb.d_off, st, nullptr, 0, nullptr,
                       gb.d_idx, classes ? classes : CLASS_GENERIC);
    if (rc) return rc;
    bdev::bccsp_status_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(gb.d_pre, gb.d_mask, gb.d_off, (uint32_t)n, gb.d_status);
    ctx->launches++;
    CK(ctx, cudaGetLastError());
    CK(ctx, cudaMemcpyAsync(gb.h_status, gb.d_status, n, cudaMemcpyDeviceToHost, st));
    gb.t_submit = t1; gb.n = n;
    ctx->timing[1] = us(t0, t1);
    return FABGPU_OK;
}

// Second half: wait for the slot's stream and hand the statuses out.
static int bccsp_device_finish(fabgpu_ctx* ctx, int slot, uint8_t* status)
{
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto us = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
        return std::chrono::duration<double, std::micro>(b - a).count();
    };
    auto& gb = ctx->gb[slot];
    CK(ctx, cudaSetDevice(ctx->devs[0].id));
    CK(ctx, cudaStreamSynchronize(ctx->devs[0].slot[slot].stream));
    auto t2 = now();
    memcpy(status, gb.h_status, gb.n);
    ctx->timing[2] = us(gb.t_submit, t2); ctx->timing[3] = us(t2, now());
    return FABGPU_OK;
}

// Which table serves each key of a call.  slot_of[k]: handle of key k's big table (>= 0), of its small table (<= -2), or -1.
//   * a key that already owns a table keeps using it, however few signatures it has in this call;
//   * >= key_min_uses signatures in this call earn the big table (what KeyImport does once per identity in the Go provider);
//   * otherwise the key's signatures are counted across calls, and small_min_uses of them earn a small table.
static int resolve_key_tables(fabgpu_ctx* ctx, const uint8_t* keys_xy, int K, const int32_t* key_idx, size_t n, std::vector<int32_t>& slot_of)
{
    slot_of.assign(K > 0 ? K : 0, -1);
    if (!(K > 0 && keys_xy && ctx->key_min_uses >= 0)) return FABGPU_OK;
    std::vector<uint32_t> uses(K, 0);
    for (size_t i = 0; i < n; i++) if (key_idx[i] >= 0 && key_idx[i] < K) uses[key_idx[i]]++;
    std::vector<int> want_big, want_small;
    {
        std::shared_lock<std::shared_mutex> rl(ctx->tab_mu);
        std::lock_guard<std::mutex> lk(ctx->mu);
        fabgpu_ctx::Key64 kk;
        bool touched = false;
        static thread_local std::string kbuf(64, '\0');          // lookup key without a heap allocation per key
        for (int k = 0; k < K; k++) {
            if (!uses[k]) continue;
            if (!ctx->key_map.empty() || uses[k] >= (uint32_t)ctx->key_min_uses) {
                memcpy(&kbuf[0], keys_xy + 64 * (size_t)k, 64);
                auto it = ctx->key_map.find(kbuf);
                if (it != ctx->key_map.end()) {
                    if (!touched) { ctx->tick++; touched = true; }
                    slot_of[k] = make_handle(ctx, it->second); ctx->slot_tick[it->second] = ctx->tick; continue;
                }
            }
            if (uses[k] >= (uint32_t)ctx->key_min_uses) { want_big.push_back(k); continue; }
            if (ctx->small_min_uses < 0) continue;
            memcpy(kk.b, keys_xy + 64 * (size_t)k, 64);
            auto sm = ctx->small_map.find(kk);
            if (sm != ctx->small_map.end()) {
                if (!touched) { ctx->tick++; touched = true; }
                slot_of[k] = make_small_handle(ctx, sm->second); ctx->small_tick[sm->second] = ctx->tick; continue;
            }
            uint32_t total = uses[k];
            if (total < (uint32_t)ctx->small_min_uses) {
                uint64_t h0, h1;
                memcpy(&h0, kk.b + 8, 8); memcpy(&h1, kk.b + 40, 8);
                const uint64_t tag = ((h0 * 0x9E3779B97F4A7C15ull) ^ (h1 * 0xC2B2AE3D27D4EB4Full)) | 1ull;
                const size_t b0 = (size_t)(tag >> 20) & (ctx->seen_tag.size() - 1) & ~(size_t)3;   // bucket of four entries
                size_t at = b0, weakest = b0;
                bool found = false;
                for (size_t q = b0; q < b0 + 4 && !found; q++) {
                    if (ctx->seen_tag[q] == tag) { at = q; found = true; }
                    else if (ctx->seen_tag[q] == 0) { if (ctx->seen_tag[weakest] != 0) weakest = q; }
                    else if (ctx->seen_tag[weakest] != 0 && ctx->seen_cnt[q] < ctx->seen_cnt[weakest]) weakest = q;
                }
                if (!found) { at = weakest; ctx->seen_tag[at] = tag; ctx->seen_cnt[at] = 0; }      // an empty entry, else the least used one
                ctx->seen_cnt[at] += uses[k];
                total = ctx->seen_cnt[at];
                if (total >= (uint32_t)ctx->small_min_uses) { ctx->seen_tag[at] = 0; ctx->seen_cnt[at] = 0; }
            }
            if (total >= (uint32_t)ctx->small_min_uses) want_small.push_back(k);
        }
    }
    if (!want_big.empty() && (int)want_big.size() <= ctx->key_slots) {
        std::vector<uint8_t> wk(64 * want_big.size());
        std::vector<int32_t> ws(want_big.size(), -1);
        for (size_t i = 0; i < want_big.size(); i++) memcpy(wk.data() + 64 * i, keys_xy + 64 * (size_t)want_big[i], 64);
        int rc = fabgpu_keys_register(ctx, wk.data(), (int)want_big.size(), ws.data());
        if (rc) return rc;
        for (size_t i = 0; i < want_big.size(); i++) slot_of[want_big[i]] = ws[i];
    } else if (ctx->small_min_uses >= 0) {
        for (int k : want_big) want_small.push_back(k);              // more busy keys than big slots: the small tier takes them
    }
    if (!want_small.empty()) {
        std::vector<uint8_t> wk(64 * want_small.size());
        std::vector<int32_t> ws(want_small.size(), -1);
        for (size_t i = 0; i < want_small.size(); i++) memcpy(wk.data() + 64 * i, keys_xy + 64 * (size_t)want_small[i], 64);
        int rc = small_register(ctx, wk.data(), (int)want_small.size(), ws.data());
        if (rc) return rc;
        for (size_t i = 0; i < want_small.size(); i++) slot_of[want_small[i]] = ws[i];
    }
    return FABGPU_OK;
}

// Default: gates on the device (one context device; a multi-device context keeps the host-gated split).
static bool device_gates_apply(const fabgpu_ctx* ctx, const uint32_t* dig_off, const uint32_t* sig_off, size_t n)
{
    const char* dg = getenv("FABGPU_BCCSP_HOST_GATES");
    return !(dg && dg[0] == '1') && ctx->devs.size() == 1 && n > 0 && n < (1u << 27) && sig_off[n] < (1u << 31) && dig_off[n] < (1u << 31);
}

static int bccsp_batch_hostgated(fabgpu_ctx* ctx, const uint8_t* keys_xy, int K, const int32_t* key_idx, const uint8_t* digests,
                                 const uint32_t* dig_off, const uint8_t* sigs, const uint32_t* sig_off, size_t n, uint8_t* status,
                                 const std::vector<int32_t>& slot_of);

int fabgpu_bccsp_verify_batch_async(fabgpu_ctx* ctx, int slot, const uint8_t* keys_xy, int K, const int32_t* key_idx, const uint8_t* digests,
                                    const uint32_t* dig_off, const uint8_t* sigs, const uint32_t* sig_off, size_t n)
{
    if (!ctx || slot < 0 || slot >= FABGPU_SLOTS || (n && (!key_idx || !dig_off || !sig_off))) return FABGPU_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->gb_mu[slot]);
    std::lock_guard<std::mutex> lk0(ctx->slot0_mu);       // host threads (staging pool) and the key cache: one submitter at a time
    auto& gb = ctx->gb[slot];
    if (gb.busy) { ctx->last_error = "slot already holds a batch: call fabgpu_bccsp_verify_batch_wait first"; return FABGPU_E_ARG; }
    auto t_start = std::chrono::steady_clock::now();
    ctx->timing[0] = ctx->timing[1] = ctx->timing[2] = ctx->timing[3] = 0;
    std::vector<int32_t> slot_of;
    int rc = resolve_key_tables(ctx, keys_xy, K, key_idx, n, slot_of);
    if (rc) return rc;
    ctx->timing[0] = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t_start).count();
    if (fault_injected()) { ctx->last_error = "fault injected (FABGPU_FAULT_INJECT=1)"; return FABGPU_E_INJECTED; }
    gb.n = n;
    if (device_gates_apply(ctx, dig_off, sig_off, n)) {
        rc = bccsp_device_submit(ctx, slot, keys_xy, K, key_idx, digests, dig_off, sigs, sig_off, n, slot_of);
        if (rc) { cudaStreamSynchronize(ctx->devs[0].slot[slot].stream); return rc; }
        gb.on_device = true;
    } else {
        // host-gated split (several devices, or FABGPU_BCCSP_HOST_GATES=1): it pipelines internally over both pinned SoA
        // slots, so it completes here and _wait only hands the statuses out
        gb.done_status.assign(n, 0);
        if (n) { rc = bccsp_batch_hostgated(ctx, keys_xy, K, key_idx, digests, dig_off, sigs, sig_off, n, gb.done_status.data(), slot_of); if (rc) return rc; }
        gb.on_device = false;
    }
    gb.busy = true;
    return FABGPU_OK;
}

int fabgpu_bccsp_batch_buffers(fabgpu_ctx* ctx, int slot, size_t n_cap, size_t sig_bytes_cap, size_t dig_bytes_cap, int k_cap, uint8_t** keys_xy,
                               int32_t** key_idx, uint8_t** digests, uint32_t** dig_off, uint8_t** sigs, uint32_t** sig_off)
{
    if (!ctx || slot < 0 || slot >= FABGPU_SLOTS || k_cap < 0 || !keys_xy || !key_idx || !digests || !dig_off || !sigs || !sig_off) return FABGPU_E_ARG;
    if (ctx->devs.size() != 1) { ctx->last_error = "the in-place batch form runs the gates on the device: single-device contexts only"; return FABGPU_E_ARG; }
    std::lock_guard<std::mutex> lk(ctx->gb_mu[slot]);
    auto& gb = ctx->gb[slot];
    if (gb.busy) { ctx->last_error = "slot holds a batch in flight"; return FABGPU_E_ARG; }
    CK(ctx, cudaSetDevice(ctx->devs[0].id));
    int rc = gate_bufs_reserve(ctx, slot, n_cap, sig_bytes_cap, dig_bytes_cap, (size_t)k_cap);
    if (rc) return rc;
    *keys_xy = gb.h_keys; *key_idx = gb.h_kidx; *digests = gb.h_digs; *dig_off = gb.h_dig_off; *sigs = gb.h_sigs; *sig_off = gb.h_sig_off;
    return FABGPU_OK;
}

int fabgpu_bccsp_verify_batch_inplace_async(fabgpu_ctx* ctx, int slot, int K, size_t n)
{
    if (!ctx || slot < 0 || slot >= FABGPU_SLOTS || K < 0) return FABGPU_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->gb_mu[slot]);
    std::lock_guard<std::mutex> lk0(ctx->slot0_mu);
    auto& gb = ctx->gb[slot];
    if (gb.busy) { ctx->last_error = "slot already holds a batch: call fabgpu_bccsp_verify_batch_wait first"; return FABGPU_E_ARG; }
    if (n > gb.n_cap || (size_t)K > gb.k_cap || !gb.h_sig_off) { ctx->last_error = "batch exceeds the capacities given to fabgpu_bccsp_batch_buffers"; return FABGPU_E_ARG; }
    if (n && (gb.h_sig_off[0] != 0 || gb.h_dig_off[0] != 0 || gb.h_sig_off[n] > gb.sig_cap || gb.h_dig_off[n] > gb.dig_cap)) {
        ctx->last_error = "offset tables must start at 0 and stay inside the buffers"; return FABGPU_E_ARG;
    }
    if (!device_gates_apply(ctx, gb.h_dig_off, gb.h_sig_off, n) && n) { ctx->last_error = "the in-place batch form needs the device gates"; return FABGPU_E_ARG; }
    auto t_start = std::chrono::steady_clock::now();
    ctx->timing[0] = ctx->timing[1] = ctx->timing[2] = ctx->timing[3] = 0;
    std::vector<int32_t> slot_of;
    int rc = resolve_key_tables(ctx, gb.h_keys, K, gb.h_kidx, n, slot_of);
    if (rc) return rc;
    ctx->timing[0] = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t_start).count();
    if (fault_injected()) { ctx->last_error = "fault injected (FABGPU_FAULT_INJECT=1)"; return FABGPU_E_INJECTED; }
    gb.n = n;
    if (n) {
        rc = bccsp_device_submit(ctx, slot, gb.h_keys, K, gb.h_kidx, gb.h_digs, gb.h_dig_off, gb.h_sigs, gb.h_sig_off, n, slot_of, true);
        if (rc) { cudaStreamSynchronize(ctx->devs[0].slot[slot].stream); return rc; }
        gb.on_device = true;
    } else { gb.done_status.clear(); gb.on_device = false; }
    gb.busy = true;
    return FABGPU_OK;
}

int fabgpu_bccsp_verify_batch_wait(fabgpu_ctx* ctx, int slot, uint8_t* status, size_t n)
{
    if (!ctx || slot < 0 || slot >= FABGPU_SLOTS) return FABGPU_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->gb_mu[slot]);
    auto& gb = ctx->gb[slot];
    if (!gb.busy) { ctx->last_error = "no batch in flight on this slot"; return FABGPU_E_ARG; }
    if (n != gb.n || (n && !status)) { ctx->last_error = "status buffer does not match the submitted batch"; return FABGPU_E_ARG; }
    gb.busy = false;
    if (gb.on_device) return bccsp_device_finish(ctx, slot, status);
    if (n) memcpy(status, gb.done_status.data(), n);
    return FABGPU_OK;
}

int fabgpu_bccsp_verify_batch(fabgpu_ctx* ctx, const uint8_t* keys_xy, int K, const int32_t* key_idx, const uint8_t* digests,
                              const uint32_t* dig_off, const uint8_t* sigs, const uint32_t* sig_off, size_t n, uint8_t* status)
{
    if (!ctx || (n && (!status || !key_idx || !dig_off || !sig_off))) return FABGPU_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->sync_mu);        // one synchronous caller at a time
    // A large call is cut into one chunk per slot: the copy of chunk c+1 runs under the kernels of chunk c and all chunks' verify
    // launches are resident together (they fill the machine like one launch).  Needs every slot free; otherwise, and for
    // small calls, the whole batch goes through slot 0.
    if (n >= 24576 && device_gates_apply(ctx, dig_off, sig_off, n)) {
        std::unique_lock<std::mutex> l[FABGPU_SLOTS];
        bool all_free = true;
        for (int c = 0; c < FABGPU_SLOTS; c++) { l[c] = std::unique_lock<std::mutex>(ctx->gb_mu[c]); all_free = all_free && !ctx->gb[c].busy; }
        if (all_free) {
            size_t lo[FABGPU_SLOTS + 1];
            for (int c = 0; c <= FABGPU_SLOTS; c++) lo[c] = n * (size_t)c / FABGPU_SLOTS;
            int submitted = 0, rc = FABGPU_OK;
            {
                std::lock_guard<std::mutex> lk0(ctx->slot0_mu);
                auto t_start = std::chrono::steady_clock::now();
                ctx->timing[0] = ctx->timing[1] = ctx->timing[2] = ctx->timing[3] = 0;
                std::vector<int32_t> slot_of;
                rc = resolve_key_tables(ctx, keys_xy, K, key_idx, n, slot_of);
                ctx->timing[0] = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t_start).count();
                if (!rc && fault_injected()) { ctx->last_error = "fault injected (FABGPU_FAULT_INJECT=1)"; rc = FABGPU_E_INJECTED; }
                for (int c = 0; c < FABGPU_SLOTS && !rc; c++) {
                    rc = bccsp_device_submit(ctx, c, keys_xy, K, key_idx + lo[c], digests, dig_off + lo[c], sigs, sig_off + lo[c], lo[c + 1] - lo[c], slot_of);
                    if (!rc) submitted++;
                }
            }
            for (int c = 0; c < submitted; c++) {                       // drain what was enqueued even after an error
                int rc2 = bccsp_device_finish(ctx, c, status + lo[c]);
                if (!rc) rc = rc2;
            }
            if (rc && submitted < FABGPU_SLOTS) cudaStreamSynchronize(ctx->devs[0].slot[submitted].stream);   // a submit that failed half-way
            return rc;
        }
    }
    int rc = fabgpu_bccsp_verify_batch_async(ctx, 0, keys_xy, K, key_idx, digests, dig_off, sigs, sig_off, n);
    if (rc) return rc;
    return fabgpu_bccsp_verify_batch_wait(ctx, 0, status, n);
}

// Host-gated form.  Gates run on the context's host threads; a signature that fails a gate keeps its position with
// r = s = 0 (the kernel rejects it at once) so that packing needs no compaction and stays parallel.
static int bccsp_batch_hostgated(fabgpu_ctx* ctx, const uint8_t* keys_xy, int K, const int32_t* key_idx, const uint8_t* digests,
                                 const uint32_t* dig_off, const uint8_t* sigs, const uint32_t* sig_off, size_t n, uint8_t* status,
                                 const std::vector<int32_t>& slot_of)
{
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto us = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
        return std::chrono::duration<double, std::micro>(b - a).count();
    };
    // The call is cut into chunks that alternate between the two pinned slots: while the GPU works on one chunk the
    // host threads gate and pack the next, and the statuses of the chunk before are scattered.
    const int T = ctx->pool->size();
    size_t chunk = ctx->max_batch;
    if (n > 16384) {
        const char* ev = getenv("FABGPU_E2E_CHUNKS");
        const size_t parts = ev ? (size_t)std::max(1, atoi(ev)) : 4;
        chunk = std::min(ctx->max_batch, std::max((size_t)8192, round_up32((n + parts - 1) / parts)));
    }
    struct InFlight { bool active = false; size_t base = 0, cnt = 0; } fl[FABGPU_SLOTS];
    auto retire = [&](int sl) -> int {
        if (!fl[sl].active) return FABGPU_OK;
        auto a = now();
        int rc = fabgpu_wait(ctx, sl);
        auto b = now();
        ctx->timing[2] += us(a, b);
        if (rc) return rc;
        HostSlot& hsl = ctx->hslot[sl];
        const size_t base = fl[sl].base, cnt = fl[sl].cnt;
        ctx->pool->run([&](int tid) {
            const size_t lo = cnt * (size_t)tid / T, hi = cnt * (size_t)(tid + 1) / T;
            for (size_t k = lo; k < hi; k++) {
                if (status[base + k] != FABGPU_ST_VALID) continue;          // decided by a gate
                const bool ok = (hsl.h_mask[k >> 5] >> (k & 31)) & 1u;
                const bool oc = (hsl.h_off[k >> 5] >> (k & 31)) & 1u;
                status[base + k] = ok ? FABGPU_ST_VALID : (oc ? FABGPU_ST_ERR_OFF_CURVE : FABGPU_ST_INVALID);
            }
        });
        fl[sl].active = false;
        ctx->timing[3] += us(b, now());
        return FABGPU_OK;
    };
    int sl = 0;
    static const uint8_t kZero32[32] = {0};
    for (size_t base = 0; base < n; base += chunk, sl = (sl + 1) % FABGPU_SLOTS) {
        const size_t cnt = std::min(chunk, n - base);
        int rc = retire(sl);
        if (rc) return rc;
        HostSlot& hs = ctx->hslot[sl];
        std::atomic<size_t> asked{0};
        auto t0 = now();
        ctx->pool->run([&](int tid) {
            const size_t b = cnt * (size_t)tid / T, e = cnt * (size_t)(tid + 1) / T;
            size_t mine = 0;
            for (size_t k = b; k < e; k++) {
                const size_t i = base + k;
                const int32_t ki = key_idx[i];
                const size_t sl_ = sig_off[i + 1] - sig_off[i], dl = dig_off[i + 1] - dig_off[i];
                uint8_t st;
                if (ki < 0) st = FABGPU_ST_ERR_NIL_KEY;                    // bccsp/sw/impl.go:249-251
                else if (sl_ == 0) st = FABGPU_ST_ERR_EMPTY_SIG;           // :252-254
                else if (dl == 0) st = FABGPU_ST_ERR_EMPTY_DIGEST;         // :255-257
                else if (ki >= K || !keys_xy) st = FABGPU_ST_ERR_UNSUPPORTED_KEY;
                else {
                    host::Gate g;
                    host::gate_signature(sigs + sig_off[i], sl_, g, false);
                    st = (uint8_t)g.status;
                    if (g.status == FABGPU_ST_VALID) {
                        uint8_t ebuf[32];
                        host::hash_to_e(digests + dig_off[i], dl, ebuf);
                        // Qx / Qy are staged even for keys with a table: the handle is resolved again at enqueue time and, had
                        // the slot been recycled by then, the generic kernel verifies against these (never against stale bytes)
                        stage32(hs.h_in[0] + 32 * k, keys_xy + 64 * (size_t)ki);
                        stage32(hs.h_in[1] + 32 * k, keys_xy + 64 * (size_t)ki + 32);
                        stage32(hs.h_in[2] + 32 * k, ebuf);
                        stage32(hs.h_in[3] + 32 * k, g.r);
                        stage32(hs.h_in[4] + 32 * k, g.s);
                        mine++;
                    }
                }
                if (st != FABGPU_ST_VALID) { stage32(hs.h_in[3] + 32 * k, kZero32); stage32(hs.h_in[4] + 32 * k, kZero32); }
                stage_i32(hs.h_key_slot + k, (st == FABGPU_ST_VALID) ? slot_of[ki] : -1);
                status[i] = st;
            }
            stage_fence();
            asked += mine;
        });
        auto t1 = now();
        ctx->timing[1] += us(t0, t1);
        if (asked.load() == 0) continue;
        rc = fabgpu_verify_p256_keyed_async(ctx, sl, cnt);
        if (rc) return rc;
        fl[sl].active = true; fl[sl].base = base; fl[sl].cnt = cnt;
        ctx->timing[2] += us(t1, now());
    }
    // drain in launch order
    for (int k = 0; k < FABGPU_SLOTS; k++, sl = (sl + 1) % FABGPU_SLOTS) {
        int rc = retire(sl);
        if (rc) return rc;
    }
    return FABGPU_OK;
}

void fabgpu_build_info(int* g_window_bits, int* key_window_bits)
{
    if (g_window_bits) *g_window_bits = FAB_WG;
    if (key_window_bits) *key_window_bits = FAB_WQ;
}

int fabgpu_last_timing(const fabgpu_ctx* ctx, double out_us[4])
{
    if (!ctx || !out_us) return FABGPU_E_ARG;
    for (int i = 0; i < 4; i++) out_us[i] = ctx->timing[i];
    return FABGPU_OK;
}

int fabgpu_bccsp_verify(fabgpu_ctx* ctx, const uint8_t* key_xy, const uint8_t* sig, size_t sig_len, const uint8_t* digest,
                        size_t digest_len, int* valid, char* err, size_t errcap)
{
    if (!ctx || !valid) return FABGPU_E_ARG;
    *valid = 0;
    std::string msg;
    auto finish = [&](const std::string& m) {
        if (err && errcap) { size_t k = std::min(errcap - 1, m.size()); memcpy(err, m.data(), k); err[k] = 0; }
        return FABGPU_OK;
    };
    // sw.CSP.Verify argument gates, reference bccsp/sw/impl.go:249-257
    if (!key_xy) return finish("Invalid Key. It must not be nil.");
    if (!sig || sig_len == 0) return finish("Invalid signature. Cannot be empty.");
    if (!digest || digest_len == 0) return finish("Invalid digest. Cannot be empty.");
    host::Gate g;
    host::gate_signature(sig, sig_len, g, true);
    if (g.status != FABGPU_ST_VALID && g.status != FABGPU_ST_INVALID)
        return finish("Failed verifing with opts [<nil>]: " + g.err);          // errors.Wrapf at impl.go:266
    if (g.status == FABGPU_ST_INVALID) return finish("");                       // r >= 2^256: (false, nil)
    uint8_t e[32];
    host::hash_to_e(digest, digest_len, e);
    uint32_t mask = 0, off = 0;
    int rc = fabgpu_verify_p256_host(ctx, key_xy, key_xy + 32, e, g.r, g.s, 1, &mask, &off);
    if (rc) return rc;
    if (off & 1u) { ctx->last_error = "public key is not on P-256"; return FABGPU_E_ARG; }
    *valid = (int)(mask & 1u);
    return finish("");
}

// ---- block-level pre-pass -------------------------------------------------------------------------------------------

// Device copy of the MSP view and the policy for block_plan_kernel / block_decide_kernel (device 0 of the context).
static int upload_msp(fabgpu_ctx* ctx, const uint8_t* id_blob, const uint32_t* id_off, const uint8_t* keys_xy, const uint8_t* valid, int n_ids,
                      const int32_t* policy_nodes, int n_nodes)
{
    std::lock_guard<std::mutex> lk0(ctx->slot0_mu);
    auto& dm = ctx->dm;
    CK(ctx, cudaSetDevice(ctx->devs[0].id));
    // blocks already enqueued on a slot were launched with the OLD tables (passed by value): let them finish before those go away
    for (auto& ds : ctx->devs[0].slot) CK(ctx, cudaStreamSynchronize(ds.stream));
    void* old[] = {dm.id_blob, dm.valid, dm.keys_xy, dm.channel, dm.id_off, dm.key_slot, dm.msp_code, dm.ht_idx, dm.nodes, dm.principal_code, dm.ht_hash,
                   dm.group, dm.ns_blob, dm.ns_off, dm.ns_root, dm.hash_kind};
    for (void* p : old) if (p) cudaFree(p);
    dm = fabgpu_ctx::DevMsp();
    // MSP-id codes: equal strings <=> equal codes, shared between identities and policy principals
    std::unordered_map<std::string, int32_t> codes;
    auto code_of = [&](const std::string& sname) { auto it = codes.find(sname); if (it != codes.end()) return it->second; int32_t c = (int32_t)codes.size(); codes[sname] = c; return c; };
    std::vector<int32_t> msp_code(n_ids > 0 ? n_ids : 1, -1), pcode(ctx->principals.size() ? ctx->principals.size() : 1, -1);
    for (int i = 0; i < n_ids; i++) msp_code[i] = code_of(ctx->msp.mspid[i]);
    for (size_t i = 0; i < ctx->principals.size(); i++) pcode[i] = code_of(ctx->principals[i]);
    uint32_t hsz = 8; while (hsz < (uint32_t)(4 * n_ids + 8)) hsz <<= 1;
    std::vector<uint64_t> hh(hsz, 0); std::vector<int32_t> hi(hsz, -1);
    for (int i = 0; i < n_ids; i++) {
        const uint64_t hv = bdev::sample_hash(id_blob + id_off[i], id_off[i + 1] - id_off[i]);
        uint32_t pos = (uint32_t)hv & (hsz - 1);
        while (hh[pos] != 0) pos = (pos + 1) & (hsz - 1);
        hh[pos] = hv; hi[pos] = i;
    }
    dm.all_slots = true;
    std::vector<int32_t> raw_slot(n_ids > 0 ? n_ids : 1, -1);
    dm.classes = 0;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        for (int i = 0; i < n_ids; i++) {
            raw_slot[i] = handle_to_slot(ctx, ctx->identity_slot[i]);
            if (raw_slot[i] < 0) { dm.all_slots = false; dm.classes |= raw_slot[i] == -1 ? CLASS_GENERIC : CLASS_SMALL; }
        }
    }
    auto up = [&](auto*& dst, const void* src, size_t bytes) -> int {
        CK(ctx, cudaMalloc(&dst, bytes + 8));                 // slack: word-wise readers may touch the aligned word past the end
        if (bytes) CK(ctx, cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice));
        return FABGPU_OK;
    };
    const size_t blob_len = n_ids ? id_off[n_ids] : 0;
    int rc = 0;
    rc |= up(dm.id_blob, id_blob, blob_len);
    rc |= up(dm.id_off, id_off, 4 * (size_t)(n_ids + 1) * (n_ids ? 1 : 0));
    rc |= up(dm.valid, valid, (size_t)n_ids);
    rc |= up(dm.keys_xy, keys_xy, 64 * (size_t)n_ids);
    rc |= up(dm.key_slot, raw_slot.data(), 4 * (size_t)n_ids);
    rc |= up(dm.msp_code, msp_code.data(), 4 * (size_t)n_ids);
    rc |= up(dm.ht_hash, hh.data(), 8 * (size_t)hsz);
    rc |= up(dm.ht_idx, hi.data(), 4 * (size_t)hsz);
    rc |= up(dm.nodes, policy_nodes, 16 * (size_t)n_nodes);
    rc |= up(dm.principal_code, pcode.data(), 4 * ctx->principals.size());
    rc |= up(dm.channel, ctx->channel.data(), ctx->channel.size());
    const std::vector<uint8_t> sha2(n_ids > 0 ? n_ids : 1, SHA_KIND_SHA2);      // every identity SHA-256 until fabgpu_msp_hash_families
    rc |= up(dm.hash_kind, sha2.data(), (size_t)n_ids);
    if (rc) return FABGPU_E_CUDA;
    dm.ht_size = n_ids ? hsz : 0; dm.n_ids = n_ids; dm.n_nodes = n_nodes; dm.n_principals = (int32_t)ctx->principals.size();
    dm.channel_len = (uint32_t)ctx->channel.size();
    return FABGPU_OK;
}


// An MSP with more identities than window-table slots: every identity gets a small table; the ones whose key ALREADY owns a window table --
// the integrator registered the few busy ones (the endorsing peers) with fabgpu_keys_register beforehand -- keep using that.
static int msp_small_tier(fabgpu_ctx* ctx, const uint8_t* keys_xy, int n_ids)
{
    int rc = small_register(ctx, keys_xy, n_ids, ctx->identity_slot.data());
    if (rc) return rc;
    std::shared_lock<std::shared_mutex> rl(ctx->tab_mu);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (ctx->key_map.empty()) return FABGPU_OK;
    std::string kbuf(64, '\0');
    for (int i = 0; i < n_ids; i++) {
        memcpy(&kbuf[0], keys_xy + 64 * (size_t)i, 64);
        auto it = ctx->key_map.find(kbuf);
        if (it != ctx->key_map.end()) ctx->identity_slot[i] = make_handle(ctx, it->second);
    }
    return FABGPU_OK;
}

int fabgpu_msp_configure(fabgpu_ctx* ctx, const uint8_t* id_blob, const uint32_t* id_off, const uint8_t* mspid_blob,
                         const uint32_t* mspid_off, const uint8_t* keys_xy, const uint8_t* valid, int n_ids,
                         const int32_t* policy_nodes, int n_nodes, const uint8_t* principal_blob, const uint32_t* principal_off,
                         int n_principals, const char* channel_id)
{
    if (!ctx || n_ids < 0 || n_nodes < 0 || n_principals < 0 || !channel_id) return FABGPU_E_ARG;
    if (n_ids && (!id_blob || !id_off || !mspid_blob || !mspid_off || !keys_xy || !valid)) return FABGPU_E_ARG;
    {
        std::lock_guard<std::mutex> lk0(ctx->slot0_mu);
        ctx->msp = blockval::MspTable();
        for (int i = 0; i < n_ids; i++) {
            ctx->msp.add(id_blob + id_off[i], id_off[i + 1] - id_off[i]);
            ctx->msp.mspid.emplace_back((const char*)mspid_blob + mspid_off[i], mspid_off[i + 1] - mspid_off[i]);
        }
        ctx->msp.keys_xy.assign(keys_xy, keys_xy + 64 * (size_t)n_ids);
        ctx->msp.valid.assign(valid, valid + n_ids);
        ctx->policy.clear();
        for (int i = 0; i < n_nodes; i++)
            ctx->policy.push_back({policy_nodes[4 * i], policy_nodes[4 * i + 1], policy_nodes[4 * i + 2], policy_nodes[4 * i + 3]});
        for (const auto& nd : ctx->policy)
            if (nd.type == 0 && (nd.first_child < 0 || nd.n_children < 0 || nd.first_child + nd.n_children > n_nodes)) {
                ctx->last_error = "policy node children out of range"; return FABGPU_E_ARG;
            }
        ctx->principals.clear();
        for (int i = 0; i < n_principals; i++)
            ctx->principals.emplace_back((const char*)principal_blob + principal_off[i], principal_off[i + 1] - principal_off[i]);
        ctx->channel = channel_id;
        ctx->identity_slot.assign(n_ids, -1);
    }
    // identities are long-lived: give every key a table now (what KeyImport does when the MSP deserialises an identity)
    // An MSP with more identities than big-table slots (client certificates) puts them in the small tier instead.
    if (n_ids > 0 && n_ids <= ctx->key_slots) {
        int rc = fabgpu_keys_register(ctx, keys_xy, n_ids, ctx->identity_slot.data());
        if (rc) return rc;
    } else if (n_ids > 0) {
        int rc = msp_small_tier(ctx, keys_xy, n_ids);             // also with the small tier off or too small: pre-registered window tables are still picked up
        if (rc) return rc;
    }
    return upload_msp(ctx, id_blob, id_off, keys_xy, valid, n_ids, policy_nodes, n_nodes);
}

// drains the block slots' streams: kernels already enqueued keep reading the tables they were launched with
static int drain_block_streams(fabgpu_ctx* ctx)
{
    CK(ctx, cudaSetDevice(ctx->devs[0].id));
    for (auto& ds : ctx->devs[0].slot) CK(ctx, cudaStreamSynchronize(ds.stream));
    return FABGPU_OK;
}

int fabgpu_msp_identity_groups(fabgpu_ctx* ctx, const int32_t* group, int n_ids)
{
    if (!ctx || n_ids < 0 || (n_ids && !group)) return FABGPU_E_ARG;
    std::lock_guard<std::mutex> lk0(ctx->slot0_mu);
    auto& dm = ctx->dm;
    if (n_ids != dm.n_ids) { ctx->last_error = "group table does not match the identities given to fabgpu_msp_configure"; return FABGPU_E_ARG; }
    int rc = drain_block_streams(ctx); if (rc) return rc;
    if (dm.group) { cudaFree(dm.group); dm.group = nullptr; }
    if (n_ids == 0) return FABGPU_OK;
    CK(ctx, cudaMalloc(&dm.group, 4 * (size_t)n_ids));
    CK(ctx, cudaMemcpy(dm.group, group, 4 * (size_t)n_ids, cudaMemcpyHostToDevice));
    return FABGPU_OK;
}

int fabgpu_namespace_policies(fabgpu_ctx* ctx, const uint8_t* ns_blob, const uint32_t* ns_off, const int32_t* ns_root, int n_ns)
{
    if (!ctx || n_ns < 0 || (n_ns && (!ns_blob || !ns_off || !ns_root))) return FABGPU_E_ARG;
    std::lock_guard<std::mutex> lk0(ctx->slot0_mu);
    auto& dm = ctx->dm;
    for (int i = 0; i < n_ns; i++)
        if (ns_root[i] < 0 || ns_root[i] >= dm.n_nodes || ns_off[i] > ns_off[i + 1]) { ctx->last_error = "namespace policy root out of range"; return FABGPU_E_ARG; }
    int rc = drain_block_streams(ctx); if (rc) return rc;
    void* old[] = {dm.ns_blob, dm.ns_off, dm.ns_root};
    for (void* p : old) if (p) cudaFree(p);
    dm.ns_blob = nullptr; dm.ns_off = nullptr; dm.ns_root = nullptr; dm.n_ns = 0;
    if (n_ns == 0) return FABGPU_OK;
    const size_t bl = ns_off[n_ns];
    CK(ctx, cudaMalloc(&dm.ns_blob, bl + 8));
    if (bl) CK(ctx, cudaMemcpy(dm.ns_blob, ns_blob, bl, cudaMemcpyHostToDevice));
    CK(ctx, cudaMalloc(&dm.ns_off, 4 * (size_t)(n_ns + 1)));
    CK(ctx, cudaMemcpy(dm.ns_off, ns_off, 4 * (size_t)(n_ns + 1), cudaMemcpyHostToDevice));
    CK(ctx, cudaMalloc(&dm.ns_root, 4 * (size_t)n_ns));
    CK(ctx, cudaMemcpy(dm.ns_root, ns_root, 4 * (size_t)n_ns, cudaMemcpyHostToDevice));
    dm.n_ns = n_ns;
    return FABGPU_OK;
}

int fabgpu_msp_hash_families(fabgpu_ctx* ctx, const uint8_t* mspid_blob, const uint32_t* mspid_off, const uint8_t* family, int n_msps)
{
    if (!ctx || n_msps < 0 || (n_msps && (!mspid_blob || !mspid_off || !family))) return FABGPU_E_ARG;
    std::lock_guard<std::mutex> lk0(ctx->slot0_mu);
    auto& dm = ctx->dm;
    std::unordered_map<std::string, uint8_t> fam;
    for (int i = 0; i < n_msps; i++) {
        const std::string id((const char*)mspid_blob + mspid_off[i], mspid_off[i + 1] - mspid_off[i]);
        if (family[i] != FABGPU_HASH_SHA2 && family[i] != FABGPU_HASH_SHA3) {
            ctx->last_error = "hash family of MSP '" + id + "' is neither FABGPU_HASH_SHA2 nor FABGPU_HASH_SHA3"; return FABGPU_E_ARG;
        }
        auto it = fam.find(id);
        if (it != fam.end() && it->second != family[i]) { ctx->last_error = "MSP '" + id + "' is listed with two hash families"; return FABGPU_E_ARG; }
        fam[id] = family[i];
    }
    for (const auto& kv : fam) {
        bool carried = false;
        for (const auto& m : ctx->msp.mspid) if (m == kv.first) { carried = true; break; }
        if (!carried) { ctx->last_error = "no identity of the MSP table belongs to MSP '" + kv.first + "'"; return FABGPU_E_ARG; }
    }
    const int n_ids = dm.n_ids;
    std::vector<uint8_t> kind(n_ids > 0 ? n_ids : 1, SHA_KIND_SHA2);
    bool any = false;
    for (int i = 0; i < n_ids; i++) {
        auto it = fam.find(ctx->msp.mspid[i]);
        if (it != fam.end() && it->second == FABGPU_HASH_SHA3) { kind[i] = SHA_KIND_SHA3; any = true; }
    }
    int rc = drain_block_streams(ctx); if (rc) return rc;
    if (n_ids) CK(ctx, cudaMemcpy(dm.hash_kind, kind.data(), (size_t)n_ids, cudaMemcpyHostToDevice));
    dm.any_sha3 = any;
    return FABGPU_OK;
}

int fabgpu_block_buffer_slot(fabgpu_ctx* ctx, int slot, size_t bytes, uint8_t** out)
{
    if (!ctx || !out || slot < 0 || slot >= FABGPU_SLOTS) return FABGPU_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->blk_mu[slot]);
    auto& bb = ctx->bbs[slot];
    CK(ctx, cudaSetDevice(ctx->devs[0].id));
    if (bytes > bb.h_block_cap) {
        if (ctx->dbs[slot].busy) { ctx->last_error = "slot holds a block in flight"; return FABGPU_E_ARG; }
        int rc = grow_host(ctx, bb.h_block, bytes); if (rc) return rc; bb.h_block_cap = bytes;
    }
    *out = bb.h_block;
    return FABGPU_OK;
}
int fabgpu_block_buffer(fabgpu_ctx* ctx, size_t bytes, uint8_t** out) { return fabgpu_block_buffer_slot(ctx, 0, bytes, out); }

// Device path of the block pre-pass: the host only copies bytes in and flags out (and marks duplicate tx ids).
//   H2D block + envelope offsets -> block_walk_kernel (per transaction) -> block_resolve_kernel (per signature: identity lookup, DER gates)
//   -> sha256_segments_kernel (signed messages + check digests; sha3_256_segments_kernel beside it for the signed messages of SHA3 MSPs)
//   -> one verify launch -> block_decide_kernel -> D2H flags.
// Everything is enqueued on the slot's stream in one go: the number of endorsement jobs (known only after the walk) stays
// on the device -- the later launches are sized for the worst case and read the count themselves.
static int block_submit(fabgpu_ctx* ctx, int slot, const uint8_t* block, size_t block_len, const uint32_t* env_off, size_t n_env)
{
    auto now = [] { return std::chrono::steady_clock::now(); };
    Device& dv = ctx->devs[0];
    DevSlot& ds = dv.slot[slot];
    auto& bb = ctx->bbs[slot]; auto& db = ctx->dbs[slot]; auto& dm = ctx->dm;
    db.t0 = now();
    CK(ctx, cudaSetDevice(dv.id));
    // Identities' key tables may have been recycled by other registrations since fabgpu_msp_configure: re-issue them.  From the
    // check to the last enqueue of this block the slot table is held shared (fabgpu_ctx::tab_mu): a concurrent
    // fabgpu_keys_register waits, so dm.key_slot's raw slots stay the tables of these identities for the whole launch sequence.
    std::shared_lock<std::shared_mutex> rl(ctx->tab_mu);
    {
        auto any_stale = [&] {
            std::lock_guard<std::mutex> lk(ctx->mu);
            for (size_t i = 0; i < ctx->identity_slot.size(); i++)
                if (ctx->identity_slot[i] != -1 && handle_to_slot(ctx, ctx->identity_slot[i]) == -1) return true;
            return false;
        };
        if (any_stale()) {
            rl.unlock();
            const int n_ids = (int)ctx->identity_slot.size();
            const bool big = n_ids <= ctx->key_slots;
            int rc = big ? fabgpu_keys_register(ctx, ctx->msp.keys_xy.data(), n_ids, ctx->identity_slot.data())     // exclusive; drains every stream first
                         : msp_small_tier(ctx, ctx->msp.keys_xy.data(), n_ids);
            if (rc) return rc;
            rl.lock();
            std::vector<int32_t> raw(n_ids, -1);
            dm.all_slots = true; dm.classes = 0;
            {
                std::lock_guard<std::mutex> lk(ctx->mu);      // a handle recycled again in the gap resolves to -1: that identity goes through the generic kernel
                for (int i = 0; i < n_ids; i++) {
                    raw[i] = handle_to_slot(ctx, ctx->identity_slot[i]);
                    if (raw[i] < 0) { dm.all_slots = false; dm.classes |= raw[i] == -1 ? CLASS_GENERIC : CLASS_SMALL; }
                }
            }
            // submitters are serialised by slot0_mu; blocks in flight on the other slots still read dm.key_slot: let them finish first
            for (auto& dsx : dv.slot) CK(ctx, cudaStreamSynchronize(dsx.stream));
            CK(ctx, cudaMemcpy(dm.key_slot, raw.data(), 4 * (size_t)n_ids, cudaMemcpyHostToDevice));
        }
    }
    if (block_len > bb.block_cap) {
        const size_t want = block_len + (block_len >> 2);
        bb.block_cap = 0;                                   // a failed grow leaves no buffer: do not remember the old capacity
        int rc = grow_dev(ctx, bb.d_block, want + 64);      // slack: word-wise readers (bytes_equal, the SHA loader) touch the aligned words past the end
        if (rc) return rc;
        bb.block_cap = want;
    }
    const char* evs = getenv("FABGPU_BLOCK_EVENTS");          // "1": time the device stages with CUDA events (diagnostics)
    db.use_ev = evs && evs[0] == '1';
    if (db.use_ev) for (auto& e : db.ev) if (!e) CK(ctx, cudaEventCreate(&e));
    if (db.use_ev) CK(ctx, cudaEventRecord(db.ev[0], ds.stream));
    std::vector<uint32_t> split;
    if (!env_off) {                                           // serialized common.Block: find the envelopes (serial, length-prefixed)
        std::vector<blockval::Seg> envs;
        if (!blockval::split_block(block, block_len, envs)) { ctx->last_error = "block does not parse"; return FABGPU_E_ARG; }
        n_env = envs.size();
        split.resize(2 * n_env + 2);
        for (size_t i = 0; i < n_env; i++) { split[2 * i] = envs[i].off; split[2 * i + 1] = envs[i].off + envs[i].len; }
    }
    const size_t T = n_env;
    db.T = T; db.block = block;
    if (T == 0) return FABGPU_OK;
    const size_t J_cap = T * (1 + BD_ENDS_HINT);
    if (T > db.tx_cap) {
        const size_t tc = T + (T >> 2) + 256, jc = tc * (1 + BD_ENDS_HINT);
        int rc = 0;
        db.tx_cap = 0; db.j_cap = 0;                        // reset first: after a partial failure the pointers are gone
        rc |= grow_dev(ctx, db.d_env_off, 8 * (tc + 1)); rc |= grow_dev(ctx, db.d_txs, sizeof(bdev::TxDev) * tc);
        rc |= grow_dev(ctx, db.d_raw, sizeof(bdev::RawJob) * jc);
        rc |= grow_dev(ctx, db.d_sha, sizeof(bdev::ShaJobD) * (jc + 2 * tc)); rc |= grow_dev(ctx, db.d_dig, 32 * (jc + 2 * tc) + 64);
        rc |= grow_dev(ctx, db.d_r, 32 * jc); rc |= grow_dev(ctx, db.d_s, 32 * jc); rc |= grow_dev(ctx, db.d_qx, 32 * jc); rc |= grow_dev(ctx, db.d_qy, 32 * jc);
        rc |= grow_dev(ctx, db.d_gate, jc); rc |= grow_dev(ctx, db.d_ks, 4 * jc); rc |= grow_dev(ctx, db.d_ident, 4 * jc); rc |= grow_dev(ctx, db.d_kind, jc);
        rc |= grow_dev(ctx, db.d_mask, jc / 8 + 8); rc |= grow_dev(ctx, db.d_off, jc / 8 + 8); rc |= grow_dev(ctx, db.d_counter, 16); rc |= grow_dev(ctx, db.d_idx, 4 * (jc + 2));
        rc |= grow_dev(ctx, db.d_flags, tc); rc |= grow_dev(ctx, db.d_hash, 8 * tc); rc |= grow_dev(ctx, db.d_seg, 8 * tc);
        rc |= grow_host(ctx, db.h_flags, tc); rc |= grow_host(ctx, db.h_hash, 8 * tc); rc |= grow_host(ctx, db.h_seg, 8 * tc);
        rc |= grow_host(ctx, db.h_counter, 16); rc |= grow_host(ctx, db.h_env_off, 8 * (tc + 1));
        if (rc) return FABGPU_E_CUDA;
        db.tx_cap = tc; db.j_cap = jc;
    }
    // envelope table on the device: pairs (begin, end) so that both entry points share one kernel
    for (size_t i = 0; i < T; i++) {
        db.h_env_off[2 * i] = env_off ? env_off[i] : split[2 * i];
        db.h_env_off[2 * i + 1] = env_off ? env_off[i + 1] : split[2 * i + 1];
    }
    cudaStream_t st = ds.stream;
    CK(ctx, cudaMemcpyAsync(db.d_env_off, db.h_env_off, 8 * T, cudaMemcpyHostToDevice, st));
    CK(ctx, cudaMemsetAsync(db.d_counter, 0, 16, st));
    bdev::MspDev m; m.id_blob = dm.id_blob; m.id_off = dm.id_off; m.key_slot = dm.key_slot; m.valid = dm.valid; m.msp_code = dm.msp_code; m.group = dm.group;
    m.keys_xy = dm.keys_xy; m.ht_hash = dm.ht_hash; m.ht_idx = dm.ht_idx; m.ht_size = dm.ht_size; m.n_ids = dm.n_ids; m.hash_kind = dm.hash_kind;
    bdev::PolicyDev pol; pol.nodes = dm.nodes; pol.n_nodes = dm.n_nodes; pol.principal_code = dm.principal_code; pol.n_principals = dm.n_principals;
    pol.ns_blob = dm.ns_blob; pol.ns_off = dm.ns_off; pol.ns_root = dm.ns_root; pol.n_ns = dm.n_ns;
    const bool need_q = (dm.classes & CLASS_GENERIC) != 0;   // only the generic arithmetic reads the key itself
    bdev::JobArrays ja; ja.sha = db.d_sha; ja.r = db.d_r; ja.s = db.d_s; ja.key_slot = db.d_ks; ja.identity = db.d_ident; ja.qx = need_q ? db.d_qx : nullptr;
    ja.qy = need_q ? db.d_qy : nullptr; ja.gate_ok = db.d_gate; ja.J_cap = (uint32_t)J_cap; ja.T = (uint32_t)T;
    // An MSP with SignatureHashFamily SHA3 in the table: resolve writes each signature job's hash kind, the SHA-256 launches skip the
    // SHA3 jobs and a SHA3-256 launch beside each hashes them into the same digest slots.  Otherwise the launches are those of a
    // SHA-256-only table (kind = null).
    const bool sha3 = dm.any_sha3;
    ja.kind = sha3 ? db.d_kind : nullptr;
    const uint32_t cnt = (uint32_t)T, E_cap = (uint32_t)(J_cap - T);
    // One copy, then the walk.  (Copying in chunks with a walk per chunk was measured slower on B200 -- 1 chunk 1.93 ms, 4 chunks
    // 2.27 ms, 8 chunks 3.52 ms per 10k-tx block: hashing a 4.6 KB payload is ~250 us of dependent rounds per thread however few
    // threads a launch has, so per-chunk launches serialise that latency.  What hides the copy is the NEXT block's copy running
    // under this block's kernels: the slots.)
    CK(ctx, cudaMemcpyAsync(bb.d_block, block, block_len, cudaMemcpyHostToDevice, st));
    bdev::block_walk_kernel<<<(cnt + 31) / 32, 32, 0, st>>>(bb.d_block, db.d_env_off, 0u, cnt, cnt, dm.channel, dm.channel_len, db.d_txs, db.d_raw, ja, db.d_counter);
    bdev::block_resolve_kernel<<<(cnt + 63) / 64, 64, 0, st>>>(bb.d_block, db.d_raw, 0u, cnt, m, ja, db.d_txs);                      // creator jobs
    sha256_segments_kernel<<<(cnt + 127) / 128, 128, 0, st>>>(bb.d_block, reinterpret_cast<const ShaJob*>(db.d_sha), cnt, db.d_dig, nullptr, ja.kind);
    if (sha3) sha3_256_segments_kernel<<<(cnt + 127) / 128, 128, 0, st>>>(bb.d_block, reinterpret_cast<const ShaJob*>(db.d_sha), cnt, db.d_dig, nullptr, ja.kind);
    // tx id and proposal hash: SHA-256 whatever the MSP family (protoutil/proputils.go:355-364, protoutil/txutils.go:431-448)
    sha256_segments_kernel<<<(2 * cnt + 127) / 128, 128, 0, st>>>(bb.d_block, reinterpret_cast<const ShaJob*>(db.d_sha + J_cap), 2 * cnt, db.d_dig + 32 * J_cap);
    ctx->launches += sha3 ? 5 : 4;
    CK(ctx, cudaGetLastError());
    if (db.use_ev) CK(ctx, cudaEventRecord(db.ev[1], st));
    if (db.use_ev) CK(ctx, cudaEventRecord(db.ev[2], st));
    // endorsement jobs [T, T + *d_counter): launches sized for the worst case, the kernels stop at the device-side count
    bdev::block_resolve_kernel<<<(E_cap + 63) / 64, 64, 0, st>>>(bb.d_block, db.d_raw, cnt, E_cap, m, ja, db.d_txs, db.d_counter);
    sha256_segments_kernel<<<(E_cap + 127) / 128, 128, 0, st>>>(bb.d_block, reinterpret_cast<const ShaJob*>(db.d_sha) + T, E_cap, db.d_dig + 32 * T, db.d_counter,
                                                               sha3 ? ja.kind + T : nullptr);
    if (sha3) sha3_256_segments_kernel<<<(E_cap + 127) / 128, 128, 0, st>>>(bb.d_block, reinterpret_cast<const ShaJob*>(db.d_sha) + T, E_cap, db.d_dig + 32 * T,
                                                                            db.d_counter, ja.kind + T);
    ctx->launches += sha3 ? 3 : 2;
    CK(ctx, cudaGetLastError());
    if (db.use_ev) CK(ctx, cudaEventRecord(db.ev[3], st));
    int rc = launch_verify(ctx, dv, dm.all_slots ? MODE_CACHED : MODE_MIXED, db.d_ks, db.d_qx, db.d_qy, db.d_dig, db.d_r, db.d_s, J_cap, db.d_mask, db.d_off, st,
                           db.d_counter, cnt, nullptr, db.d_idx, dm.classes ? dm.classes : CLASS_GENERIC);
    if (rc) return rc;
    if (db.use_ev) CK(ctx, cudaEventRecord(db.ev[4], st));
    bdev::block_decide_kernel<<<(cnt + 127) / 128, 128, 0, st>>>(bb.d_block, db.d_txs, cnt, m, pol, db.d_mask, db.d_gate, db.d_ident, db.d_dig, (uint32_t)J_cap, db.d_flags,
                                                               db.d_hash, db.d_seg);
    ctx->launches++;
    CK(ctx, cudaGetLastError());
    if (db.use_ev) CK(ctx, cudaEventRecord(db.ev[5], st));
    CK(ctx, cudaMemcpyAsync(db.h_flags, db.d_flags, T, cudaMemcpyDeviceToHost, st));
    CK(ctx, cudaMemcpyAsync(db.h_hash, db.d_hash, 8 * T, cudaMemcpyDeviceToHost, st));
    CK(ctx, cudaMemcpyAsync(db.h_seg, db.d_seg, 8 * T, cudaMemcpyDeviceToHost, st));
    db.t1 = now();
    return FABGPU_OK;
}

// Waits for the slot's block and finishes on the host: markTXIdDuplicates (v20/validator.go:283-297) -- among VALID
// transactions, a later one with an already seen tx id.  Reads the caller's block bytes to confirm equal hashes.
static int block_finish(fabgpu_ctx* ctx, int slot, uint8_t* flags)
{
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto us = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
        return std::chrono::duration<double, std::micro>(b - a).count();
    };
    auto& db = ctx->dbs[slot];
    const size_t T = db.T;
    const uint8_t* block = db.block;
    CK(ctx, cudaSetDevice(ctx->devs[0].id));
    CK(ctx, cudaStreamSynchronize(ctx->devs[0].slot[slot].stream));
    auto t3 = now();
    if (T == 0) return FABGPU_OK;
    memcpy(flags, db.h_flags, T);
    {
        // flat open-addressing table keyed by the 64-bit tx-id hash (0 = empty); equal hashes are confirmed on the bytes
        size_t cap = 16; while (cap < 4 * T) cap <<= 1;
        db.dup_keys.assign(cap, 0); db.dup_idx.resize(cap);
        uint64_t* keys = db.dup_keys.data(); uint32_t* idx = db.dup_idx.data();
        for (size_t t = 0; t < T; t++) {
            if (flags[t] != blockval::TX_VALID) continue;
            const bdev::Seg id = db.h_seg[t];
            const uint64_t h = db.h_hash[t] ? db.h_hash[t] : 1;
            bool dup = false;
            size_t pos = (size_t)h & (cap - 1);
            for (;; pos = (pos + 1) & (cap - 1)) {
                if (keys[pos] == 0) break;
                if (keys[pos] != h) continue;
                const bdev::Seg o = db.h_seg[idx[pos]];
                if (o.len == id.len && memcmp(block + o.off, block + id.off, id.len) == 0) { dup = true; break; }
            }
            if (dup) flags[t] = blockval::TX_DUPLICATE_TXID;
            else { keys[pos] = h; idx[pos] = (uint32_t)t; }
        }
    }
    auto t4 = now();
    ctx->block_timing[0] = us(db.t0, db.t1); ctx->block_timing[1] = 0; ctx->block_timing[2] = us(db.t1, t3); ctx->block_timing[3] = us(t3, t4);
    ctx->block_timing[4] = us(db.t0, t4);
    for (int k = 0; k < 5; k++) { float ms = 0; if (db.use_ev) cudaEventElapsedTime(&ms, db.ev[k], db.ev[k + 1]); ctx->block_timing[5 + k] = 1e3 * ms; }
    return FABGPU_OK;
}

// serialized: 1 = `block` is a serialized common.Block (env_off unused), 0 = concatenated envelopes with an offset table
static int validate_submit(fabgpu_ctx* ctx, int slot, const uint8_t* block, size_t block_len, const uint32_t* env_off, size_t n_env)
{
    if (!ctx || !block || slot < 0 || slot >= FABGPU_SLOTS) return FABGPU_E_ARG;
    if (block_len >= (1ull << 32)) { ctx->last_error = "block larger than 4 GiB"; return FABGPU_E_ARG; }
    if (env_off) {                                            // the table must be non-decreasing and stay inside the blob
        for (size_t i = 0; i < n_env; i++)
            if (env_off[i] > env_off[i + 1]) { ctx->last_error = "envelope offsets are not non-decreasing"; return FABGPU_E_ARG; }
        if (n_env && env_off[n_env] > block_len) { ctx->last_error = "envelope offsets exceed the blob length"; return FABGPU_E_ARG; }
    }
    std::lock_guard<std::mutex> lk(ctx->blk_mu[slot]);
    auto& db = ctx->dbs[slot];
    if (db.busy) { ctx->last_error = "slot already holds a block: call fabgpu_validate_wait first"; return FABGPU_E_ARG; }
    if (fault_injected()) { ctx->last_error = "fault injected (FABGPU_FAULT_INJECT=1)"; return FABGPU_E_INJECTED; }
    int rc;
    {
        std::lock_guard<std::mutex> lk0(ctx->slot0_mu);      // key-cache / MSP state: one submitter at a time
        rc = block_submit(ctx, slot, block, block_len, env_off, n_env);
        if (rc) { cudaStreamSynchronize(ctx->devs[0].slot[slot].stream); return rc; }
        db.on_device = true;
    }
    db.busy = true;
    return FABGPU_OK;
}

int fabgpu_validate_block_async(fabgpu_ctx* ctx, int slot, const uint8_t* block, size_t block_len)
{
    return validate_submit(ctx, slot, block, block_len, nullptr, 0);
}

int fabgpu_validate_envelopes_async(fabgpu_ctx* ctx, int slot, const uint8_t* blob, const uint32_t* env_off, size_t n_env)
{
    if (!env_off && n_env) return FABGPU_E_ARG;
    if (n_env == 0) {                                         // nothing to do, but keep the slot protocol
        if (!ctx || slot < 0 || slot >= FABGPU_SLOTS) return FABGPU_E_ARG;
        std::lock_guard<std::mutex> lk(ctx->blk_mu[slot]);
        auto& db = ctx->dbs[slot];
        if (db.busy) { ctx->last_error = "slot already holds a block: call fabgpu_validate_wait first"; return FABGPU_E_ARG; }
        db.T = 0; db.on_device = false; db.done_flags.clear(); db.busy = true;
        return FABGPU_OK;
    }
    return validate_submit(ctx, slot, blob, env_off[n_env], env_off, n_env);
}

int fabgpu_validate_wait(fabgpu_ctx* ctx, int slot, uint8_t* flags, size_t flags_cap, size_t* n_tx_out)
{
    if (!ctx || slot < 0 || slot >= FABGPU_SLOTS || !n_tx_out) return FABGPU_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->blk_mu[slot]);
    auto& db = ctx->dbs[slot];
    if (!db.busy) { ctx->last_error = "no block in flight on this slot"; return FABGPU_E_ARG; }
    db.busy = false;
    *n_tx_out = db.T;
    if (db.T > flags_cap || (db.T && !flags)) {
        if (db.on_device) cudaStreamSynchronize(ctx->devs[0].slot[slot].stream);
        ctx->last_error = "flags buffer too small";
        return FABGPU_E_ARG;
    }
    if (db.on_device) return block_finish(ctx, slot, flags);
    if (db.T) memcpy(flags, db.done_flags.data(), db.T);
    return FABGPU_OK;
}

int fabgpu_validate_block(fabgpu_ctx* ctx, const uint8_t* block, size_t block_len, uint8_t* flags, size_t flags_cap, size_t* n_tx_out)
{
    if (!ctx || !block || !flags || !n_tx_out) return FABGPU_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->sync_blk_mu);
    int rc = fabgpu_validate_block_async(ctx, 0, block, block_len);
    if (rc) return rc;
    return fabgpu_validate_wait(ctx, 0, flags, flags_cap, n_tx_out);
}

int fabgpu_validate_envelopes(fabgpu_ctx* ctx, const uint8_t* blob, const uint32_t* env_off, size_t n_env, uint8_t* flags, size_t flags_cap,
                              size_t* n_tx_out)
{
    if (!ctx || !blob || !env_off || !flags || !n_tx_out) return FABGPU_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->sync_blk_mu);
    int rc = fabgpu_validate_envelopes_async(ctx, 0, blob, env_off, n_env);
    if (rc) return rc;
    return fabgpu_validate_wait(ctx, 0, flags, flags_cap, n_tx_out);
}

int fabgpu_block_timing(const fabgpu_ctx* ctx, double out_us[10])
{
    if (!ctx || !out_us) return FABGPU_E_ARG;
    for (int i = 0; i < 10; i++) out_us[i] = ctx->block_timing[i];
    return FABGPU_OK;
}

// digests[j] = SHA-256(buf[off0..) || buf[off1..) || buf[off2..)) on the device; jobs: n x 6 uint32 (off0,off1,off2,len0,len1,len2)
int fabgpu_sha256_segments(fabgpu_ctx* ctx, const uint8_t* buf, size_t buf_len, const uint32_t* jobs, size_t n, uint8_t* digests)
{
    if (!ctx || !buf || !jobs || !digests) return FABGPU_E_ARG;
    std::lock_guard<std::mutex> lk0(ctx->slot0_mu);
    Device& dv = ctx->devs[0];
    CK(ctx, cudaSetDevice(dv.id));
    uint8_t *d_buf = nullptr, *d_dig = nullptr; ShaJob* d_jobs = nullptr;
    CK(ctx, cudaMalloc(&d_buf, buf_len ? buf_len : 1)); CK(ctx, cudaMalloc(&d_jobs, sizeof(ShaJob) * (n ? n : 1))); CK(ctx, cudaMalloc(&d_dig, 32 * (n ? n : 1)));
    CK(ctx, cudaMemcpy(d_buf, buf, buf_len, cudaMemcpyHostToDevice));
    CK(ctx, cudaMemcpy(d_jobs, jobs, sizeof(ShaJob) * n, cudaMemcpyHostToDevice));
    if (n) {
        sha256_segments_kernel<<<(unsigned)((n + 127) / 128), 128>>>(d_buf, d_jobs, (uint32_t)n, d_dig);
        ctx->launches++;
        CK(ctx, cudaGetLastError());
    }
    CK(ctx, cudaMemcpy(digests, d_dig, 32 * n, cudaMemcpyDeviceToHost));
    cudaFree(d_buf); cudaFree(d_jobs); cudaFree(d_dig);
    return FABGPU_OK;
}

// digests[j] = SHA3-256(buf[off0..) || buf[off1..) || buf[off2..)) on the device; same job layout as fabgpu_sha256_segments
int fabgpu_sha3_256_segments(fabgpu_ctx* ctx, const uint8_t* buf, size_t buf_len, const uint32_t* jobs, size_t n, uint8_t* digests)
{
    if (!ctx || !buf || !jobs || !digests) return FABGPU_E_ARG;
    std::lock_guard<std::mutex> lk0(ctx->slot0_mu);
    Device& dv = ctx->devs[0];
    CK(ctx, cudaSetDevice(dv.id));
    uint8_t *d_buf = nullptr, *d_dig = nullptr; ShaJob* d_jobs = nullptr;
    // slack: the block loader reads the aligned word past a range's end
    CK(ctx, cudaMalloc(&d_buf, buf_len + 8)); CK(ctx, cudaMalloc(&d_jobs, sizeof(ShaJob) * (n ? n : 1))); CK(ctx, cudaMalloc(&d_dig, 32 * (n ? n : 1)));
    CK(ctx, cudaMemcpy(d_buf, buf, buf_len, cudaMemcpyHostToDevice));
    CK(ctx, cudaMemcpy(d_jobs, jobs, sizeof(ShaJob) * n, cudaMemcpyHostToDevice));
    if (n) {
        sha3_256_segments_kernel<<<(unsigned)((n + 127) / 128), 128>>>(d_buf, d_jobs, (uint32_t)n, d_dig);
        ctx->launches++;
        CK(ctx, cudaGetLastError());
    }
    CK(ctx, cudaMemcpy(digests, d_dig, 32 * n, cudaMemcpyDeviceToHost));
    cudaFree(d_buf); cudaFree(d_jobs); cudaFree(d_dig);
    return FABGPU_OK;
}

int fabgpu_test_fieldop(fabgpu_ctx* ctx, int op, const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out)
{
    if (!ctx || !a || !b || !out) return FABGPU_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    Device& dv = ctx->devs[0];
    CK(ctx, cudaSetDevice(dv.id));
    uint8_t *da = nullptr, *db = nullptr, *dout = nullptr;
    CK(ctx, cudaMalloc(&da, 32 * n)); CK(ctx, cudaMalloc(&db, 32 * n)); CK(ctx, cudaMalloc(&dout, 32 * n));
    CK(ctx, cudaMemcpy(da, a, 32 * n, cudaMemcpyHostToDevice));
    CK(ctx, cudaMemcpy(db, b, 32 * n, cudaMemcpyHostToDevice));
    fieldop_kernel<<<(unsigned)((n + 63) / 64), 64>>>(op, da, db, (int)n, dout);
    ctx->launches++;
    CK(ctx, cudaGetLastError());
    CK(ctx, cudaMemcpy(out, dout, 32 * n, cudaMemcpyDeviceToHost));
    cudaFree(da); cudaFree(db); cudaFree(dout);
    return FABGPU_OK;
}

int fabgpu_test_table_entries(fabgpu_ctx* ctx, int key_slot, const uint32_t* window, const uint32_t* digit, size_t n, uint8_t* out)
{
    if (!ctx || !window || !digit || !out || key_slot >= ctx->key_slots) return FABGPU_E_ARG;
    const int wbits = key_slot < 0 ? FAB_WG : FAB_WQ, windows = key_slot < 0 ? FAB_G_WINDOWS : FAB_Q_WINDOWS;
    for (size_t i = 0; i < n; i++)
        if (window[i] >= (uint32_t)windows || digit[i] == 0 || digit[i] >= (1u << wbits)) return FABGPU_E_ARG;
    if (n == 0) return FABGPU_OK;
    Device& dv = ctx->devs[0];
    CK(ctx, cudaSetDevice(dv.id));
    const aff* tab = key_slot < 0 ? dv.gtab : dv.qtab + (size_t)key_slot * FAB_Q_WINDOWS * FAB_Q_ENTRIES;
    uint32_t *d_w = nullptr, *d_d = nullptr; aff* d_out = nullptr;
    CK(ctx, cudaMalloc(&d_w, 4 * n)); CK(ctx, cudaMalloc(&d_d, 4 * n)); CK(ctx, cudaMalloc(&d_out, sizeof(aff) * n));
    CK(ctx, cudaMemcpy(d_w, window, 4 * n, cudaMemcpyHostToDevice));
    CK(ctx, cudaMemcpy(d_d, digit, 4 * n, cudaMemcpyHostToDevice));
    table_entries_kernel<<<(unsigned)((n + 127) / 128), 128>>>(tab, wbits, d_w, d_d, (uint32_t)n, d_out);
    CK(ctx, cudaGetLastError());
    CK(ctx, cudaMemcpy(out, d_out, sizeof(aff) * n, cudaMemcpyDeviceToHost));
    cudaFree(d_w); cudaFree(d_d); cudaFree(d_out);
    return FABGPU_OK;
}

}  // extern "C"
