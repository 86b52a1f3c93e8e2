// TEST HELPER (not product code): the SHA3-256 code of fabric-mod_b200/csrc/sha3.cuh and the block logic of blockdev.cuh with
// per-MSP hash families, built for the host.  Extends blockdev_host.cpp (included whole: same handle, same exports) with
//   sha3_host_segments  -- sha3_256_message, the function sha3_256_segments_kernel runs per job;
//   bd_plan_families    -- bd_plan with the identities' hash kinds installed, recording the kind resolve_job assigns to each job;
//   bd_job_kind         -- that kind.
#include <map>
#include <vector>
#include "../../fabric-mod_b200/csrc/sha3.cuh"
#include "blockdev_host.cpp"

namespace {
std::map<const void*, std::vector<uint8_t>> g_job_kind;    // per handle: kind of every signature job of the last bd_plan_families
}

extern "C" {

// jobs: n x {off0, off1, off2, len0, len1, len2}; digests: n x 32 bytes.  `buf` must be readable 4 bytes past the last range.
void sha3_host_segments(const uint8_t* buf, const uint32_t* jobs, int n, uint8_t* digests)
{
    for (int j = 0; j < n; j++) {
        uint32_t w[8];
        fabgpu::sha3_256_message(buf, jobs + 6 * j, jobs + 6 * j + 3, w);
        for (int k = 0; k < 32; k++) digests[32 * j + k] = (uint8_t)(w[k / 4] >> (8 * (k % 4)));
    }
}

// hash_kind: per identity of bd_new's table, 0 = SHA-256, 1 = SHA3-256
int bd_plan_families(void* p, const uint8_t* blob, const uint32_t* env_off, int n_env, const uint8_t* hash_kind)
{
    const int n_end = bd_plan(p, blob, env_off, n_env);
    H* h = (H*)p;
    std::vector<uint8_t>& kind = g_job_kind[p];
    kind.assign(h->J_cap, 0xff);
    // resolve again with the kinds installed (resolve_job rewrites the same records and adds the job's kind)
    JobArrays ja; ja.sha = h->sha.data(); ja.r = h->r.data(); ja.s = h->s.data(); ja.key_slot = h->jks.data(); ja.identity = h->jid.data();
    ja.qx = nullptr; ja.qy = nullptr; ja.gate_ok = h->gate_ok.data(); ja.J_cap = h->J_cap; ja.T = h->T; ja.kind = kind.data();
    MspDev m = h->msp(); m.hash_kind = hash_kind;
    for (uint32_t j = 0; j < h->T + h->n_end; j++) resolve_job(h->block.data(), j, h->raw.data(), m, ja, h->txs.data());
    return n_end;
}

int bd_job_kind(void* p, int j) { return g_job_kind[p][j]; }

void bd_forget_kinds(void* p) { g_job_kind.erase(p); }

}  // extern "C"
