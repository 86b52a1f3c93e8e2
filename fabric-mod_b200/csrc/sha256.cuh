// Batched SHA-256 on the device (SURVEY.md section 8f rank 2): the digest msp identity.Verify computes before every
// bccsp.Verify (msp/identities.go:178 -> bccsp/sw/hash.go:29-33), plus the two digests the transaction checks need
// (tx id: protoutil/proputils.go:357-364; proposal hash: protoutil/txutils.go:431-448).
//
// A message is the concatenation of up to three byte ranges of one device buffer (the block), e.g. the signed bytes of
// an endorsement are  ProposalResponsePayload || endorser  (core/common/validation/statebased/validator_keylevel.go:
// 246-249) -- two ranges of the block, never copied together on the host.  One thread hashes one message; the digest is
// written as 32 big-endian bytes, which is exactly the `e` operand layout of the verify kernels (hashToInt of a 32-byte
// digest is the identity).  HBM-streaming work: ~2 KiB read per message, 32 B written.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace fabgpu {

struct ShaJob { uint32_t off[3]; uint32_t len[3]; };

// Hash of a signed message on the block path (bdev::JobArrays::kind): the SignatureHashFamily of the signer's MSP.
enum : uint8_t { SHA_KIND_SHA2 = 0, SHA_KIND_SHA3 = 1 };

__device__ __constant__ uint32_t kSha256K[64] = {
    0x428a2f98, 0x71374491, 0xb5c0fbcf, 0xe9b5dba5, 0x3956c25b, 0x59f111f1, 0x923f82a4, 0xab1c5ed5, 0xd807aa98, 0x12835b01, 0x243185be,
    0x550c7dc3, 0x72be5d74, 0x80deb1fe, 0x9bdc06a7, 0xc19bf174, 0xe49b69c1, 0xefbe4786, 0x0fc19dc6, 0x240ca1cc, 0x2de92c6f, 0x4a7484aa,
    0x5cb0a9dc, 0x76f988da, 0x983e5152, 0xa831c66d, 0xb00327c8, 0xbf597fc7, 0xc6e00bf3, 0xd5a79147, 0x06ca6351, 0x14292967, 0x27b70a85,
    0x2e1b2138, 0x4d2c6dfc, 0x53380d13, 0x650a7354, 0x766a0abb, 0x81c2c92e, 0x92722c85, 0xa2bfe8a1, 0xa81a664b, 0xc24b8b70, 0xc76c51a3,
    0xd192e819, 0xd6990624, 0xf40e3585, 0x106aa070, 0x19a4c116, 0x1e376c08, 0x2748774c, 0x34b0bcb5, 0x391c0cb3, 0x4ed8aa4a, 0x5b9cca4f,
    0x682e6ff3, 0x748f82ee, 0x78a5636f, 0x84c87814, 0x8cc70208, 0x90befffa, 0xa4506ceb, 0xbef9a3f7, 0xc67178f2};

__device__ __forceinline__ uint32_t rotr32(uint32_t x, int n) { return __funnelshift_r(x, x, n); }

__device__ __forceinline__ void sha256_compress(uint32_t* h, uint32_t* w)
{
    uint32_t a = h[0], b = h[1], c = h[2], d = h[3], e = h[4], f = h[5], g = h[6], hh = h[7];
#pragma unroll
    for (int i = 0; i < 64; i++) {
        if (i >= 16) {
            const uint32_t w15 = w[(i + 1) & 15], w2 = w[(i + 14) & 15];
            const uint32_t s0 = rotr32(w15, 7) ^ rotr32(w15, 18) ^ (w15 >> 3);
            const uint32_t s1 = rotr32(w2, 17) ^ rotr32(w2, 19) ^ (w2 >> 10);
            w[i & 15] = w[i & 15] + s0 + w[(i + 9) & 15] + s1;
        }
        const uint32_t S1 = rotr32(e, 6) ^ rotr32(e, 11) ^ rotr32(e, 25);
        const uint32_t ch = (e & f) ^ (~e & g);
        const uint32_t t1 = hh + S1 + ch + kSha256K[i] + w[i & 15];
        const uint32_t S0 = rotr32(a, 2) ^ rotr32(a, 13) ^ rotr32(a, 22);
        const uint32_t mj = (a & b) ^ (a & c) ^ (b & c);
        const uint32_t t2 = S0 + mj;
        hh = g; g = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
    }
    h[0] += a; h[1] += b; h[2] += c; h[3] += d; h[4] += e; h[5] += f; h[6] += g; h[7] += hh;
}

// Byte x of the padded message: the three ranges back to back, then 0x80, zeros and the 64-bit big-endian bit length.
__device__ __forceinline__ uint32_t sha_msg_byte(const uint8_t* __restrict__ buf, const ShaJob& job, uint64_t total, uint64_t padded, uint64_t x)
{
    if (x < total) {
        uint64_t y = x;
        if (y < job.len[0]) return buf[job.off[0] + y];
        y -= job.len[0];
        if (y < job.len[1]) return buf[job.off[1] + y];
        y -= job.len[1];
        return buf[job.off[2] + y];
    }
    if (x == total) return 0x80u;
    if (x >= padded - 8) return (uint32_t)(((total * 8) >> (8 * (padded - 1 - x))) & 0xff);
    return 0u;
}

// digests[j] = SHA-256(buf[off0 .. off0+len0) || buf[off1 ..) || buf[off2 ..)).  One thread per message, the sixteen message
// words of a block stay in registers: a 64-byte block that lies inside one range is fetched as 17 aligned 32-bit loads
// (issued together) and re-aligned with funnel shifts, whatever the byte offset of the range; blocks that straddle two
// ranges or contain padding are assembled byte by byte (at most three or four per message).
// `buf` must be readable 4 bytes past the last range (the block buffer is allocated with slack).
// kind != null: the jobs with kind[j] == SHA_KIND_SHA3 are skipped (sha3_256_segments_kernel hashes those).
__global__ void __launch_bounds__(128)
sha256_segments_kernel(const uint8_t* __restrict__ buf, const ShaJob* __restrict__ jobs, uint32_t n, uint8_t* __restrict__ digests,
                       const uint32_t* __restrict__ n_dev = nullptr, const uint8_t* __restrict__ kind = nullptr)
{
    if (n_dev) n = min(n, *n_dev);               // message count produced by an earlier kernel of the stream; n is the launch bound
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    if (kind && kind[j] == SHA_KIND_SHA3) return;
    const ShaJob job = jobs[j];
    uint32_t h[8] = {0x6a09e667, 0xbb67ae85, 0x3c6ef372, 0xa54ff53a, 0x510e527f, 0x9b05688c, 0x1f83d9ab, 0x5be0cd19};
    const uint64_t total = (uint64_t)job.len[0] + job.len[1] + job.len[2];
    const uint64_t padded = (total + 9 + 63) / 64 * 64;
    const uint64_t e0 = job.len[0], e1 = e0 + job.len[1];
    for (uint64_t o = 0; o < padded; o += 64) {
        uint32_t w[16];
        // which range holds [o, o+64) entirely, if any
        const uint8_t* src = nullptr;
        if (o + 64 <= e0) src = buf + job.off[0] + o;
        else if (o >= e0 && o + 64 <= e1) src = buf + job.off[1] + (o - e0);
        else if (o >= e1 && o + 64 <= total) src = buf + job.off[2] + (o - e1);
        if (src) {
            const uint32_t sh = 8u * (uint32_t)((uintptr_t)src & 3u);
            const uint32_t* p32 = reinterpret_cast<const uint32_t*>((uintptr_t)src & ~(uintptr_t)3);
            uint32_t x[17];
#pragma unroll
            for (int k = 0; k < 17; k++) x[k] = __ldg(p32 + k);
#pragma unroll
            for (int k = 0; k < 16; k++) w[k] = __byte_perm(__funnelshift_r(x[k], x[k + 1], sh), 0, 0x0123);
        } else {
#pragma unroll 1
            for (int k = 0; k < 16; k++) {
                uint32_t v = 0;
                for (int b = 0; b < 4; b++) v = (v << 8) | sha_msg_byte(buf, job, total, padded, o + 4 * k + b);
                // w[k] with a run-time k: select without dynamic indexing
#pragma unroll
                for (int q = 0; q < 16; q++) if (q == k) w[q] = v;
            }
        }
        sha256_compress(h, w);
    }
    uint32_t* out = reinterpret_cast<uint32_t*>(digests + 32 * (size_t)j);
#pragma unroll
    for (int k = 0; k < 8; k++) out[k] = __byte_perm(h[k], 0, 0x0123);      // big-endian bytes
}

}  // namespace fabgpu
