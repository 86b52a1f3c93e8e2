// Batched SHA3-256 (FIPS 202) on the device: the digest msp identity.Verify computes instead of SHA-256 when the signer's MSP
// is configured with SignatureHashFamily = SHA3 (msp/identities.go:169-196,216-224; mspimplsetup.go:80-99).  Same job format and
// launch contract as sha256_segments_kernel (sha256.cuh): a message is up to three byte ranges of one device buffer, one thread
// hashes one message, the digest is 32 bytes.  SHA3-256's digest is the first four state lanes as little-endian bytes, which is
// already the big-endian `e` layout the verify kernels read.
//
// Keccak-f[1600] on 25 64-bit lanes held in registers (every lane index is a compile-time constant), rate 136 bytes, domain
// padding 0x06 ... 0x80.  The permutation, the block loaders and the whole per-message hash are host+device functions, so the
// host build of this file (tests/host_sim/sha3_host.cpp) runs the code the kernel runs.
#pragma once
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#include <cuda_runtime.h>
#include "sha256.cuh"
#define SHA3_HD __host__ __device__ __forceinline__
#else
#define SHA3_HD inline
#endif

namespace fabgpu {

#define SHA3_RATE 136

#define SHA3_KECCAK_RC                                                                                                             \
    0x0000000000000001ull, 0x0000000000008082ull, 0x800000000000808Aull, 0x8000000080008000ull, 0x000000000000808Bull,               \
    0x0000000080000001ull, 0x8000000080008081ull, 0x8000000000008009ull, 0x000000000000008Aull, 0x0000000000000088ull,               \
    0x0000000080008009ull, 0x000000008000000Aull, 0x000000008000808Bull, 0x800000000000008Bull, 0x8000000000008089ull,               \
    0x8000000000008003ull, 0x8000000000008002ull, 0x8000000000000080ull, 0x000000000000800Aull, 0x800000008000000Aull,               \
    0x8000000080008081ull, 0x8000000000008080ull, 0x0000000080000001ull, 0x8000000080008008ull
#if defined(__CUDACC__)
__device__ __constant__ uint64_t kKeccakRCDev[24] = {SHA3_KECCAK_RC};
#endif
static const uint64_t kKeccakRCHost[24] = {SHA3_KECCAK_RC};

SHA3_HD uint64_t keccak_rc(int i)
{
#if defined(__CUDA_ARCH__)
    return kKeccakRCDev[i];
#else
    return kKeccakRCHost[i];
#endif
}

SHA3_HD uint64_t rotl64(uint64_t x, int n) { return (x << n) | (x >> (64 - n)); }

// (lo, hi) >> sh for sh in {0, 8, 16, 24}: the 32-bit word that starts sh/8 bytes into lo
SHA3_HD uint32_t sha3_funnel(uint32_t lo, uint32_t hi, uint32_t sh)
{
#if defined(__CUDA_ARCH__)
    return __funnelshift_r(lo, hi, sh);
#else
    return sh ? (lo >> sh) | (hi << (32 - sh)) : lo;
#endif
}

SHA3_HD uint32_t sha3_load32(const uint32_t* p)
{
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    uint32_t v; memcpy(&v, p, 4); return v;
#endif
}

// Keccak-f[1600]: 24 rounds of theta, rho + pi, chi, iota.  The round body is unrolled; the round loop is not (one round is
// ~200 instructions, the whole permutation unrolled would not stay in the instruction cache).
SHA3_HD void keccak_f1600(uint64_t* a)
{
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int round = 0; round < 24; round++) {
        uint64_t c[5];
#pragma unroll
        for (int x = 0; x < 5; x++) c[x] = a[x] ^ a[x + 5] ^ a[x + 10] ^ a[x + 15] ^ a[x + 20];
#pragma unroll
        for (int x = 0; x < 5; x++) {
            const uint64_t d = c[(x + 4) % 5] ^ rotl64(c[(x + 1) % 5], 1);
#pragma unroll
            for (int y = 0; y < 25; y += 5) a[y + x] ^= d;
        }
        // rho + pi: lane (x, y) moves to (y, 2x + 3y) rotated by its offset, followed along the single 24-lane cycle from lane 1
        uint64_t t = a[1];
#define SHA3_RP(j, r) { const uint64_t b_ = a[j]; a[j] = rotl64(t, r); t = b_; }
        SHA3_RP(10, 1) SHA3_RP(7, 3) SHA3_RP(11, 6) SHA3_RP(17, 10) SHA3_RP(18, 15) SHA3_RP(3, 21) SHA3_RP(5, 28) SHA3_RP(16, 36)
        SHA3_RP(8, 45) SHA3_RP(21, 55) SHA3_RP(24, 2) SHA3_RP(4, 14) SHA3_RP(15, 27) SHA3_RP(23, 41) SHA3_RP(19, 56) SHA3_RP(13, 8)
        SHA3_RP(12, 25) SHA3_RP(2, 43) SHA3_RP(20, 62) SHA3_RP(14, 18) SHA3_RP(22, 39) SHA3_RP(9, 61) SHA3_RP(6, 20) SHA3_RP(1, 44)
#undef SHA3_RP
#pragma unroll
        for (int y = 0; y < 25; y += 5) {
            const uint64_t b0 = a[y], b1 = a[y + 1], b2 = a[y + 2], b3 = a[y + 3], b4 = a[y + 4];
            a[y] = b0 ^ (~b1 & b2); a[y + 1] = b1 ^ (~b2 & b3); a[y + 2] = b2 ^ (~b3 & b4); a[y + 3] = b3 ^ (~b4 & b0); a[y + 4] = b4 ^ (~b0 & b1);
        }
        a[0] ^= keccak_rc(round);
    }
}

// Byte x of the padded message: the three ranges back to back, then 0x06, zeros, and 0x80 in the last byte of the last block
// (0x86 when both fall on one byte).  padded = (total / 136 + 1) * 136.
SHA3_HD uint32_t sha3_msg_byte(const uint8_t* buf, const uint32_t* off, const uint32_t* len, uint64_t total, uint64_t padded, uint64_t x)
{
    if (x < total) {
        uint64_t y = x;
        if (y < len[0]) return buf[off[0] + y];
        y -= len[0];
        if (y < len[1]) return buf[off[1] + y];
        y -= len[1];
        return buf[off[2] + y];
    }
    uint32_t v = x == total ? 0x06u : 0u;
    if (x == padded - 1) v |= 0x80u;
    return v;
}

// XOR the 136-byte block at `src` (inside one range, any byte offset) into the first 17 lanes: 35 aligned 32-bit loads issued
// together, re-aligned with funnel shifts.  Reads up to 3 bytes before `src` (same aligned word) and up to 4 bytes past the block.
SHA3_HD void sha3_absorb_aligned(uint64_t* a, const uint8_t* src)
{
    const uint32_t sh = 8u * (uint32_t)((uintptr_t)src & 3u);
    const uint32_t* p32 = reinterpret_cast<const uint32_t*>((uintptr_t)src & ~(uintptr_t)3);
    uint32_t w[SHA3_RATE / 4 + 1];
#pragma unroll
    for (int k = 0; k < SHA3_RATE / 4 + 1; k++) w[k] = sha3_load32(p32 + k);
#pragma unroll
    for (int k = 0; k < SHA3_RATE / 8; k++)
        a[k] ^= (uint64_t)sha3_funnel(w[2 * k], w[2 * k + 1], sh) | ((uint64_t)sha3_funnel(w[2 * k + 1], w[2 * k + 2], sh) << 32);
}

// XOR the block [o, o + 136) of the padded message into the state byte by byte: blocks that straddle two ranges or hold padding
// (one to three per message).
SHA3_HD void sha3_absorb_bytes(uint64_t* a, const uint8_t* buf, const uint32_t* off, const uint32_t* len, uint64_t total, uint64_t padded, uint64_t o)
{
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int k = 0; k < SHA3_RATE / 8; k++) {
        uint64_t v = 0;
        for (int b = 7; b >= 0; b--) v = (v << 8) | sha3_msg_byte(buf, off, len, total, padded, o + 8 * k + b);
        // a[k] with a run-time k: select without dynamic indexing
#pragma unroll
        for (int q = 0; q < SHA3_RATE / 8; q++) if (q == k) a[q] ^= v;
    }
}

// SHA3-256(buf[off0 .. off0+len0) || buf[off1 ..) || buf[off2 ..)) -> out[8]: the digest as little-endian 32-bit words (bytes
// 4i .. 4i+3 of the digest are word i).  `buf` must be readable 4 bytes past the last range.
SHA3_HD void sha3_256_message(const uint8_t* buf, const uint32_t* off, const uint32_t* len, uint32_t* out)
{
    uint64_t a[25];
#pragma unroll
    for (int i = 0; i < 25; i++) a[i] = 0;
    const uint64_t total = (uint64_t)len[0] + len[1] + len[2];
    const uint64_t padded = (total / SHA3_RATE + 1) * SHA3_RATE;
    const uint64_t e0 = len[0], e1 = e0 + len[1];
    for (uint64_t o = 0; o < padded; o += SHA3_RATE) {
        // which range holds [o, o+136) entirely, if any
        const uint8_t* src = nullptr;
        if (o + SHA3_RATE <= e0) src = buf + off[0] + o;
        else if (o >= e0 && o + SHA3_RATE <= e1) src = buf + off[1] + (o - e0);
        else if (o >= e1 && o + SHA3_RATE <= total) src = buf + off[2] + (o - e1);
        if (src) sha3_absorb_aligned(a, src);
        else sha3_absorb_bytes(a, buf, off, len, total, padded, o);
        keccak_f1600(a);
    }
#pragma unroll
    for (int k = 0; k < 4; k++) { out[2 * k] = (uint32_t)a[k]; out[2 * k + 1] = (uint32_t)(a[k] >> 32); }
}

#if defined(__CUDACC__)
// digests[j] = SHA3-256 of job j, one thread per message; the launch contract of sha256_segments_kernel (n_dev: message count
// produced by an earlier kernel of the stream, n the launch bound).  kind != null: only the jobs with kind[j] == SHA_KIND_SHA3
// are hashed (the block path hashes each signed message with its signer's MSP family; sha256_segments_kernel takes the rest).
__global__ void __launch_bounds__(128)
sha3_256_segments_kernel(const uint8_t* __restrict__ buf, const ShaJob* __restrict__ jobs, uint32_t n, uint8_t* __restrict__ digests,
                         const uint32_t* __restrict__ n_dev = nullptr, const uint8_t* __restrict__ kind = nullptr)
{
    if (n_dev) n = min(n, *n_dev);
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    if (kind && kind[j] != SHA_KIND_SHA3) return;
    const ShaJob job = jobs[j];
    uint32_t h[8];
    sha3_256_message(buf, job.off, job.len, h);
    uint32_t* out = reinterpret_cast<uint32_t*>(digests + 32 * (size_t)j);
#pragma unroll
    for (int k = 0; k < 8; k++) out[k] = h[k];
}
#endif

}  // namespace fabgpu
