// logmel_kernel.cuh -- the fused log-mel kernel for sm_100a (B200).
//
// One persistent CTA per SM, 16 warps = TWO INDEPENDENT GROUPS of 8 warps.  A group is a
// "virtual CTA": it owns whole clips, one at a time (the first 2 * gridDim clips are dealt statically,
// every further one is fetched with atomicAdd on a per-launch work counter, so ragged batches stay
// balanced), walks the clip's (clip, tile) items on its own, and synchronises only with itself
// (named barrier 1 + group, mbarrier [group]).  The groups share the constant tables in shared
// memory and nothing else; two of them keep the scheduler's dispatch port busier than one 16-warp
// CTA whose warps all sit in the same phase (DESIGN.md section 5: the relative phase of the groups
// does not matter, `stagger_ns` is kept as an experiment knob only).
//
// A tile is 8 frames (16 / 32 / 64 for n_fft = 1024 / 512 / 256).  Two frame layouts (Geo): one real frame per warp at
// n_fft = 2048; below that, 1024 / n_fft complex FFTs side by side in the warp, each carrying two real frames packed
// as a + i b.  Per item, inside a group:
//
//   stage   (one item ahead, into the group's single buffer as soon as every warp has pulled its
//           frame into registers) the tile's samples -> shared memory, once per sample although
//           every sample feeds 4 frames.  The contiguous interior of a plain clip is one
//           cp.async.bulk (TMA, 1-D) completing on an mbarrier; whatever is left -- torch.stft's
//           reflect padding, zero padding, and whole tiles of augmented clips -- goes through the
//           gather path, one loop (stage_slots) that does pad/crop (R/src/data/preprocessing.py:70-83),
//           noise and roll (:85-93) as index arithmetic for every sample source: an fp32 or 16-bit
//           sample of the clip, or one computed by the resampler (lm_forward_resampled; lm_forward_spans when only the
//           native samples a clip's features read are stored: rs_read_span is that set, the same code on host and device).
//   FFT     x Hann fused with the first butterfly stage (hann[n + n_fft/2] = 1 - hann[n]: one
//           window load per two samples), 2048 real -> 1024 complex points held as 32
//           registers/lane; register radix-32 FFT over the lane-local index, twiddle, 32x32
//           transpose through the warp's shared-memory row, second radix-32 FFT, then the real-FFT
//           untangle with the partner bin fetched by warp shuffle; 4|X|^2 overwrites the warp's
//           row (never HBM).  (TA/functional/functional.py:123-145: torch.stft + abs().pow(2))
//   mel     on the tensor cores, filterbank-stationary: mma.sync m16n8k8 TF32 with
//           A = [8 mels x {hi, lo}] x 8 bins (the 16 MMA rows hold the TF32 head and the residual
//           of the same 8 filters), B = 8 bins x 8 frames of the power rows, once with the head
//           and once with the residual of the power: 2 MMAs per 8 bins give all four partial
//           products, error ~2^-21.  Only the band of bins the 8 filters touch is walked
//           (TA/transforms/_transforms.py:417).  Epilogue in registers: 10*log10(max(x, amin))
//           (TA/functional/functional.py:390-391), SpecAugment intervals (:939-953), store,
//           fp64 sum / sum-of-squares.
//   silent  tiles that lie entirely in a plain clip's zero padding skip all of the above and write the floor /
//           mask values and their statistics directly (bit-identical to the full path on a zero spectrum).
//   split   small batches (B < number of groups on the GPU): a clip's tiles are dealt to `split` groups as
//           "virtual clips" (clip, tile range); the per-clip statistics are 64-bit fixed-point sums (exact,
//           order-independent integer adds), combined with atomics, and the group that arrives last
//           normalises the whole clip.  Bit-identical to the unsplit path.
//   norm    when the clip is finished the same group re-reads its (L2-resident) dB block and
//           writes (x - mean) / (std + eps)  (R/src/data/preprocessing.py:111-116); for lm_forward_gather
//           the same pass also stores the result into the other ranks' gathered buffers (multimem.st
//           through the NVSwitch, or plain stores to peer-mapped memory).
//
//   pcm16   (Pcm16 instantiation, lm_forward_pcm16) the clips are 16-bit PCM, the sample format of the ICBHI wav
//           files (R/src/data/preprocessing.py:55-68 decodes them with torchaudio.load): the bulk copy brings the
//           tile's raw samples (2 bytes each) to the END of the staging buffer and the group expands them in place to
//           fp32 (x / 32768, as lm_pcm16_decode) before the FFT reads them; the gather path converts sample by sample.
//           HBM sees 2 bytes per sample and there is no decode kernel in front.
//
// Algorithmic HBM bytes per clip: 4*min(len, T) read (2*min(len, T) for pcm16) + 4*n_mels*frames written.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/logmel_b200.h"
#include "fft_gen.cuh"
#include "resample.cuh"

// Build-time experiment switches (tools/build_variants.py); the shipped kernel is LM_EXP=0, LM_TIMING=0.
//   LM_EXP     1: no mel phase (FFT only)   2: no FFT (mel phase on stale rows)   3: no FFT part 2
//   LM_TIMING  1: every warp accumulates clock64() deltas per phase into lm::g_timing[block][warp][8]
//              (read back with lm_debug_timing)
#ifndef LM_EXP
#define LM_EXP 0
#endif
#ifndef LM_TIMING
#define LM_TIMING 0
#endif
#if LM_TIMING
#define LM_T(slot) do { const long long t_now_ = clock64(); t_acc[slot] += t_now_ - t_last; t_last = t_now_; } while (0)
#else
#define LM_T(slot) do { } while (0)
#endif

namespace lm {

#if LM_TIMING
__device__ long long g_timing[160 * 16 * 8];
#endif

constexpr int kGroups = 2;
constexpr int kGroupWarps = 8;
constexpr int kGroupThreads = kGroupWarps * 32;
constexpr int kWarps = kGroups * kGroupWarps;
constexpr int kThreads = kWarps * 32;
constexpr int kScrPitch = 36;                 // transpose rows: 32 + 4 (16 B aligned, LDS.128 conflict-free)
constexpr int kRowFloats = 1168;              // per-warp row: >= 32*36 and == 16 (mod 32) for the MMA loads
constexpr int kMaxMelTiles = 32;              // n_mels <= 256
constexpr int kMaxPeers = 7;                  // other GPUs of one NVSwitch domain
constexpr int kTileSlots = kMaxMelTiles / kGroupWarps;   // mel tiles per warp, at most
constexpr int kMaxDk = 96;                    // 16-bin steps of banded filterbank kept on chip (1 KB each)

// What one logmel_kernel instantiation is built for: fp32 clips (Plain), + dB and mel power outputs (ExtraOut), 16-bit
// PCM clips (Pcm16), on-device Philox noise (DeviceNoise), resampling in the staging (Resampled).  One per launch.
enum class Variant { Plain, ExtraOut, Pcm16, DeviceNoise, Resampled };
constexpr int kVariants = static_cast<int>(Variant::Resampled) + 1;

struct MelTable {                             // lives in global memory, copied to shared
    int kb[kMaxMelTiles];                     // first bin of the tile's band (multiple of 4)
    int ndk[kMaxMelTiles];                    // 16-bin steps in the band
    int off[kMaxMelTiles];                    // first step's index into melw (units of 64 float4)
    int warp_tile[kGroupWarps][kTileSlots];   // mel tiles owned by each warp of a group (-1 = none)
};

struct KParams {
    // batch
    const void* __restrict__ wave;        // fp32 samples, int16 for PCM16 and for RESAMPLE with pcm16 (offsets count samples)
    const long long* __restrict__ offset;
    const int* __restrict__ length;
    const lm_aug* __restrict__ aug;
    const float* __restrict__ noise;
    float* __restrict__ out_norm;
    float* __restrict__ out_db;
    float* __restrict__ out_melpow;
    int B;
    int normalize;
    // fused feature all-gather (lm_forward_gather): besides out_norm, the normalised features of clip i go to
    // peer[r] + i * n_mels * frames for r < n_peer (the same slice of the other ranks' gathered buffers,
    // mapped over NVLink), or through one multicast store per value when mc_out is set (NVSwitch replicates
    // it into every rank's buffer, this rank's included)
    float* peer[kMaxPeers];
    int n_peer;
    float* mc_out;
    // dynamic clip scheduling: clips [0, 2*gridDim) are dealt statically (one per group); every further clip
    // is fetched with atomicAdd on work_counter[0] when a group starts the last tile of its current clip, so that
    // ragged batches (unequal numbers of silent tiles) stay balanced.  work_counter[1] counts the groups that have
    // finished; the last one puts both back to zero, so a launch needs no memset (the counters start at zero when
    // the plan is created and every launch leaves them at zero).
    int* work_counter;
    // small-batch mode: every clip is cut into `split` chunks of `tiles_per_chunk` tiles (the last one may be
    // shorter, none is empty); virtual clip v = clip * split + chunk.  clip_stats[2 clip .. 2 clip + 1] and
    // clip_cnt[clip] are zero before the launch and put back to zero by the group that completes the clip
    // (used only when split > 1).
    int split, tiles_per_chunk;
    unsigned long long* clip_stats;
    int* clip_cnt;
    // plan
    int T, hop, frames, n_mels, n_tiles;
    int ns;          // staged floats per tile = (TILE_F-1)*hop + NFFT, rounded up to 4
    int n_dk;        // total 16-bin steps in melw
    int use_tma;
    int stagger_ns;  // head start of group 0 over group 1
    float db_scale;  // db_multiplier * log10(2): dB = db_scale * log2(x) - db_offset
    float amin, db_offset, floor_db, norm_eps;
    const float* __restrict__ window;   // [NFFT] (the first half is used)
    const float2* __restrict__ tw;      // [kTwRows*32]  W1024^(n2*k1) = (cos, -sin), rows k1 = 1,2,3,4,8,...,28
    const float2* __restrict__ utw;     // [512]    (cos, sin)(2 pi k / 2048)
    const float4* __restrict__ melw;    // [n_dk][2 k-steps][32 lanes]: mma A fragments (head, residual, head, residual)
    const MelTable* __restrict__ mel_table;
    // lm_forward_resampled (Resampled instantiation): clip i is at the rate of rate pair source[i] (-1: the plan's rate)
    // and is resampled inside the staging; `wave` holds int16 samples when pcm16 is set.  rs[s]: rate pair s, the
    // tables lm_resample reads (resample.cuh).
    const int* __restrict__ source;
    int pcm16;
    int n_rs;
    RsTaps rs[LM_MAX_RESAMPLERS];
    // lm_forward_spans (Resampled instantiation): clip i stores only its native samples [first[i], first[i] + stored[i]),
    // starting at wave + offset[i]; length[i] is still the whole clip's.  Null for lm_forward_resampled.
    const long long* __restrict__ first;
    const int* __restrict__ stored;
};

// ---------------------------------------------------------------------------------------
// PTX helpers: mbarrier + 1-D bulk copy (TMA) global -> shared, named barrier, TF32 mma
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "LAB_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONE;\n\t"
        "bra LAB_WAIT;\n\t"
        "DONE:\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// barrier of one 8-warp group (ids 1 and 2; id 0 is __syncthreads)
__device__ __forceinline__ void group_bar(int group) {
    asm volatile("bar.sync %0, %1;" ::"r"(group + 1), "n"(kGroupThreads) : "memory");
}
// D += A(16x8, row) * B(8x8, col), TF32 inputs (low 13 mantissa bits ignored), fp32 accumulate
__device__ __forceinline__ void mma_tf32(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3,
                                         uint32_t b0, uint32_t b1) {
    asm(
        "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
// Opaque copy: stops the compiler from hoisting address arithmetic that depends on `v` out of the
// item loop and keeping it alive across the register-heavy FFT (it is recomputed per phase instead).
__device__ __forceinline__ int launder(int v) {
    asm volatile("" : "+r"(v));
    return v;
}
// one 16-byte store replicated by the NVSwitch into every GPU of the multicast group
__device__ __forceinline__ void multimem_st_v4(float* mc_addr, float4 v) {
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc_addr), "f"(v.x), "f"(v.y),
                 "f"(v.z), "f"(v.w)
                 : "memory");
}
// log2 of a normal positive number: plain MUFU.LG2, no denormal pre-scaling (callers pass x > amin)
__device__ __forceinline__ float lg2_ftz(float x) {
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ uint32_t tf32_hi(float x) { return __float_as_uint(x) & 0xffffe000u; }
__device__ __forceinline__ uint32_t tf32_lo(float x, uint32_t hi) { return __float_as_uint(x - __uint_as_float(hi)); }

// Per-clip statistics are exact integers: a thread's fp32 partial sums of one item are rounded once to
// 2^-24 (sum) / 2^-16 (sum of squares) and added as 64-bit integers, so the totals do not depend on which
// group processed which tile, nor on the order of the additions (small-batch mode relies on this).
constexpr float kStatScaleS = 16777216.0f, kStatScaleQ = 65536.0f;
__device__ __forceinline__ void stat_add(longlong2* __restrict__ slot, float ssum, float qsum) {
    longlong2 st = *slot;
    // through fp64: a three-instruction conversion (the fp32 -> int64 intrinsic expands to a dozen), exact scaling
    st.x += __double2ll_rn(static_cast<double>(ssum) * static_cast<double>(kStatScaleS));
    st.y += __double2ll_rn(static_cast<double>(qsum) * static_cast<double>(kStatScaleQ));
    *slot = st;
}

// ---------------------------------------------------------------------------------------
// Philox4x32-10 -> N(0,1): throughput-mode noise when no host-drawn noise is supplied
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float philox_normal(uint64_t seed, uint32_t idx) {
    uint32_t c0 = idx >> 2, c1 = 0u, c2 = 0x6c6f676du, c3 = 0x656c0000u;
    uint32_t k0 = static_cast<uint32_t>(seed), k1 = static_cast<uint32_t>(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        const uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        c0 = h1 ^ c1 ^ k0; c1 = l1; c2 = h0 ^ c3 ^ k1; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    const uint32_t a = (idx & 2u) ? c2 : c0, b = (idx & 2u) ? c3 : c1;
    const float u1 = (static_cast<float>(a >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float u2 = (static_cast<float>(b >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float r = sqrtf(-2.0f * __logf(u1));
    float s, c;
    __sincosf(6.283185307179586f * u2, &s, &c);
    return (idx & 1u) ? r * s : r * c;
}

// ---------------------------------------------------------------------------------------
// 1024-point complex FFT of one warp, in two halves so that the group barrier can sit between them.
// Lane n2 holds z[32*n1 + n2] in z[n1] (re, im packed in one 64-bit register); on exit lane
// k1 holds Z[k1 + 32*k2] in (xr[k2], xi[k2]).
//   part 1 (registers only): packed complex radix-32 FFT over the lane-local index.  Its first
//           butterfly stage (z[r] +- z[r+16]) is done by the caller, fused with the window.
//   part 2: twiddle, 32x32 transpose through the warp's private row `scr` (real and imaginary planes
//           separately; the LDS.128 reads hand the second FFT register pairs of neighbouring
//           points, the layout its packed stages 1-4 want -- see gen_fft.py) + second radix-32 FFT.
// ---------------------------------------------------------------------------------------
constexpr int kTwRows = 10;   // twiddle table rows kept on chip: k1 = 1, 2, 3, 4, 8, 12, ..., 28
__device__ __forceinline__ void warp_twiddle(lm_f2 (&z)[32], const float2* __restrict__ tw, int lane) {
    // Twiddle W1024^(lane*k1), k1 = 4a + b, as the product of two table entries W^(4a*lane) * W^(b*lane):
    // 10 shared-memory loads instead of 31 (the shared-memory pipe is the tighter resource here, and
    // 31 loads in flight on top of z do not fit the register file), one extra rounding per twiddle.
    // tw holds (cos, -sin); (r + i m)(wx + i wy) = (r wx - m wy, m wx + r wy).
    auto cmul = [](lm_f2 v, lm_f2 w) {
        return lm_fma2(lm_swap(v), lm_pack(-lm_hi(w), lm_hi(w)), lm_mul2(v, lm_bcast(lm_lo(w))));
    };
    auto ldtw = [&](int row) {
        const float2 w = tw[row * 32 + lane];
        return lm_pack(w.x, w.y);
    };
    const lm_f2 B1 = ldtw(0), B2 = ldtw(1), B3 = ldtw(2);
    z[1] = cmul(z[1], B1);
    z[2] = cmul(z[2], B2);
    z[3] = cmul(z[3], B3);
#pragma unroll
    for (int a = 1; a < 8; ++a) {
        const lm_f2 A = ldtw(2 + a);
        z[4 * a] = cmul(z[4 * a], A);
        z[4 * a + 1] = cmul(z[4 * a + 1], cmul(A, B1));
        z[4 * a + 2] = cmul(z[4 * a + 2], cmul(A, B2));
        z[4 * a + 3] = cmul(z[4 * a + 3], cmul(A, B3));
    }
}
// n_fft = 512 / 256 (R = 16 / 8): lane s R + n2 holds z_s[R n1 + n2] of sub-FFT s in z[n1].  Part 1 is the same
// radix-32 FFT over n1; the twiddle is W_n_fft^(n2 k1) (the table is built per n_fft, the code is the same); after
// the transpose lane k1 holds the R values n2 of each sub-FFT side by side, and the second stage is 32 / R
// radix-R FFTs: lane k1 ends with Z_s[k1 + 32 k2] in (xr[s R + k2], xi[s R + k2]).
template <int NFFT>
__device__ __forceinline__ void warp_cfft_part2(lm_f2 (&z)[32], float (&xr)[32], float (&xi)[32],
                                                float* __restrict__ scr, const float2* __restrict__ tw, int lane) {
    warp_twiddle(z, tw, lane);
    lm_f2 pr[16], pi[16];
#pragma unroll
    for (int k1 = 0; k1 < 32; ++k1) scr[k1 * kScrPitch + lane] = lm_lo(z[k1]);
    __syncwarp();
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const float4 v = *reinterpret_cast<const float4*>(scr + lane * kScrPitch + 4 * q);
        pr[2 * q] = lm_pack(v.x, v.y);
        pr[2 * q + 1] = lm_pack(v.z, v.w);
    }
    __syncwarp();
#pragma unroll
    for (int k1 = 0; k1 < 32; ++k1) scr[k1 * kScrPitch + lane] = lm_hi(z[k1]);
    __syncwarp();
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const float4 v = *reinterpret_cast<const float4*>(scr + lane * kScrPitch + 4 * q);
        pi[2 * q] = lm_pack(v.x, v.y);
        pi[2 * q + 1] = lm_pack(v.z, v.w);
    }
    __syncwarp();
    if (NFFT == 512) lm_fft16x2_soa(pr, pi, xr, xi);
    else if (NFFT == 256) lm_fft8x4_soa(pr, pi, xr, xi);
    else lm_fft32_soa(pr, pi, xr, xi);
}

// The four normals of one Philox block: z[j] == philox_normal(seed, 4 * blk + j), bit for bit (same operations),
// for the staging of noisy clips, which walks four consecutive samples per thread: one block serves up to four
// samples and one log / sincos serves two of them.
__device__ __forceinline__ void philox_normal4(uint64_t seed, uint32_t blk, float (&z)[4]) {
    uint32_t c0 = blk, c1 = 0u, c2 = 0x6c6f676du, c3 = 0x656c0000u;
    uint32_t k0 = static_cast<uint32_t>(seed), k1 = static_cast<uint32_t>(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        const uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        c0 = h1 ^ c1 ^ k0; c1 = l1; c2 = h0 ^ c3 ^ k1; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const uint32_t a = h ? c2 : c0, b = h ? c3 : c1;
        const float u1 = (static_cast<float>(a >> 8) + 0.5f) * (1.0f / 16777216.0f);
        const float u2 = (static_cast<float>(b >> 8) + 0.5f) * (1.0f / 16777216.0f);
        const float r = sqrtf(-2.0f * __logf(u1));
        float sn, cs;
        __sincosf(6.283185307179586f * u2, &sn, &cs);
        z[2 * h] = r * cs;
        z[2 * h + 1] = r * sn;
    }
}

struct ClipCtx;
// Staging of one tile of a clip with on-device Philox noise (gain, roll, reflect padding as in stage_slots): four
// consecutive slots per thread, so one Philox block serves up to four samples.  Kept out of line: it is the rare
// path and must not change the register allocation or the code layout of the kernel's main loop.
__device__ __noinline__ void stage_noisy_tile(const ClipCtx& c, float* __restrict__ sb, int ns, int need, int j0, int T, int gtid);

// The two frame layouts.  n_fft = 2048: one real frame per warp (a 1024-point complex FFT of its even / odd samples).
// n_fft <= 1024: the warp's 1024 complex points are P = 1024 / n_fft independent n_fft-point FFTs of R points per lane
// (one FFT over the whole warp at 1024), each carrying two real frames as a + i b, so FPW = 2 P frames per warp.
// Frame j of a warp leaves its power spectrum at j * OFF in the warp's row.
template <int NFFT>
struct Geo {
    static_assert(NFFT == 2048 || NFFT == 1024 || NFFT == 512 || NFFT == 256, "n_fft");
    static constexpr int FPW = 2048 / NFFT;              // frames per warp pass
    static constexpr int TILE_F = kGroupWarps * FPW;     // frames per item
    static constexpr int NB = TILE_F / 8;                // 8-frame MMA column blocks per tile
    // spectrum pitch inside a row: >= n_fft/2 + 1 bins, == 16 (mod 32) so that the two frames g, g+1 that one
    // quarter-warp's LDS.128 B-operand loads touch sit 16 banks apart (1024: 528, 512: 272, 256: 144)
    static constexpr int OFF = NFFT / 2 + 16;
    static constexpr int R = (NFFT >= 1024 ? 1024 : NFFT) / 32;   // points per lane of one complex FFT (second radix)
    static_assert(OFF % 32 == 16 && (FPW - 1) * OFF + NFFT / 2 + 1 <= kRowFloats, "row layout");
};

// Shared-memory carve-up, shared by host (size) and device (pointers).  Everything of fixed size
// comes first so that its addresses are compile-time constants (no registers spent on pointers);
// the run-time sized arrays (staging buffers, filterbank) sit at the end.
template <int NFFT>
struct Smem {
    static constexpr size_t kBar = 0;                                    // kGroups mbarriers + 'TMA pending' flags
    static constexpr size_t kRed = kBar + 48;                            // + the filterbank-copy mbarrier at +32                            // per group: reduction scratch + broadcast
    static constexpr size_t kRedGroup = sizeof(long long) * 2 * kGroupWarps + 16;   // + bcast[3]: mean, std + eps, 'this group normalises'
    static constexpr size_t kCtx = kRed + kGroups * kRedGroup;           // per group two ClipCtx slots (ordinal & 1)
    static constexpr size_t kTab = kCtx + kGroups * 2 * 80;
    static constexpr size_t kStat = kTab + ((sizeof(MelTable) + 15) & ~size_t(15));   // per-thread fixed-point (sum, sumsq)
    static constexpr size_t kWin = kStat + sizeof(double) * 2 * kThreads;
    static constexpr size_t kTw = kWin + sizeof(float) * (NFFT / 2);     // first half of the window
    static constexpr size_t kUtw = kTw + sizeof(float2) * 32 * kTwRows;
    static constexpr size_t kScr = kUtw + ((NFFT == 2048) ? sizeof(float2) * 512 : 0);
    static constexpr size_t kSbuf = kScr + sizeof(float) * kWarps * kRowFloats;
    static_assert(kSbuf % 16 == 0 && kScr % 16 == 0 && kStat % 16 == 0 && kCtx % 16 == 0 && kRedGroup % 16 == 0, "alignment");
    static __host__ __device__ size_t melw_offset(int ns) { return kSbuf + sizeof(float) * kGroups * static_cast<size_t>(ns); }
    static __host__ __device__ size_t total(int ns, int n_dk) {
        return melw_offset(ns) + sizeof(float4) * 64 * static_cast<size_t>(n_dk);
    }
};

// Everything the staging and epilogue code needs to know about one clip.  Two slots per group live
// in shared memory (clip ordinal & 1: staging runs one item ahead of the epilogue) so that none of
// it occupies registers across the FFT.
struct alignas(16) ClipCtx {
    const void* src;     // first sample after the centre crop (fp32, or int16: see KParams::wave)
    const float* nz;     // host-drawn noise row or nullptr
    uint64_t seed;
    int lc;              // valid samples after pad/crop
    int shift, f0, f1, t0, t1;
    float nscale, gain;
    int plain;
    int silent_from;     // first tile that lies entirely in the zero padding (n_tiles if none); plain clips only
    int clip;            // index of the clip in the batch; -1 in the "next clip" slot = the batch is exhausted
    int t_begin, t_end;  // tile range of this virtual clip
};
__device__ __noinline__ void stage_noisy_tile(const ClipCtx& c, float* __restrict__ sb, int ns, int need, int j0, int T, int gtid) {
    const float* __restrict__ src = static_cast<const float*>(c.src);
    const int shift = c.shift, lc = c.lc;
    const float gain = c.gain, nscale = c.nscale;
    const uint64_t seed = c.seed;
    for (int q = gtid; 4 * q < ns; q += kGroupThreads) {
        float v4[4], zc[4];
        uint32_t blk_c = 0xffffffffu;   // block held in zc
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int e = 4 * q + k;
            int j = j0 + e;
            if (j < 0) j = -j;
            else if (j >= T) j = 2 * (T - 1) - j;
            float v = 0.0f;
            if (e < need && j >= 0 && j < T) {
                int i = j - shift;               // torch.roll: out[j] = in[(j - shift) mod T]
                if (i < 0) i += T;
                else if (i >= T) i -= T;
                if (i < lc) v = __ldg(src + i) * gain;
                const uint32_t blk = static_cast<uint32_t>(i) >> 2;
                if (blk != blk_c) { philox_normal4(seed, blk, zc); blk_c = blk; }
                const float z = (i & 2) ? ((i & 1) ? zc[3] : zc[2]) : ((i & 1) ? zc[1] : zc[0]);
                v = fmaf(z, nscale, v);
            }
            v4[k] = v;
        }
        *reinterpret_cast<float4*>(sb + 4 * q) = make_float4(v4[0], v4[1], v4[2], v4[3]);
    }
}
constexpr int kCtxSlot = 80;
static_assert(sizeof(ClipCtx) <= kCtxSlot && kCtxSlot % 16 == 0, "ClipCtx slot size");

// The address of sample k of clip samples x (fp32, or 16-bit PCM when PCM); its value as fp32 is clip_sample (resample.cuh).
template <bool PCM>
__device__ __forceinline__ const void* sample_addr(const void* x, long long k) {
    return PCM ? static_cast<const void*>(static_cast<const short*>(x) + k) : static_cast<const float*>(x) + k;
}

// The staging of a tile, slot by slot, for the slots [0, e_lo) and [e_lo + cnt, ns) that the bulk copy does not cover
// (rest = ns - cnt of them): reflect (torch.stft center=True) -> roll -> pad/crop -> gain, + noise; slots past `need`
// feed only frames >= `frames` and are zeroed.  `sample(i)` is clip sample i after the crop (i < lc).
template <class Sample>
__device__ __forceinline__ void stage_slots(const ClipCtx& c, float* __restrict__ sb, int rest, int e_lo, int cnt, int need, int j0,
                                            int T, int gtid, Sample sample) {
    const int shift = c.shift, lc = c.lc;
    for (int idx = gtid; idx < rest; idx += kGroupThreads) {
        const int e = idx < e_lo ? idx : idx + cnt;
        int j = j0 + e;
        if (j < 0) j = -j;
        else if (j >= T) j = 2 * (T - 1) - j;
        float v = 0.0f;
        if (e < need && j >= 0 && j < T) {
            int i = j - shift;               // torch.roll: out[j] = in[(j - shift) mod T]
            if (i < 0) i += T;
            else if (i >= T) i -= T;
            if (i < lc) v = sample(i) * c.gain;
            if (c.nscale != 0.0f) {
                const float z = c.nz ? __ldg(c.nz + i) : philox_normal(c.seed, static_cast<uint32_t>(i));
                v = fmaf(z, c.nscale, v);
            }
        }
        sb[e] = v;
    }
}

// ---------------------------------------------------------------------------------------
// Resampling inside the staging (Resampled instantiation, lm_forward_resampled).  Clip i holds len native samples;
// its resampled signal y has L' = ceil(q len / o) samples and is padded / centre-cropped like any clip, so staged
// sample i (after reflect and roll, i < lc = min(L', T)) is y[crop + i], crop = (L' - T) / 2 when L' > T.  y[m q + ph]
// is rs_sample (resample.cuh): the chain of lm_resample's kernels over the same padded tap row and the same x values (0
// outside [0, len)), hence bit-identical to lm_resample.
// ClipCtx has no room for the rate pair: the staging reads source / length / offset of the clip again per tile.
// lm_forward_spans stores only native samples [first, first + stored) of a clip: ClipCtx::src is then wave + offset - first
// (+ crop for a clip at the plan's rate), so x[k] is read where it is stored; lc, the crop, L' and the silent tiles still
// come from the whole clip's length.
// ---------------------------------------------------------------------------------------
struct RsClip {
    RsTaps g;         // g.q == 0: the clip is at the plan's rate (src already points past its crop)
    long long len;    // native samples (0 for a source index outside [-1, n_rs))
    long long lp;     // L': samples of y (len when the clip is at the plan's rate)
    long long crop;   // first sample of y kept by the centre crop
};
__device__ __forceinline__ RsClip rs_clip(const KParams& p, int clip) {
    RsClip r{{nullptr, nullptr, 1, 0, 0, 0}, p.length[clip], 0, 0};
    const int s = p.source[clip];
    r.lp = r.len;
    if (s < -1 || s >= p.n_rs) {   // device data: an invalid index makes an empty clip, nothing is read
        r.len = 0; r.lp = 0;
    } else if (s >= 0) {
        r.g = p.rs[s];
        r.lp = (static_cast<long long>(r.g.q) * r.len + r.g.o - 1) / r.g.o;   // 64-bit: q len overflows int for long recordings
    }
    r.crop = r.lp > p.T ? (r.lp - p.T) / 2 : 0;
    return r;
}

// lm_forward_spans: whether the stored span [f, f + stored) holds every native sample the staging of a clip reads: the
// resampler's read set (rs_read_span), or for a clip at the plan's rate (g.q == 0) its lc samples from the crop on.  Once
// per clip, by one thread.  Inline: as an out-of-line call from load_clip it cost the Resampled instantiations 32-56 bytes
// of stack and spills across the call.
__device__ __forceinline__ bool span_stored(const RsTaps& g, long long len, long long crop, int lc, int T, long long f,
                                            int stored) {
    long long lo = crop, hi = crop + lc;
    if (g.q) rs_read_span(g, len, T, &lo, &hi);
    return hi <= lo || (f <= lo && hi <= f + stored);
}

// One tile of a clip of lm_forward_resampled: stage_slots with the sample computed by rs_sample.  Kept out of line like
// stage_noisy_tile.
template <bool PCM>
__device__ __forceinline__ void stage_resampled_impl(const ClipCtx& c, const RsClip& r, float* __restrict__ sb, int ns, int need,
                                                     int j0, int T, int gtid) {
    const void* x = c.src;
    stage_slots(c, sb, ns, 0, 0, need, j0, T, gtid,
                [&](int i) { return r.g.q ? rs_sample<PCM>(r.g, x, r.len, r.crop + i) : clip_sample<PCM>(x, i); });
}
__device__ __noinline__ void stage_resampled_tile(const ClipCtx& c, const RsClip r, int pcm16, float* __restrict__ sb, int ns,
                                                  int need, int j0, int T, int gtid) {
    if (pcm16) stage_resampled_impl<true>(c, r, sb, ns, need, j0, T, gtid);
    else stage_resampled_impl<false>(c, r, sb, ns, need, j0, T, gtid);
}

// `nfft` is NFFT passed as a value: with the compile-time constant in the padded-signal bounds below, the compiler
// reassociates them and the churn that follows through the whole kernel measured 0.1-0.2 % slower at n_fft = 512.
// Resampled: lc = min(L', T) and src is the clip's first native sample, or its first sample after the crop for a clip at
// the plan's rate (rs_clip); `plain` then only decides silent tiles, the staging never takes the bulk-copy path.  With
// stored spans (lm_forward_spans) a clip whose span misses a sample the staging reads gets lc = 0: a zero-length clip.
template <int NFFT, Variant V>
__device__ __forceinline__ void load_clip(const KParams& p, int vclip, ClipCtx* __restrict__ c, int nfft) {
    constexpr bool PCM16 = V == Variant::Pcm16, RESAMPLE = V == Variant::Resampled;
    const int clip = vclip / p.split, chunk = vclip - clip * p.split;
    c->t_begin = chunk * p.tiles_per_chunk;
    c->t_end = (c->t_begin + p.tiles_per_chunk < p.n_tiles) ? c->t_begin + p.tiles_per_chunk : p.n_tiles;
    const long long off = p.offset[clip];
    const int len = p.length[clip];
    const int crop = len > p.T ? (len - p.T) / 2 : 0;       // centre crop
    c->clip = clip;
    c->lc = len < p.T ? len : p.T;
    c->src = sample_addr<PCM16>(p.wave, off + crop);
    if (RESAMPLE) {   // overrides the lines above rather than replacing them: an if / else moved the register allocation of every other instantiation
        const RsClip r = rs_clip(p, clip);
        long long start = off + (r.g.q ? 0 : r.crop);
        c->lc = r.lp < p.T ? static_cast<int>(r.lp) : p.T;
        if (p.first != nullptr) {   // lm_forward_spans: native sample k sits at wave[offset + k - first]
            const long long f = p.first[clip];
            if (!span_stored(r.g, r.len, r.crop, c->lc, p.T, f, p.stored[clip]))
                c->lc = 0;   // a sample the staging needs is not stored: a zero-length clip, nothing is read
            start -= f;
        }
        c->src = p.pcm16 ? sample_addr<true>(p.wave, start) : sample_addr<false>(p.wave, start);
    }
    int shift = 0, f0 = 0, f1 = 0, t0 = 0, t1 = 0;
    float nscale = 0.0f, gain = 1.0f;
    uint64_t seed = 0;
    if (p.aug != nullptr) {
        const lm_aug a = p.aug[clip];
        shift = a.shift % p.T;   // torch.roll takes any shift; the staging wraps once
        nscale = a.noise_scale; gain = a.gain;
        f0 = a.f0; f1 = a.f1; t0 = a.t0; t1 = a.t1; seed = a.seed;
    }
    c->shift = shift; c->f0 = f0; c->f1 = f1; c->t0 = t0; c->t1 = t1;
    c->nscale = nscale; c->gain = gain; c->seed = seed;
    c->nz = (p.noise != nullptr && nscale != 0.0f) ? p.noise + static_cast<size_t>(clip) * p.T : nullptr;
    c->plain = (shift == 0) && (nscale == 0.0f) && (gain == 1.0f);
    // A tile is silent when every sample it touches -- reflect padding included -- lies in the zero padding of a
    // plain clip: its power spectrum is exactly 0 and every feature sits at the dB floor, so FFT and mel are
    // skipped (ICBHI cycles average 2.7 s of the 5 s target).  Silence is monotone in the tile index.
    int silent_from = p.n_tiles;
    if (c->plain) {
        constexpr int tile_f = Geo<NFFT>::TILE_F;
        for (int t = p.n_tiles - 1; t >= 0; --t) {
            const int tf = t * tile_f;
            const int nf = (p.frames - tf) < tile_f ? (p.frames - tf) : tile_f;
            const int j0 = tf * p.hop - nfft / 2, j1 = j0 + (nf - 1) * p.hop + nfft - 1;   // first / last padded-signal index
            int lowest = j0 < 0 ? 0 : j0;                                                  // lowest clip index the tile reads
            if (j1 >= p.T) { const int r = 2 * (p.T - 1) - j1; lowest = r < lowest ? r : lowest; }
            if (c->lc > lowest) break;
            silent_from = t;
        }
    }
    c->silent_from = silent_from;
}

// DeviceNoise: tiles of clips with on-device Philox noise are staged four samples per thread (stage_noisy_tile).  The call
// costs the main loop ~3 % (registers live across it), so the host launches this instantiation only when the batch can
// contain such clips (augmentation records given, no host-drawn noise tensor); the headline path launches Plain.
// Resampled: lm_forward_resampled.  Every tile goes through stage_resampled_tile (no bulk copy; fp32 or 16-bit samples by
// p.pcm16 at run time, Philox noise drawn per sample); silent tiles still apply to un-augmented clips.
template <int NFFT, Variant V>
__global__ void __launch_bounds__(kThreads, 1) logmel_kernel(const KParams p) {
    constexpr bool EXTRA_OUT = V == Variant::ExtraOut, FASTNOISE = V == Variant::DeviceNoise;
    constexpr bool PCM16 = V == Variant::Pcm16, RESAMPLE = V == Variant::Resampled;
    using G = Geo<NFFT>;
    constexpr int TILE_F = G::TILE_F;
    constexpr int HALF = NFFT / 2;
    constexpr int ES = PCM16 ? 2 : 4;               // bytes per sample on the bulk-copy path (RESAMPLE never takes it)
    constexpr int NBC = G::NB < 4 ? G::NB : 4;   // MMA column blocks per walk of a mel tile's band
    constexpr int DUNROLL = G::NB > 2 ? 1 : 2;     // unroll of the band walk (n_fft <= 512: 4 blocks per step are enough)

    extern __shared__ __align__(128) unsigned char smem_raw[];
    using L = Smem<NFFT>;
    const int tid = threadIdx.x, lane_ = tid & 31;
    const int group = tid >> 8;                       // warp-uniform
    const int gtid = tid & (kGroupThreads - 1), gwarp_ = gtid >> 5;

    uint64_t* const mbar = reinterpret_cast<uint64_t*>(smem_raw + L::kBar) + group;
    volatile int* const s_pend = reinterpret_cast<volatile int*>(smem_raw + L::kBar + 16) + group;
    long long* const red = reinterpret_cast<long long*>(smem_raw + L::kRed + group * L::kRedGroup);
    float* const bcast = reinterpret_cast<float*>(smem_raw + L::kRed + group * L::kRedGroup + sizeof(long long) * 2 * kGroupWarps);
    ClipCtx* const s_ctx = reinterpret_cast<ClipCtx*>(smem_raw + L::kCtx) + 2 * group;
    const MelTable* const s_tab = reinterpret_cast<const MelTable*>(smem_raw + L::kTab);
    longlong2* const s_stat = reinterpret_cast<longlong2*>(smem_raw + L::kStat);
    float* const s_win = reinterpret_cast<float*>(smem_raw + L::kWin);
    float2* const s_tw = reinterpret_cast<float2*>(smem_raw + L::kTw);
    float2* const s_utw = reinterpret_cast<float2*>(smem_raw + L::kUtw);
    float* const rows = reinterpret_cast<float*>(smem_raw + L::kScr) + group * (kGroupWarps * kRowFloats);
    float* const sb = reinterpret_cast<float*>(smem_raw + L::kSbuf) + static_cast<size_t>(group) * p.ns;
    float4* const s_melw = reinterpret_cast<float4*>(smem_raw + L::melw_offset(p.ns));

    // ---- constants -> shared memory, once per (persistent) CTA, by all 16 warps -----------------
    for (int i = tid; i < HALF; i += kThreads) s_win[i] = p.window[i];
    for (int i = tid; i < 32 * kTwRows; i += kThreads) s_tw[i] = p.tw[i];
    if (NFFT == 2048)
        for (int i = tid; i < 512; i += kThreads) s_utw[i] = p.utw[i];
    // the banded filterbank (up to 96 KB) is needed first in the mel phase of the first item: one bulk copy, in flight
    // during the first FFT, completing on its own mbarrier (every thread waits for it once, before its first mel phase)
    uint64_t* const mbar_fb = reinterpret_cast<uint64_t*>(smem_raw + L::kBar + 32);
    if (tid == 0) {
        mbar_init(mbar_fb, 1);
        fence_mbar_init();
        mbar_expect_tx(mbar_fb, static_cast<uint32_t>(p.n_dk) * 1024u);
        bulk_g2s(s_melw, p.melw, static_cast<uint32_t>(p.n_dk) * 1024u, mbar_fb);
    }
    for (int i = tid; i < static_cast<int>(sizeof(MelTable) / 4); i += kThreads)
        reinterpret_cast<int*>(smem_raw + L::kTab)[i] = reinterpret_cast<const int*>(p.mel_table)[i];
    for (int i = gtid; i < kGroupWarps * kRowFloats; i += kGroupThreads) rows[i] = 0.0f;   // pad columns stay finite
    for (int i = gtid; i < p.ns; i += kGroupThreads) sb[i] = 0.0f;
    if (gtid == 0) {
        mbar_init(mbar, 1);
        fence_mbar_init();
        *s_pend = 0;
    }
    __syncthreads();   // the only CTA-wide barrier: from here on the groups never meet again

    // ---- this group's clips -----------------------------------------------------------------------
    const int nv = static_cast<int>(gridDim.x) * kGroups;
    const int n_virtual = p.B * p.split;
    const int clip0 = group * static_cast<int>(gridDim.x) + static_cast<int>(blockIdx.x);   // first (virtual) clip: static
    if (clip0 >= n_virtual) return;

    const int T = p.T, hop = p.hop, frames = p.frames, n_mels = p.n_mels;
    const size_t clip_elems = static_cast<size_t>(n_mels) * frames;

    uint32_t parity = 0;                   // mbarrier phase of the staging buffer (group-uniform)

    // ---- staging of one item into the group's buffer -------------------------------------------------
    // bulk part: [e_lo, e_lo + cnt) of the tile is src[j0 + e_lo ...] verbatim (plain clips only)
    auto bulk_range = [&](const ClipCtx* __restrict__ c, int tile_, int& e_lo, int& cnt) {
        e_lo = 0; cnt = 0;
        if (RESAMPLE || !p.use_tma || !c->plain) return;
        const int tf = tile_ * TILE_F;
        const int nf = (frames - tf) < TILE_F ? (frames - tf) : TILE_F;
        const int need = (nf - 1) * hop + NFFT;
        const int j0 = tf * hop - HALF;
        const int lo = j0 < 0 ? -j0 : 0;
        int hi = c->lc - j0;
        if (hi > need) hi = need;
        if (hi <= lo) return;
        if ((reinterpret_cast<uintptr_t>(sample_addr<PCM16>(c->src, j0 + lo)) & 15u) != 0 || (lo & 3) != 0) return;
        e_lo = lo;
        cnt = (hi - lo) & ~(16 / ES - 1);   // whole 16-byte units
    };
    auto tile_silent = [&](const ClipCtx* __restrict__ c, int tile_) -> bool {   // group-uniform
        return tile_ >= c->silent_from;
    };
    auto stage_bulk = [&](const ClipCtx* __restrict__ c, int tile_) {   // ONE thread of the group
        int e_lo, cnt;
        bulk_range(c, tile_, e_lo, cnt);
        if (cnt != 0) {
            const int j0 = tile_ * TILE_F * hop - HALF;
            const uint32_t bytes = static_cast<uint32_t>(cnt) * ES;
            // PCM16: raw samples to the end of the buffer; stage_gather expands them in place
            void* const dst = PCM16 ? static_cast<void*>(reinterpret_cast<unsigned char*>(sb) + 4 * p.ns - bytes) : sb + e_lo;
            fence_proxy_async();
            mbar_expect_tx(mbar, bytes);
            bulk_g2s(dst, sample_addr<PCM16>(c->src, j0 + e_lo), bytes, mbar);
        }
        *s_pend = (cnt != 0 ? 1 : 0) | (tile_silent(c, tile_) ? 2 : 0);   // bit 0: bulk copy pending, bit 1: silent tile
    };
    // returns (group-uniform) whether anything was written
    auto stage_gather = [&](const ClipCtx* __restrict__ cc, int tile_) -> bool {   // all threads of the group
        if (tile_silent(cc, tile_)) return false;   // nobody will read the buffer
        int e_lo, cnt;
        bulk_range(cc, tile_, e_lo, cnt);
        if (PCM16 && cnt != 0) {
            // The bulk copy left the raw samples of [e_lo, e_lo + cnt) in the last 2 cnt bytes of the buffer.  Expand them
            // to fp32 in place, 8 samples (16 bytes) per step and thread: every thread of a batch reads before any writes
            // (barrier), and a chunk's fp32 image never reaches the raw bytes of a LATER chunk (4 e_lo + 32 (c + 1) <=
            // 4 ns - 2 cnt + 16 c' for c' > c), so the batches can follow each other without a second barrier.
            mbar_wait(mbar, parity);
            parity ^= 1u;
            const int nch = cnt >> 3;
            const uint4* __restrict__ rawp = reinterpret_cast<const uint4*>(reinterpret_cast<const unsigned char*>(sb) + 4 * p.ns - 2 * cnt);
            float4* __restrict__ dst = reinterpret_cast<float4*>(sb + e_lo);
            constexpr float k = 1.0f / 32768.0f;   // as lm_pcm16_decode
            for (int c0 = 0; c0 < nch; c0 += 3 * kGroupThreads) {
                uint4 raw[3];
#pragma unroll
                for (int u = 0; u < 3; ++u) {
                    const int ch = c0 + u * kGroupThreads + gtid;
                    if (ch < nch) raw[u] = rawp[ch];
                }
                group_bar(group);
                if (c0 == 0 && gtid == 0) *s_pend = *s_pend & ~1;   // the copy has been waited for here, not at the top of the item
#pragma unroll
                for (int u = 0; u < 3; ++u) {
                    const int ch = c0 + u * kGroupThreads + gtid;
                    if (ch < nch) {
                        const int4 v = make_int4(static_cast<int>(raw[u].x), static_cast<int>(raw[u].y), static_cast<int>(raw[u].z), static_cast<int>(raw[u].w));
                        dst[2 * ch] = make_float4(static_cast<float>(static_cast<short>(v.x & 0xffff)) * k, static_cast<float>(v.x >> 16) * k,
                                                  static_cast<float>(static_cast<short>(v.y & 0xffff)) * k, static_cast<float>(v.y >> 16) * k);
                        dst[2 * ch + 1] = make_float4(static_cast<float>(static_cast<short>(v.z & 0xffff)) * k, static_cast<float>(v.z >> 16) * k,
                                                      static_cast<float>(static_cast<short>(v.w & 0xffff)) * k, static_cast<float>(v.w >> 16) * k);
                    }
                }
            }
        }
        const int rest = p.ns - cnt;   // slots the bulk copy does not cover: [0, e_lo) and [e_lo + cnt, ns)
        if (rest <= 0) return PCM16 && cnt != 0;
        const ClipCtx c = *cc;
        const int tf = tile_ * TILE_F;
        const int nf = (frames - tf) < TILE_F ? (frames - tf) : TILE_F;
        const int need = (nf - 1) * hop + NFFT;
        const int j0 = tf * hop - HALF;
        if (RESAMPLE) {
            stage_resampled_tile(*cc, rs_clip(p, c.clip), p.pcm16, sb, p.ns, need, j0, T, gtid);
            return true;
        }
        if (FASTNOISE && c.nscale != 0.0f && c.nz == nullptr && cnt == 0) {   // on-device noise (training batches): out of line
            stage_noisy_tile(*cc, sb, p.ns, need, j0, T, gtid);   // the context in shared memory, not the register copy
            return true;
        }
        stage_slots(c, sb, rest, e_lo, cnt, need, j0, T, gtid, [&](int i) { return clip_sample<PCM16>(c.src, i); });
        return true;
    };

    // ---- prologue: item 0 is staged before the loop; item it+1 is staged during item it ----------------
    if (gtid == 0) {
        load_clip<NFFT, V>(p, clip0, &s_ctx[0], NFFT);
        stage_bulk(&s_ctx[0], s_ctx[0].t_begin);
    }
    group_bar(group);
    stage_gather(&s_ctx[0], s_ctx[0].t_begin);
    group_bar(group);
    if (group == 1 && p.stagger_ns > 0) {   // spin (nanosleep may return early): ~2 cycles per ns
        const long long t_end = clock64() + 2LL * p.stagger_ns;
        while (clock64() < t_end) {}
    }

    bool fb_ready = false;                 // this thread has seen the filterbank copy complete
    s_stat[tid] = make_longlong2(0, 0);    // this thread's running (sum, sum of squares) of the clip's dB values, fixed point
    int tile = s_ctx[0].t_begin, t_end = s_ctx[0].t_end, ord = 0, clip = s_ctx[0].clip;   // tile, end of the tile range, clip ordinal (context slot = ord & 1), clip index

#if LM_TIMING
    long long t_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long t_last = clock64();
#endif
#pragma unroll 1
    for (;;) {
        const int tf = tile * TILE_F;                  // first frame of the tile
        const int st_item = *s_pend;
        if (st_item & 1) {
            mbar_wait(mbar, parity);
            parity ^= 1u;
        }
        LM_T(0);   // staging wait

        // ---- window + first butterfly stage + rest of FFT part 1 (registers; reads the staged samples) ----
        // hann[n + NFFT/2] = 1 - hann[n]:  a = v1 w + v2 (1 - w) = (v1 - v2) w + v2,  b = v1 w - v2 (1 - w) = (v1 + v2) w - v2
        // item it+1: its TMA part goes into the buffer consumed by (A); one thread; the clip's context slot is
        // filled when its first tile comes up
        const bool wrap = (tile + 1 == t_end);   // last tile of this (virtual) clip
        int tile1 = tile + 1, ord1 = ord;        // tile1 of a new clip is its t_begin: read from the context after barrier (B)
        if (wrap) ++ord1;
        auto issue_next = [&]() {
            if (gtid == 0) {
                ClipCtx* const cn = &s_ctx[ord1 & 1];
                if (wrap) {   // fetch the group's next (virtual) clip
                    const int nxt = nv + atomicAdd(p.work_counter, 1);
                    if (nxt < n_virtual) {
                        load_clip<NFFT, V>(p, nxt, cn, NFFT);
                        stage_bulk(cn, cn->t_begin);
                    } else {
                        cn->clip = -1;
                    }
                } else {
                    stage_bulk(cn, tile1);
                }
            }
        };
        if (__builtin_expect((st_item & 2) != 0, 0)) {
            group_bar(group);   // (A)
            issue_next();
            group_bar(group);   // (B)
            // ---- silent tile: every feature is the floor (or a mask's 0) ----------------------------------------
            const int nf = (frames - tf) < TILE_F ? (frames - tf) : TILE_F;
            const ClipCtx* __restrict__ cx = &s_ctx[ord & 1];
            float* __restrict__ out = p.out_norm + static_cast<size_t>(clip) * clip_elems;
            float* __restrict__ odb = (EXTRA_OUT && p.out_db) ? p.out_db + static_cast<size_t>(clip) * clip_elems : nullptr;
            float* __restrict__ omp = (EXTRA_OUT && p.out_melpow) ? p.out_melpow + static_cast<size_t>(clip) * clip_elems : nullptr;
            const int cf0 = cx->f0, cf1 = cx->f1, ct0 = cx->t0, ct1 = cx->t1;
            float ssum = 0.0f, qsum = 0.0f;
            for (int idx = gtid; idx < n_mels * TILE_F; idx += kGroupThreads) {
                const int m = idx / TILE_F, f = idx - m * TILE_F, tt = tf + f;
                if (f < nf) {
                    const float v = ((m >= cf0 && m < cf1) || (tt >= ct0 && tt < ct1)) ? 0.0f : p.floor_db;
                    const int o = m * frames + tt;
                    out[o] = v;
                    if (EXTRA_OUT) {
                        if (odb) odb[o] = v;
                        if (omp) omp[o] = 0.0f;
                    }
                    ssum += v;
                    qsum = fmaf(v, v, qsum);
                }
            }
            stat_add(&s_stat[tid], ssum, qsum);
        } else {
        lm_f2 z[32];
        if (LM_EXP != 2) {
            const int lane = launder(lane_), gw = launder(gwarp_);
            if (NFFT == 2048) {
                const float2* __restrict__ s2 = reinterpret_cast<const float2*>(sb + gw * hop);
                const float2* __restrict__ w2 = reinterpret_cast<const float2*>(s_win);
#pragma unroll
                for (int r = 0; r < 16; ++r) {
                    const float2 v1 = s2[32 * r + lane];
                    const float2 v2 = s2[32 * (r + 16) + lane];
                    const float2 w = w2[32 * r + lane];
                    const lm_f2 V1 = lm_pack(v1.x, v1.y), V2 = lm_pack(v2.x, v2.y), W = lm_pack(w.x, w.y);
                    z[r] = lm_fma2(lm_sub2(V1, V2), W, V2);
                    z[r + 16] = lm_fma2(lm_add2(V1, V2), W, lm_pack(-v2.x, -v2.y));
                }
            } else {
                // n_fft <= 1024: sub-FFT s = lane / R of the warp carries frames 2s (re) and 2s + 1 (im) as one complex
                // signal z = a + i b; lane s R + n2 takes samples n = R n1 + n2, so z[r] and z[r + 16] are n and
                // n + n_fft/2 as above.  (lane is laundered: at R = 32 the compiler cannot fold lane / R to 0 itself.)
                constexpr int R = G::R;
                const int n2 = R == 32 ? lane : lane & (R - 1), sub = R == 32 ? 0 : lane / R;
                const float* __restrict__ sa = sb + (G::FPW * gw + 2 * sub) * hop + n2;
                const float* __restrict__ sbb = sa + hop;
#pragma unroll
                for (int r = 0; r < 16; ++r) {
                    const float a1 = sa[R * r], a2 = sa[R * (r + 16)];
                    const float b1 = sbb[R * r], b2 = sbb[R * (r + 16)];
                    const lm_f2 V1 = lm_pack(a1, b1), V2 = lm_pack(a2, b2), W = lm_bcast(s_win[R * r + n2]);
                    z[r] = lm_fma2(lm_sub2(V1, V2), W, V2);
                    z[r + 16] = lm_fma2(lm_add2(V1, V2), W, lm_pack(-a2, -b2));
                }
            }
            lm_fft32_aos_from2(z);
        }
        LM_T(1);   // FFT part 1
        group_bar(group);   // (A) every warp of the group is done with the mel phase of the previous item
                            //     (rows are free) and with this item's staged samples (buffer is free)

        LM_T(2);   // barrier A
        issue_next();

        // ---- FFT part 2: transpose, second FFT, untangle -> 4|X|^2 in the warp's row ----------------------------
        if (LM_EXP == 3) {
            float acc = 0.f;
#pragma unroll
            for (int k = 0; k < 32; ++k) acc += lm_lo(z[k]) + lm_hi(z[k]);
            rows[gwarp_ * kRowFloats + lane_] = acc;
        }
        if (LM_EXP != 2 && LM_EXP != 3) {
            const int lane = launder(lane_), gw = launder(gwarp_);
            float* const scr = rows + gw * kRowFloats;
            float xr[32], xi[32];
            warp_cfft_part2<NFFT>(z, xr, xi, scr, s_tw, lane);
            const int srcl = (32 - lane) & 31;
            const bool l0 = (lane == 0);
            if (NFFT == 2048) {
                // Real-FFT untangle.  Bin k = lane + 32*k2 pairs with 1024-k, which lives in lane
                // (32-lane)&31 at slot 31-k2 (lane 0: slot (32-k2)&31) and comes over by warp shuffle.
                // Two pairs per packed op: k2 = i (lo half) and k2 = i+16 (hi half), i = 0..7; their
                // partners are the other lane's slots 31-i and 15-i, and the hi twiddle is the lo one
                // turned by pi/2: (c, s)(k+512) = (-s, c)(k).  The row was last read inside part 2
                // (followed by __syncwarp): 4|X|^2 goes straight into it, bin-major.
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float s_lr = l0 ? xr[(32 - i) & 31] : xr[31 - i];
                    const float s_li = l0 ? xi[(32 - i) & 31] : xi[31 - i];
                    const float s_hr = l0 ? xr[(16 - i) & 31] : xr[15 - i];
                    const float s_hi = l0 ? xi[(16 - i) & 31] : xi[15 - i];
                    const float b_lr = __shfl_sync(0xffffffffu, s_lr, srcl);
                    const float b_li = __shfl_sync(0xffffffffu, s_li, srcl);
                    const float b_hr = __shfl_sync(0xffffffffu, s_hr, srcl);
                    const float b_hi = __shfl_sync(0xffffffffu, s_hi, srcl);
                    const lm_f2 Ar = lm_pack(xr[i], xr[i + 16]), Ai = lm_pack(xi[i], xi[i + 16]);
                    const lm_f2 Br = lm_pack(b_lr, b_hr), Bi = lm_pack(b_li, b_hi);
                    const lm_f2 Er = lm_add2(Ar, Br), Ei = lm_sub2(Ai, Bi), Or = lm_add2(Ai, Bi), Oi = lm_sub2(Br, Ar);
                    const float2 cs = s_utw[lane + 32 * i];
                    const lm_f2 C = lm_pack(cs.x, -cs.y), S = lm_pack(cs.y, cs.x), nS = lm_pack(-cs.y, -cs.x);
                    const lm_f2 Tr = lm_fma2(C, Or, lm_mul2(S, Oi));
                    const lm_f2 Ti = lm_fma2(C, Oi, lm_mul2(nS, Or));
                    const lm_f2 Ur = lm_add2(Er, Tr), Ui = lm_add2(Ei, Ti), Vr = lm_sub2(Er, Tr), Vi = lm_sub2(Ei, Ti);
                    const lm_f2 PU = lm_fma2(Ur, Ur, lm_mul2(Ui, Ui)), PV = lm_fma2(Vr, Vr, lm_mul2(Vi, Vi));
                    scr[lane + 32 * i] = lm_lo(PU);
                    scr[lane + 32 * i + 512] = lm_hi(PU);
                    scr[1024 - lane - 32 * i] = lm_lo(PV);
                    scr[512 - lane - 32 * i] = lm_hi(PV);
                }
                {   // lane 0 only: bins 256 and 768 pair with each other (slots 8 and 24), twiddle pi/4
                    const float ar = xr[8], ai = xi[8], br = xr[24], bi = xi[24];
                    const float er = ar + br, ei = ai - bi, orr = ai + bi, oi = br - ar;
                    const float c = 0.70710678118654752440f;
                    const float tr = c * (orr + oi), ti = c * (oi - orr);
                    const float ur = er + tr, ui = ei + ti, vr = er - tr, vi = ei - ti;
                    if (l0) {
                        scr[256] = fmaf(ur, ur, ui * ui);
                        scr[768] = fmaf(vr, vr, vi * vi);
                    }
                }
            } else {
                // Per sub-FFT s, with R slots per lane: Z_s[k] = (xr, xi)[s R + k2] at k = lane + 32 k2, its partner
                // B = Z_s[n_fft - k] in lane (32 - lane) & 31 at slot R - 1 - k2 (lane 0: its own slot (R - k2) mod R).
                // A = Z_s[k]:  |Xa|^2 = |A + conj B|^2 / 4, |Xb|^2 = |A - conj B|^2 / 4.  Frames 2s and 2s + 1 go to
                // 2s OFF and (2s + 1) OFF in the row.
                constexpr int R = G::R;
#pragma unroll
                for (int s = 0; s < 32 / R; ++s) {
                    float* Pa = scr + (2 * s) * G::OFF;
                    float* Pb = Pa + G::OFF;
#pragma unroll
                    for (int k2 = 0; k2 < R / 2; ++k2) {
                        float br = __shfl_sync(0xffffffffu, xr[s * R + R - 1 - k2], srcl);
                        float bi = __shfl_sync(0xffffffffu, xi[s * R + R - 1 - k2], srcl);
                        if (l0) { br = xr[s * R + ((R - k2) & (R - 1))]; bi = xi[s * R + ((R - k2) & (R - 1))]; }
                        const float ar = xr[s * R + k2], ai = xi[s * R + k2];
                        const float ur = ar + br, ui = ai - bi, vr = ar - br, vi = ai + bi;
                        Pa[lane + 32 * k2] = fmaf(ur, ur, ui * ui);
                        Pb[lane + 32 * k2] = fmaf(vr, vr, vi * vi);
                    }
                    if (l0) {   // k = n_fft/2 pairs with itself: A = B
                        const float zr = xr[s * R + R / 2], zi = xi[s * R + R / 2];
                        Pa[NFFT / 2] = 4.0f * zr * zr;
                        Pb[NFFT / 2] = 4.0f * zi * zi;
                    }
                }
            }
        }
        LM_T(3);   // FFT part 2 (+ TMA issue)
        group_bar(group);   // (B) all power rows of the tile are in shared memory
        LM_T(4);   // barrier B

        // ---- mel phase: tensor cores, filterbank-stationary, up to kTileSlots 8-mel tiles per warp -------------
        if (!fb_ready) { mbar_wait(mbar_fb, 0); fb_ready = true; }
        {
            const int lane = launder(lane_), gw = launder(gwarp_);
            const int g = lane >> 2, tg = lane & 3;
            const int nf = (frames - tf) < TILE_F ? (frames - tf) : TILE_F;
            const ClipCtx* __restrict__ cx = &s_ctx[ord & 1];
            float* __restrict__ out = p.out_norm + static_cast<size_t>(clip) * clip_elems;
            float* __restrict__ odb = (EXTRA_OUT && p.out_db) ? p.out_db + static_cast<size_t>(clip) * clip_elems : nullptr;
            float* __restrict__ omp = (EXTRA_OUT && p.out_melpow) ? p.out_melpow + static_cast<size_t>(clip) * clip_elems : nullptr;
            const int cf0 = cx->f0, cf1 = cx->f1, ct0 = cx->t0, ct1 = cx->t1;
            float ssum = 0.0f, qsum = 0.0f;   // fp32 over this item's (at most 4 NB kTileSlots) values, fp64 across items
#pragma unroll 1
            for (int slot = 0; slot < kTileSlots; ++slot) {
                const int mt = s_tab->warp_tile[gw][slot];
                if (mt < 0 || LM_EXP == 1) break;
                const int kb = s_tab->kb[mt], ndk = s_tab->ndk[mt];
                const float4* __restrict__ wp = s_melw + static_cast<size_t>(s_tab->off[mt]) * 64 + lane;
                // B operand: frame n = g of column block nb lives in warp row (8 nb + g) / FPW at ((8 nb + g) % FPW) OFF;
                // this lane reads bins kb + 16 d + 4 tg .. +3 of it.  The band is walked once per NBC column blocks: at
                // n_fft = 256 (NB = 8) all accumulators at once would not fit in the registers beside the rest.
#pragma unroll 1
                for (int nb0 = 0; nb0 < G::NB; nb0 += NBC) {
                    const float* rp[NBC];
                    float acc_h[NBC][4], acc_l[NBC][4];   // products with the head / the residual of the power
#pragma unroll
                    for (int nb = 0; nb < NBC; ++nb) {
                        const int f = 8 * (nb0 + nb) + g;
                        rp[nb] = rows + (f / G::FPW) * kRowFloats + (f % G::FPW) * G::OFF + kb + 4 * tg;
#pragma unroll
                        for (int q = 0; q < 4; ++q) { acc_h[nb][q] = 0.f; acc_l[nb][q] = 0.f; }
                    }
#pragma unroll DUNROLL
                    for (int d = 0; d < ndk; ++d) {
                        // A operand rows 0-7: TF32 head of fb[., mel g], rows 8-15: its residual; one LDS.128 is one
                        // k-step's fragment.  k-step 1: logical k = tg -> bin 4tg, k = tg+4 -> bin 4tg+1; k-step 2: bins 4tg+2, 4tg+3
                        const float4 w1 = wp[64 * d], w2 = wp[64 * d + 32];
#pragma unroll
                        for (int nb = 0; nb < NBC; ++nb) {
                            const float4 pv = *reinterpret_cast<const float4*>(rp[nb] + 16 * d);
                            const uint32_t p0 = tf32_hi(pv.x), p1 = tf32_hi(pv.y), p2 = tf32_hi(pv.z), p3 = tf32_hi(pv.w);
                            const lm_f2 r01 = lm_sub2(lm_pack(pv.x, pv.y), lm_pack(__uint_as_float(p0), __uint_as_float(p1)));
                            const lm_f2 r23 = lm_sub2(lm_pack(pv.z, pv.w), lm_pack(__uint_as_float(p2), __uint_as_float(p3)));
                            mma_tf32(acc_h[nb], __float_as_uint(w1.x), __float_as_uint(w1.y), __float_as_uint(w1.z), __float_as_uint(w1.w), p0, p1);
                            mma_tf32(acc_l[nb], __float_as_uint(w1.x), __float_as_uint(w1.y), __float_as_uint(w1.z), __float_as_uint(w1.w),
                                     __float_as_uint(lm_lo(r01)), __float_as_uint(lm_hi(r01)));
                            mma_tf32(acc_h[nb], __float_as_uint(w2.x), __float_as_uint(w2.y), __float_as_uint(w2.z), __float_as_uint(w2.w), p2, p3);
                            mma_tf32(acc_l[nb], __float_as_uint(w2.x), __float_as_uint(w2.y), __float_as_uint(w2.z), __float_as_uint(w2.w),
                                     __float_as_uint(lm_lo(r23)), __float_as_uint(lm_hi(r23)));
                        }
                    }
                    // epilogue: c0:(head row, frame 2tg) c1:(head, 2tg+1) c2:(residual row, 2tg) c3:(residual, 2tg+1)
                    const int m = mt * 8 + g;
                    const bool ok_m = m < n_mels;
                    const bool mk_m = (m >= cf0) && (m < cf1);
#pragma unroll
                    for (int nb = 0; nb < NBC; ++nb) {
                        const lm_f2 mp2 = lm_add2(lm_add2(lm_pack(acc_h[nb][0], acc_h[nb][1]), lm_pack(acc_h[nb][2], acc_h[nb][3])),
                                                  lm_add2(lm_pack(acc_l[nb][0], acc_l[nb][1]), lm_pack(acc_l[nb][2], acc_l[nb][3])));
                        const int fl = 8 * (nb0 + nb) + 2 * tg, tt = tf + fl;
                        const int o = m * frames + tt;
                        const float mp0 = lm_lo(mp2), mp1 = lm_hi(mp2);
                        float v0 = (mp0 <= p.amin) ? p.floor_db : fmaf(p.db_scale, lg2_ftz(mp0), -p.db_offset);
                        float v1 = (mp1 <= p.amin) ? p.floor_db : fmaf(p.db_scale, lg2_ftz(mp1), -p.db_offset);
                        if (mk_m || ((tt >= ct0) && (tt < ct1))) v0 = 0.0f;
                        if (mk_m || ((tt + 1 >= ct0) && (tt + 1 < ct1))) v1 = 0.0f;
                        const bool ok0 = ok_m && (fl < nf), ok1 = ok_m && (fl + 1 < nf);
                        if (ok0) out[o] = v0;
                        if (ok1) out[o + 1] = v1;
                        if (EXTRA_OUT) {
                            if (odb) { if (ok0) odb[o] = v0; if (ok1) odb[o + 1] = v1; }
                            if (omp) { if (ok0) omp[o] = mp0; if (ok1) omp[o + 1] = mp1; }
                        }
                        const float u0 = ok0 ? v0 : 0.0f, u1 = ok1 ? v1 : 0.0f;
                        ssum += u0 + u1;
                        qsum = fmaf(u0, u0, fmaf(u1, u1, qsum));
                    }
                }
            }
            stat_add(&s_stat[tid], ssum, qsum);
        }

        }   // not silent
        LM_T(5);   // mel phase
        // ---- gather part of item it+1 (its TMA part is already in flight) -----------------------------
        const bool has1 = !wrap || (s_ctx[ord1 & 1].clip >= 0);   // written before (B) by thread 0
        if (wrap && has1) tile1 = s_ctx[ord1 & 1].t_begin;
        if (has1) {
            if (stage_gather(&s_ctx[ord1 & 1], tile1)) group_bar(group);   // (C) only for tiles that touch a clip edge
        }

        LM_T(6);   // gather + barrier C
        // ---- per-clip normalisation --------------------------------------------------------------------
        if (wrap) {
            if (p.normalize) {
                float* __restrict__ out = p.out_norm + static_cast<size_t>(clip) * clip_elems;
                long long s_acc = s_stat[tid].x, q_acc = s_stat[tid].y;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    s_acc += __shfl_xor_sync(0xffffffffu, s_acc, o);
                    q_acc += __shfl_xor_sync(0xffffffffu, q_acc, o);
                }
                if (lane_ == 0) { red[gwarp_] = s_acc; red[kGroupWarps + gwarp_] = q_acc; }
                group_bar(group);   // also orders every thread's dB stores before the re-read below
                if (gtid == 0) {
                    long long si = 0, qi = 0;
                    for (int w = 0; w < kGroupWarps; ++w) { si += red[w]; qi += red[kGroupWarps + w]; }
                    bool last = true;
                    if (p.split > 1) {
                        // this chunk's sums join the clip's; the group whose arrival completes the clip normalises it.
                        // The fence makes the group's dB stores (ordered before it by the barrier above) visible GPU-wide
                        // before the arrival counter moves.
                        atomicAdd(p.clip_stats + 2 * clip, static_cast<unsigned long long>(si));
                        atomicAdd(p.clip_stats + 2 * clip + 1, static_cast<unsigned long long>(qi));
                        __threadfence();
                        last = atomicAdd(p.clip_cnt + clip, 1) == p.split - 1;
                        if (last) {
                            __threadfence();
                            si = static_cast<long long>(__ldcg(p.clip_stats + 2 * clip));
                            qi = static_cast<long long>(__ldcg(p.clip_stats + 2 * clip + 1));
                            p.clip_stats[2 * clip] = 0ull;       // nobody else touches this clip's scratch any more
                            p.clip_stats[2 * clip + 1] = 0ull;
                            p.clip_cnt[clip] = 0;
                        }
                    }
                    const double s = static_cast<double>(si) * (1.0 / kStatScaleS), q = static_cast<double>(qi) * (1.0 / kStatScaleQ);
                    const double n = static_cast<double>(clip_elems);
                    const double mean = s / n;
                    double var = (q - s * mean) / (n - 1.0);   // unbiased, as torch.std
                    if (!(var > 0.0)) var = 0.0;
                    bcast[0] = static_cast<float>(mean);
                    bcast[1] = static_cast<float>(sqrt(var)) + p.norm_eps;
                    bcast[2] = last ? 1.0f : 0.0f;
                }
                group_bar(group);
                if (bcast[2] != 0.0f) {
                const float mean = bcast[0], inv = 1.0f / bcast[1];
                float4* __restrict__ o4 = reinterpret_cast<float4*>(out);
                const int n4 = (reinterpret_cast<uintptr_t>(out) & 15u) == 0 ? static_cast<int>(clip_elems >> 2) : 0;
                if (p.mc_out == nullptr && p.n_peer == 0) {
                    for (int i = gtid; i < n4; i += kGroupThreads) {
                        float4 v = __ldcg(o4 + i);
                        v.x = (v.x - mean) * inv;
                        v.y = (v.y - mean) * inv;
                        v.z = (v.z - mean) * inv;
                        v.w = (v.w - mean) * inv;
                        o4[i] = v;
                    }
                } else {
                    // fused all-gather: the same 16 bytes also go to the other ranks' buffers
                    const size_t gofs = static_cast<size_t>(clip) * clip_elems;   // the clip's offset inside a rank's slice
                    for (int i = gtid; i < n4; i += kGroupThreads) {
                        float4 v = __ldcg(o4 + i);
                        v.x = (v.x - mean) * inv;
                        v.y = (v.y - mean) * inv;
                        v.z = (v.z - mean) * inv;
                        v.w = (v.w - mean) * inv;
                        if (p.mc_out != nullptr) {
                            multimem_st_v4(p.mc_out + gofs + 4 * static_cast<size_t>(i), v);   // lands here and on every peer
                        } else {
                            o4[i] = v;
                            for (int r = 0; r < p.n_peer; ++r) reinterpret_cast<float4*>(p.peer[r] + gofs)[i] = v;
                        }
                    }
                }
                for (int i = (n4 << 2) + gtid; i < static_cast<int>(clip_elems); i += kGroupThreads)
                    out[i] = (__ldcg(out + i) - mean) * inv;
                }   // this group finishes the clip
                group_bar(group);   // bcast is rewritten at the next clip end
            }
            if (!has1) break;
            s_stat[tid] = make_longlong2(0, 0);
            clip = s_ctx[ord1 & 1].clip;
            tile = tile1;
            t_end = s_ctx[ord1 & 1].t_end;
            ++ord;
        } else {
            ++tile;
        }
        LM_T(7);   // normalisation
    }
    if (!fb_ready) mbar_wait(mbar_fb, 0);   // (all tiles silent) never leave a bulk copy in flight behind an exiting CTA
    // the last group to finish leaves the launch's counters at zero for the next launch that uses this slot
    if (gtid == 0) {
        const int active = n_virtual < nv ? n_virtual : nv;
        __threadfence();
        if (atomicAdd(p.work_counter + 1, 1) == active - 1) {
            p.work_counter[0] = 0;
            p.work_counter[1] = 0;
        }
    }
#if LM_TIMING
    if (lane_ == 0) {
        long long* o = g_timing + (static_cast<size_t>(blockIdx.x) * kWarps + (tid >> 5)) * 8;
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] = t_acc[i];
    }
#endif
}

}  // namespace lm
