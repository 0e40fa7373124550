// resample.cuh -- the polyphase sinc resampler's device code: one view of a rate pair (RsTaps), the one tap chain every
// resampling path runs (rs_chain), the read span of a resampled clip (rs_read_span, host and device), and the two
// standalone kernels behind lm_resample.  The log-mel kernel's staging (logmel_kernel.cuh, Resampled) uses the same
// rs_sample.
//
// Polyphase sinc resampler = torchaudio.transforms.Resample(orig, new) with its defaults, the resampler of
// AudioPreprocessor.load_audio (R/src/data/preprocessing.py:63-65; TA/functional/functional.py
// _get_sinc_resample_kernel / _apply_sinc_resample_kernel).  With o = orig/gcd, q = new/gcd and
// xpad = pad(x, (width, width + o)):   y[m q + p] = sum_k kernel[p][k] xpad[m o + k],  k < 2 width + o.
// torchaudio runs that as a dense conv1d; all but ~2 width + 1 taps of a phase are (numerically) zero, so the host
// (logmel_capi.cu rs_design) keeps, per phase, the window of ntaps taps from k0[p] on, zero-padded to nt4 float4.
#pragma once
#include <cuda_runtime.h>

namespace lm {

// One rate pair as every resampling path reads it.  Device pointers in lm_resampler and KParams; lm_clip_span passes a
// view of its host design with the host k0 and no taps.
struct RsTaps {
    const float4* taps4;   // [q][nt4]: phase p's taps from k0[p] on, zero past its ntaps
    const int* k0;         // [q]: index of each phase's first kept tap in torchaudio's 2 width + o kernel
    int o, q, nt4, width;
};
static_assert(sizeof(RsTaps) == 32, "KParams holds LM_MAX_RESAMPLERS of them in 256 bytes");

// y = sum_t w[t] x(t) over the 4 nt4 padded taps of one phase, as one fmaf chain in t order.  Every resampler output --
// both standalone kernels and the log-mel staging -- is this chain over the same row and the same x values (0 outside
// the clip), so they agree bit for bit, non-finite input included (a zero padding tap over inf gives NaN everywhere).
template <class X>
__device__ __forceinline__ float rs_chain(const float4* __restrict__ w, int nt4, X x) {
    float acc = 0.0f;
    for (int t = 0; t < nt4; ++t) {
        const float4 wv = __ldg(w + t);
        acc = fmaf(wv.x, x(4 * t), acc);
        acc = fmaf(wv.y, x(4 * t + 1), acc);
        acc = fmaf(wv.z, x(4 * t + 2), acc);
        acc = fmaf(wv.w, x(4 * t + 3), acc);
    }
    return acc;
}

// Sample k of clip samples x (fp32, or 16-bit PCM when PCM) as fp32: x / 32768 for 16-bit PCM, as lm_pcm16_decode.
template <bool PCM>
__device__ __forceinline__ float clip_sample(const void* x, long long k) {
    return PCM ? static_cast<float>(__ldg(static_cast<const short*>(x) + k)) * (1.0f / 32768.0f) : __ldg(static_cast<const float*>(x) + k);
}

// y[mp] of a clip of len native samples x: the chain of phase mp mod q over x[m o + k0[ph] - width + t], x = 0 outside
// [0, len).  An output whose whole (padded) tap window lies inside the clip skips the bounds checks.
template <bool PCM>
__device__ __forceinline__ float rs_sample(const RsTaps& g, const void* x, long long len, long long mp) {
    const long long m = mp / g.q;
    const int ph = static_cast<int>(mp - m * g.q);
    const long long base = m * g.o + __ldg(g.k0 + ph) - g.width;   // native index of tap 0
    const float4* __restrict__ w = g.taps4 + static_cast<size_t>(ph) * g.nt4;
    if (base >= 0 && base + 4 * g.nt4 <= len) return rs_chain(w, g.nt4, [&](int i) { return clip_sample<PCM>(x, base + i); });
    return rs_chain(w, g.nt4, [&](int i) {
        const long long k = base + i;
        return (k >= 0 && k < len) ? clip_sample<PCM>(x, k) : 0.0f;
    });
}

// The native samples [*lo, *hi) that the staging of a resampled clip of len samples reads (lm_clip_span): every x[k],
// 0 <= k < len, that the chain of an output y[crop + i], i < lc, touches, zero padding taps included (a non-finite sample
// under a zero tap still poisons the sum).  Empty: *lo == *hi == 0.  For one phase the tap window moves right with m, so
// the lowest index comes from the first q outputs of the crop and the highest from the last q; the windows of
// neighbouring outputs overlap, so the indices in between are all read.  Host (lm_clip_span) and device (the
// lm_forward_spans check) run this same code on the same k0 table; it reads no taps.
__host__ __device__ inline void rs_read_span(const RsTaps& g, long long len, int T, long long* lo, long long* hi) {
    const int o = g.o, q = g.q;
    const long long lp = (static_cast<long long>(q) * len + o - 1) / o;
    const long long lc = lp < T ? lp : T, crop = lp > T ? (lp - T) / 2 : 0;
    *lo = 0; *hi = 0;
    if (lc <= 0) return;
    const int n = lc < q ? static_cast<int>(lc) : q;
    long long a = 0, b = 0;
    for (int side = 0; side < 2; ++side) {
        const long long mp0 = side ? crop + lc - n : crop;
        long long m = mp0 / q;
        int ph = static_cast<int>(mp0 - m * q);
        for (int j = 0; j < n; ++j) {
            const long long base = m * o + g.k0[ph] - g.width;
            if (side == 0 && (j == 0 || base < a)) a = base;
            if (side == 1 && (j == 0 || base + 4 * g.nt4 > b)) b = base + 4 * g.nt4;
            if (++ph == q) { ph = 0; ++m; }
        }
    }
    if (a < 0) a = 0;
    if (b > len) b = len;
    if (b > a) { *lo = a; *hi = b; }
}

// lm_resample for rate pairs whose tiled span does not fit in shared memory: one output sample per thread (rs_sample);
// a block's outputs share their input span through L1.
// grid.y = row (channel / clip): rows of equal length `n_in`, `in_stride` / `out_stride` floats apart
__global__ void resample_kernel(const float* __restrict__ x_all, long long n_in, long long in_stride,
                                float* __restrict__ y_all, long long n_out, long long out_stride, const RsTaps g) {
    const long long j = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (j >= n_out) return;
    const float* __restrict__ x = x_all + static_cast<long long>(blockIdx.y) * in_stride;
    y_all[static_cast<long long>(blockIdx.y) * out_stride + j] = rs_sample<false>(g, x, n_in, j);
}

// The same resampler, tiled: a block produces kRsChunk consecutive outputs of one row from ONE copy of their input
// span in shared memory (loaded coalesced, zero outside the row: each input sample feeds ~ntaps * q / o outputs), the
// taps fetched as 128-bit read-only loads.  k0max = the largest k0[p].
constexpr int kRsChunk = 1024, kRsThreads = 256;
__global__ void __launch_bounds__(kRsThreads) resample_tiled_kernel(const float* __restrict__ x_all, long long n_in, long long in_stride,
                                                                     float* __restrict__ y_all, long long n_out, long long out_stride,
                                                                     const RsTaps g, int k0max) {
    extern __shared__ float sx[];
    const int o = g.o, q = g.q, nt4 = g.nt4;
    const float* __restrict__ x = x_all + static_cast<long long>(blockIdx.y) * in_stride;
    float* __restrict__ y = y_all + static_cast<long long>(blockIdx.y) * out_stride;
    const long long j0 = static_cast<long long>(blockIdx.x) * kRsChunk;
    const int n_here = static_cast<int>((n_out - j0 < kRsChunk) ? (n_out - j0) : kRsChunk);
    const long long m0 = j0 / q;
    const unsigned p0 = static_cast<unsigned>(j0 - m0 * q);
    const long long x_lo = m0 * o - g.width;                                           // tap 0 of the first output at the earliest
    const int m_span = static_cast<int>((p0 + static_cast<unsigned>(n_here) - 1u) / static_cast<unsigned>(q));
    const int span = m_span * o + k0max + 4 * nt4;                                     // covers the last output's last (padded) tap
    for (int i = threadIdx.x; i < span; i += kRsThreads) {
        const long long xi = x_lo + i;
        sx[i] = (xi >= 0 && xi < n_in) ? __ldg(x + xi) : 0.0f;
    }
    __syncthreads();
    for (int d = threadIdx.x; d < n_here; d += kRsThreads) {
        const unsigned t = p0 + static_cast<unsigned>(d);
        const unsigned dm = t / static_cast<unsigned>(q), p = t - dm * static_cast<unsigned>(q);
        // an index into sx, not a pointer: through a pointer argument the loop-invariant tail arithmetic of the chain
        // moved into this loop (34 registers, 3-4 % slower at 4 and 10 kHz)
        const int s0 = dm * o + __ldg(g.k0 + p);
        y[j0 + d] = rs_chain(g.taps4 + static_cast<size_t>(p) * nt4, nt4, [&](int i) { return sx[s0 + i]; });
    }
}

}  // namespace lm
