// logmel_aux.cuh -- small companion kernels of the log-mel path.
//
//   resize_finish_kernel   FlexibleAudioPreprocessor.resize_spectrogram + augment_spectrogram + normalize
//                          (R/data/preprocessing_flexible.py:118-154, :106-116, order of :182-190):
//                          bilinear F.interpolate(size=(n_mels, target), align_corners=False).  The mel
//                          axis keeps its size, so the kernel is a 1-D linear interpolation along time
//                          (aten/src/ATen/native/UpSample.h: src = scale*(dst+0.5)-0.5 clamped at 0,
//                          scale = in/out), then the SpecAugment intervals, then (x-mean)/(std+eps).
//   pcm16_roundtrip_kernel the analyzers write every window to a temp .wav with soundfile's default
//                          PCM_16 subtype and read it back (R/realtime_analyzer_parallel.py:181-184):
//                          y = rint(clamp(x) * 32767) / 32768.  "Parity unpinned" (libsndfile is not in
//                          the reference tree); offered so window features can follow that accident.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/logmel_b200.h"

namespace lm {

constexpr int kAuxThreads = 512;

__device__ __forceinline__ float resize_sample(const float* __restrict__ row, int fin, int t, float scale) {
    float src = fmaf(scale, static_cast<float>(t) + 0.5f, -0.5f);
    if (src < 0.0f) src = 0.0f;
    int i0 = static_cast<int>(src);
    if (i0 > fin - 1) i0 = fin - 1;
    float lam = src - static_cast<float>(i0);
    lam = fminf(fmaxf(lam, 0.0f), 1.0f);
    const int i1 = (i0 + 1 < fin) ? i0 + 1 : i0;
    return (1.0f - lam) * row[i0] + lam * row[i1];
}

// one CTA per clip; in [B, n_mels, fin] -> out [B, n_mels, fout]
__global__ void __launch_bounds__(kAuxThreads) resize_finish_kernel(const float* __restrict__ in, float* __restrict__ out,
                                                                     const lm_aug* __restrict__ aug, int n_mels, int fin,
                                                                     int fout, int normalize, float eps) {
    __shared__ double red[2 * (kAuxThreads / 32)];
    __shared__ float bc[2];
    const int clip = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float* __restrict__ src = in + static_cast<size_t>(clip) * n_mels * fin;
    float* __restrict__ dst = out + static_cast<size_t>(clip) * n_mels * fout;
    int f0 = 0, f1 = 0, t0 = 0, t1 = 0;
    if (aug != nullptr) { f0 = aug[clip].f0; f1 = aug[clip].f1; t0 = aug[clip].t0; t1 = aug[clip].t1; }
    const float scale = static_cast<float>(fin) / static_cast<float>(fout);
    const int n = n_mels * fout;
    double s = 0.0, q = 0.0;
    for (int i = tid; i < n; i += kAuxThreads) {
        const int m = i / fout, t = i - m * fout;
        float v = (fin == fout) ? src[m * fin + t] : resize_sample(src + m * fin, fin, t, scale);
        if ((m >= f0 && m < f1) || (t >= t0 && t < t1)) v = 0.0f;
        dst[i] = v;
        const double d = static_cast<double>(v);
        s += d;
        q = fma(d, d, q);
    }
    if (!normalize) return;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        q += __shfl_xor_sync(0xffffffffu, q, o);
    }
    if (lane == 0) { red[warp] = s; red[kAuxThreads / 32 + warp] = q; }
    __syncthreads();
    if (tid == 0) {
        double ss = 0.0, qq = 0.0;
        for (int w = 0; w < kAuxThreads / 32; ++w) { ss += red[w]; qq += red[kAuxThreads / 32 + w]; }
        const double mean = ss / n;
        double var = (qq - ss * mean) / (static_cast<double>(n) - 1.0);
        if (!(var > 0.0)) var = 0.0;
        bc[0] = static_cast<float>(mean);
        bc[1] = static_cast<float>(sqrt(var)) + eps;
    }
    __syncthreads();
    const float mean = bc[0], inv = 1.0f / bc[1];
    for (int i = tid; i < n; i += kAuxThreads) dst[i] = (dst[i] - mean) * inv;   // own writes: same thread
}

__global__ void pcm16_roundtrip_kernel(const float* __restrict__ in, float* __restrict__ out, long long n) {
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
        float x = in[i];
        x = fminf(fmaxf(x, -1.0f), 1.0f);
        out[i] = rintf(x * 32767.0f) * (1.0f / 32768.0f);
    }
}

// T.AmplitudeToDB() on its own (R/src/data/preprocessing.py:46, TA/functional/functional.py:390-391):
// y = multiplier * log10(max(x, amin)) - offset, element-wise; the drop-in preprocessor's `amplitude_to_db` attribute.
__global__ void amplitude_to_db_kernel(const float* __restrict__ in, float* __restrict__ out, long long n, float db_scale, float amin,
                                       float db_offset) {
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride)
        out[i] = fmaf(db_scale, log2f(fmaxf(in[i], amin)), -db_offset);
}

// 16-bit PCM -> fp32: x / 32768 (exact), what torchaudio.load(normalize=True) hands the reference for a
// PCM_16 wav (R/src/data/preprocessing.py:57).  Eight samples per thread per pass: one 128-bit load, two
// 128-bit stores; `in` and `out` must be 16-byte aligned, the tail is done element-wise.
__global__ void pcm16_decode_kernel(const int16_t* __restrict__ in, float* __restrict__ out, long long n) {
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    const long long tid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const long long n8 = n >> 3;
    const int4* __restrict__ in8 = reinterpret_cast<const int4*>(in);
    float4* __restrict__ out4 = reinterpret_cast<float4*>(out);
    constexpr float k = 1.0f / 32768.0f;
    for (long long i = tid; i < n8; i += stride) {
        const int4 v = __ldcs(in8 + i);
        float4 a, b;
        a.x = static_cast<float>(static_cast<short>(v.x & 0xffff)) * k;
        a.y = static_cast<float>(v.x >> 16) * k;
        a.z = static_cast<float>(static_cast<short>(v.y & 0xffff)) * k;
        a.w = static_cast<float>(v.y >> 16) * k;
        b.x = static_cast<float>(static_cast<short>(v.z & 0xffff)) * k;
        b.y = static_cast<float>(v.z >> 16) * k;
        b.z = static_cast<float>(static_cast<short>(v.w & 0xffff)) * k;
        b.w = static_cast<float>(v.w >> 16) * k;
        out4[2 * i] = a;
        out4[2 * i + 1] = b;
    }
    for (long long i = (n8 << 3) + tid; i < n; i += stride) out[i] = static_cast<float>(in[i]) * k;
}

}  // namespace lm
