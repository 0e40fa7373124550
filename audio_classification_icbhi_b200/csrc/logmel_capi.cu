// logmel_capi.cu -- extern "C" boundary of liblogmel_b200.so (see include/logmel_b200.h).
//
// Host side only: plan construction (twiddles, banded filterbank rows), launch, and the
// host-buffer pipeline.  No torch types, no ATen: plain pointers and sizes.
#include <math.h>
#include <stdlib.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <iterator>
#include <map>
#include <mutex>
#include <new>
#include <utility>
#include <vector>

#include <nvtx3/nvToolsExt.h>   // header-only NVTX v3: ranges are no-ops unless a profiler is attached

#include "logmel_kernel.cuh"
#include "logmel_aux.cuh"

namespace {

thread_local char g_cuda_err[256] = "";

int cuda_fail(cudaError_t e, const char* what) {
    snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", what, cudaGetErrorString(e));
    return LM_ERR_CUDA;
}
#define LM_CUDA(call)                                        \
    do {                                                     \
        cudaError_t _e = (call);                             \
        if (_e != cudaSuccess) return cuda_fail(_e, #call);  \
    } while (0)

// Makes a device current for the guard's lifetime and restores the caller's device afterwards, so that every entry
// point returns with the caller's device current.  DeviceOf(ptr) picks the device that owns a pointer: the companion
// entry points take raw device pointers and a stream but no plan (a caller on cuda:0 may hold tensors of cuda:1).
struct DeviceOf {
    int prev = -1, dev = -1;   // dev >= 0: switched away from prev
    cudaError_t err = cudaSuccess;
    explicit DeviceOf(int device) { enter(device); }
    explicit DeviceOf(const void* ptr) {
        cudaPointerAttributes a{};
        if (ptr && cudaPointerGetAttributes(&a, ptr) == cudaSuccess && a.type == cudaMemoryTypeDevice) enter(a.device);
        cudaGetLastError();
    }
    ~DeviceOf() { if (dev >= 0) cudaSetDevice(prev); }
    DeviceOf(const DeviceOf&) = delete;
    DeviceOf& operator=(const DeviceOf&) = delete;

  private:
    void enter(int device) {
        if ((err = cudaGetDevice(&prev)) != cudaSuccess || device == prev) return;
        if ((err = cudaSetDevice(device)) == cudaSuccess) dev = device;
    }
};

// NVTX range around a C-ABI entry point (SURVEY.md section 5: ranges around plan / execute), visible in Nsight Systems / Compute
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

constexpr int kSlots = 3;   // host pipeline depth
constexpr int kCounters = 1024;      // launches of one plan that may be in flight at once (on any streams); a slot is
                                     // re-zeroed on the launching stream right before its kernel, so launches on ONE
                                     // stream never interfere, and 1024 concurrent streams per plan are out of reach
constexpr int kMaxSplitClips = 512;  // small-batch mode is used below 2 * SM count clips

struct HostSlot {
    cudaStream_t stream = nullptr;
    unsigned char* d_wave = nullptr;  size_t cap_wave = 0; // bytes of fp32 or 16-bit samples
    float* d_noise = nullptr;     size_t cap_noise = 0;
    float* d_out = nullptr;       size_t cap_out = 0;
    // per-chunk metadata, one pinned staging block and one device block: [offset int64 x n][aug 40 B x n][length int32 x n]
    // (a copy from the caller's pageable arrays would make cudaMemcpyAsync wait for the stream, i.e. for the
    //  chunk's waveform copy, and stall the pipeline once per chunk)
    unsigned char* d_meta = nullptr;
    unsigned char* h_meta = nullptr;   // pinned
    int cap_clips = 0;
};

using KernelFn = void (*)(lm::KParams);

// What a plan of one n_fft and hop needs from the kernel's compile-time layout (lm::Geo, lm::Smem).
struct Geometry {
    int tile_f;    // frames per item
    int ns;        // staged floats per item: (tile_f - 1) * hop + n_fft, rounded up to 4
    int row_cap;   // a mel band of the last frame of a warp row (at (FPW - 1) * OFF) must end before this row offset
    int nc;        // points of one complex FFT: the twiddle between its two stages is W_nc^(k1 n2)
    size_t (*smem_total)(int ns, int n_dk);
    KernelFn kernels[lm::kVariants];   // by lm::Variant
};

template <int NFFT>
Geometry geometry(int hop) {
    using G = lm::Geo<NFFT>;
    using V = lm::Variant;
    // Philox noise drawn in the kernel has its own staging instantiation (DeviceNoise) at n_fft = 2048 only; the other
    // sizes stage it in the Plain kernel.
    constexpr V device_noise = NFFT == 2048 ? V::DeviceNoise : V::Plain;
    return {G::TILE_F, ((G::TILE_F - 1) * hop + NFFT + 3) & ~3, lm::kRowFloats - (G::FPW - 1) * G::OFF, 32 * G::R,
            &lm::Smem<NFFT>::total,
            {lm::logmel_kernel<NFFT, V::Plain>, lm::logmel_kernel<NFFT, V::ExtraOut>, lm::logmel_kernel<NFFT, V::Pcm16>,
             lm::logmel_kernel<NFFT, device_noise>, lm::logmel_kernel<NFFT, V::Resampled>}};
}

// The one place where a run-time n_fft (validated by lm_plan_create) becomes a compile-time size.
Geometry geometry(int n_fft, int hop) {
    switch (n_fft) {
        case 2048: return geometry<2048>(hop);
        case 1024: return geometry<1024>(hop);
        case 512: return geometry<512>(hop);
        default: return geometry<256>(hop);
    }
}

}  // namespace

// ---- polyphase sinc resampler (torchaudio.transforms.Resample defaults) ---------------------------------------
struct lm_resampler {
    int device = 0;
    lm::RsTaps rs{};          // device tables (rs_design), read by both lm_resample kernels and lm_forward_resampled
    int k0max = 0;
    size_t tile_smem = 0;     // tiled kernel: shared memory for the widest input span of a 1024-output chunk; 0 = the
                              // span does not fit: the untiled kernel is used
};

struct lm_plan {
    int device = 0;
    int n_fft = 0, hop = 0, n_mels = 0, T = 0, frames = 0, n_freqs = 0;
    int tile_f = 0, n_tiles = 0, ns = 0, n_dk = 0, fb_nnz = 0;
    int sm_count = 0, max_ctas = 0, use_tma = 1, stagger_ns = 0;
    int host_chunk_clips = 0;   // lm_forward_host chunk size; 0 = automatic
    size_t smem_bytes = 0;
    KernelFn kernels[lm::kVariants] = {};
    float db_mult = 10.f, amin = 1e-10f, db_offset = 0.f, floor_db = -100.f, norm_eps = 1e-8f;
    // device constants
    float* d_window = nullptr;
    float2* d_tw = nullptr;
    float2* d_utw = nullptr;
    float4* d_melw = nullptr;
    lm::MelTable* d_tab = nullptr;
    // host pipeline
    HostSlot slots[kSlots];
    bool slots_ready = false;
    std::atomic<long long> launches{0};
    int* d_counters = nullptr;   // kCounters x {work counter, finished groups} for the kernel's dynamic clip scheduling, one pair per launch in flight
    // small-batch mode scratch, one block per launch in flight: [kMaxSplitClips][2] 64-bit sums, then [kMaxSplitClips] arrival counters
    unsigned char* d_split = nullptr;
    int split_override = 0;      // 0 = automatic, 1 = never split, k > 1 = at most k chunks per clip
    std::mutex host_mu;          // lm_forward_host*: one caller at a time per plan (plan-owned staging buffers)
};

namespace {

int free_plan(lm_plan* p) {
    if (!p) return LM_OK;
    DeviceOf on(p->device);
    cudaFree(p->d_window); cudaFree(p->d_tw); cudaFree(p->d_utw); cudaFree(p->d_melw); cudaFree(p->d_tab); cudaFree(p->d_counters); cudaFree(p->d_split);
    for (auto& s : p->slots) {
        if (s.stream) cudaStreamDestroy(s.stream);
        cudaFree(s.d_wave); cudaFree(s.d_noise); cudaFree(s.d_out);
        cudaFree(s.d_meta);
        if (s.h_meta) cudaFreeHost(s.h_meta);
    }
    delete p;
    return LM_OK;
}

lm::KParams make_params(const lm_plan* p) {
    lm::KParams k{};
    k.T = p->T; k.hop = p->hop; k.frames = p->frames; k.n_mels = p->n_mels; k.n_tiles = p->n_tiles;
    k.ns = p->ns; k.n_dk = p->n_dk; k.use_tma = p->use_tma; k.stagger_ns = p->stagger_ns;
    k.db_scale = static_cast<float>(static_cast<double>(p->db_mult) * 0.30102999566398119521);
    k.amin = p->amin; k.db_offset = p->db_offset; k.floor_db = p->floor_db;
    k.norm_eps = p->norm_eps;
    k.window = p->d_window; k.tw = p->d_tw; k.utw = p->d_utw; k.melw = p->d_melw; k.mel_table = p->d_tab;
    return k;
}

// Raises the dynamic shared-memory limit of a plan's kernel instantiations.  The limit belongs to the kernel on the
// current device, not to the plan, and plans of one n_fft with other hops or mel counts need different sizes: it only
// ever grows, so creating a smaller plan cannot break launches of a larger one made earlier.
std::mutex g_smem_mu;
std::map<std::pair<const void*, int>, size_t> g_smem_limit;   // (kernel, device) -> limit set so far

cudaError_t set_smem_limit(const KernelFn (&kernels)[lm::kVariants], int device, size_t bytes) {
    std::lock_guard<std::mutex> lock(g_smem_mu);
    for (KernelFn f : kernels) {
        size_t& cur = g_smem_limit[std::make_pair(reinterpret_cast<const void*>(f), device)];
        if (bytes <= cur) continue;
        const cudaError_t e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes));
        if (e != cudaSuccess) return e;
        cur = bytes;
    }
    return cudaSuccess;
}

// Small batches: fewer clips than 8-warp groups on the GPU.  Cut every clip into `split` chunks of `tiles_per_chunk`
// whole tiles so that (almost) every group gets one chunk, and at most `split_override` chunks when that is > 1.  When
// normalising, the chunks' statistics are combined with integer atomics (logmel_kernel.cuh) in a scratch block that
// holds kMaxSplitClips clips.
void choose_split(const lm_plan* p, int B, int groups, bool normalize, int* split, int* tiles_per_chunk) {
    *split = 1;
    *tiles_per_chunk = p->n_tiles;
    if (p->split_override == 1 || B >= groups || p->n_tiles < 2 || (normalize && B > kMaxSplitClips)) return;
    int want = groups / B;
    if (p->split_override > 1) want = std::min(want, p->split_override);
    want = std::max(1, std::min(want, p->n_tiles));
    *tiles_per_chunk = (p->n_tiles + want - 1) / want;
    *split = (p->n_tiles + *tiles_per_chunk - 1) / *tiles_per_chunk;
}

// A batch as the kernel reads it: clip i is samples [offset[i], offset[i] + length[i]), fp32 or, when pcm16, 16-bit PCM
// expanded to x / 32768 inside the staging (no decode kernel).  lm_forward_resampled adds the rate of each clip: that of
// resamplers[source[i]], or the plan's rate for -1.
// lm_forward_spans adds the stored span of each clip: native samples [first[i], first[i] + stored[i]) from offset[i] on.
struct Batch {
    const void* samples; int32_t pcm16;   // 0 or 1; lm_forward_resampled / lm_forward_spans take it from the caller
    const int64_t* offset; const int32_t* length; int32_t B;
    const lm_aug* aug; const float* noise;
    const int32_t* source = nullptr; const lm_resampler* const* resamplers = nullptr; int n_resamplers = 0;
    const int64_t* first = nullptr; const int32_t* stored = nullptr;
};

// Where the features go: `norm` always, dB and mel power when given.  lm_forward_gather also stores the normalised
// features into the other ranks' gathered buffers (`peers`) or through a multicast address (`mc`).
struct Outputs {
    float* norm; float* db = nullptr; float* melpow = nullptr;
    float* const* peers = nullptr; int n_peers = 0; float* mc = nullptr;
};

// The kernel instantiation of a launch: resampled and 16-bit batches have no dB / mel power outputs.
int pick_variant(const Batch& b, const Outputs& o, lm::Variant* v) {
    using V = lm::Variant;
    const bool extra = (o.db != nullptr) || (o.melpow != nullptr);
    if ((b.source != nullptr || b.pcm16) && extra) return LM_ERR_UNSUPPORTED;
    const bool device_noise = (b.aug != nullptr) && (b.noise == nullptr);   // clips may ask for Philox noise drawn in the kernel
    *v = b.source ? V::Resampled : b.pcm16 ? V::Pcm16 : extra ? V::ExtraOut : device_noise ? V::DeviceNoise : V::Plain;
    return LM_OK;
}

int launch(lm_plan* p, const Batch& b, const Outputs& o, int32_t normalize, cudaStream_t stream) {
    if (b.B == 0) return LM_OK;
    lm::Variant v;
    if (const int rc = pick_variant(b, o, &v)) return rc;
    lm::KParams k = make_params(p);
    for (int r = 0; r < o.n_peers; ++r) k.peer[r] = o.peers[r];
    k.n_peer = o.n_peers; k.mc_out = o.mc;
    k.wave = b.samples; k.offset = reinterpret_cast<const long long*>(b.offset); k.length = b.length;
    k.aug = b.aug; k.noise = b.noise; k.out_norm = o.norm; k.out_db = o.db; k.out_melpow = o.melpow;
    k.B = b.B; k.normalize = normalize;
    // lm_forward_resampled: every clip through the resampling staging, the sample format a run-time flag
    k.source = b.source; k.pcm16 = b.pcm16; k.n_rs = b.n_resamplers;
    for (int r = 0; r < b.n_resamplers; ++r) k.rs[r] = b.resamplers[r]->rs;
    k.first = reinterpret_cast<const long long*>(b.first); k.stored = b.stored;
    const long long seq = p->launches.fetch_add(1);
    k.work_counter = p->d_counters + 2 * (seq % kCounters);   // zero now, left at zero by the kernel (no memset per launch)
    const int cap = p->max_ctas > 0 ? p->max_ctas : p->sm_count;
    choose_split(p, b.B, cap * lm::kGroups, normalize != 0, &k.split, &k.tiles_per_chunk);
    if (k.split > 1 && normalize) {
        unsigned char* blk = p->d_split + static_cast<size_t>(seq % kCounters) * (kMaxSplitClips * 20);
        k.clip_stats = reinterpret_cast<unsigned long long*>(blk);
        k.clip_cnt = reinterpret_cast<int*>(blk + kMaxSplitClips * 16);
        // zero at plan creation; the group that completes a clip resets its entries
    }
    const int grid = std::min<int>(b.B * k.split, cap);
    p->kernels[static_cast<int>(v)]<<<grid, lm::kThreads, p->smem_bytes, stream>>>(k);
    LM_CUDA(cudaGetLastError());
    return LM_OK;
}

// What an entry point needs beyond plan, clips and `norm`: `source` (Resampled, Spans), `first` / `stored` (Spans),
// 16-byte aligned outputs (Gather).
enum class Call { Plain, Gather, Resampled, Spans };

// Every device-input entry point: the argument check, in the order its statuses are returned (device-free up to the
// first plan dereference), then an NVTX range named after the entry point, the plan's device made current, one launch.
int forward_on_device(const char* name, Call call, lm_plan* p, const Batch& b, const Outputs& o, int32_t normalize,
                      void* stream) {
    if (!p || b.B < 0 || b.n_resamplers < 0 || b.n_resamplers > LM_MAX_RESAMPLERS || (b.n_resamplers > 0 && !b.resamplers) ||
        (b.pcm16 != 0 && b.pcm16 != 1) || o.n_peers < 0 || o.n_peers > lm::kMaxPeers)
        return LM_ERR_INVALID_ARG;
    for (int r = 0; r < b.n_resamplers; ++r)
        if (!b.resamplers[r]) return LM_ERR_INVALID_ARG;
    if (b.B == 0) return LM_OK;
    const bool resampled = call == Call::Resampled || call == Call::Spans;
    if (!b.samples || !b.offset || !b.length || !o.norm || (resampled && !b.source) ||
        (call == Call::Spans && (!b.first || !b.stored)) || (o.n_peers > 0 && !o.peers))
        return LM_ERR_INVALID_ARG;
    if (call == Call::Gather) {
        // the gather rides on the 16-byte stores of the normalisation pass
        if ((static_cast<size_t>(p->n_mels) * p->frames) % 4 != 0) return LM_ERR_UNSUPPORTED;
        if ((reinterpret_cast<uintptr_t>(o.norm) & 15u) || (reinterpret_cast<uintptr_t>(o.mc) & 15u)) return LM_ERR_INVALID_ARG;
        for (int r = 0; r < o.n_peers; ++r)
            if (!o.peers[r] || (reinterpret_cast<uintptr_t>(o.peers[r]) & 15u)) return LM_ERR_INVALID_ARG;
    }
    for (int r = 0; r < b.n_resamplers; ++r)
        if (b.resamplers[r]->device != p->device) return LM_ERR_INVALID_ARG;
    NvtxRange nvtx(name);
    DeviceOf on(p->device);
    if (on.err) return cuda_fail(on.err, "cudaSetDevice");
    return launch(p, b, o, normalize, static_cast<cudaStream_t>(stream));
}

int ensure_slots(lm_plan* p) {
    if (p->slots_ready) return LM_OK;
    for (auto& s : p->slots) LM_CUDA(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
    p->slots_ready = true;
    return LM_OK;
}

template <class Tp>
int grow(Tp** ptr, size_t* cap, size_t want) {
    if (want <= *cap) return LM_OK;
    if (*ptr) LM_CUDA(cudaFree(*ptr));
    *ptr = nullptr; *cap = 0;
    LM_CUDA(cudaMalloc(reinterpret_cast<void**>(ptr), want * sizeof(Tp)));
    *cap = want;
    return LM_OK;
}

// ---- plan creation steps ------------------------------------------------------------------------------------------

// The checks of lm_plan_create that need no device, in the order the status codes are returned.
int validate_config(const lm_config& cfg) {
    if (cfg.n_fft != 2048 && cfg.n_fft != 1024 && cfg.n_fft != 512 && cfg.n_fft != 256) return LM_ERR_UNSUPPORTED;
    if (cfg.hop < 2 || (cfg.hop & 1) || cfg.hop > cfg.n_fft / 4) return LM_ERR_UNSUPPORTED;
    if (cfg.n_mels < 1 || cfg.n_mels > 256) return LM_ERR_UNSUPPORTED;
    if (cfg.target_len <= cfg.n_fft / 2) return LM_ERR_TOO_SHORT;
    if (!(cfg.amin > 0.f)) return LM_ERR_INVALID_ARG;
    // The kernel keeps half of the window and fuses it with the first butterfly through w[n + N/2] = 1 - w[n], which
    // holds for the periodic Hann window of the reference (torch.hann_window, TA/transforms/_transforms.py:86-87) and
    // for nothing else in common use: refuse other windows instead of computing wrong spectra.
    for (int n = 0; n < cfg.n_fft / 2; ++n)
        if (!(fabsf(cfg.window[n] + cfg.window[n + cfg.n_fft / 2] - 1.0f) <= 2e-6f)) return LM_ERR_UNSUPPORTED;
    return LM_OK;
}

int check_device(int device, cudaDeviceProp* prop) {
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || device < 0 || device >= n_dev) {
        cudaGetLastError();
        return LM_ERR_NO_DEVICE;
    }
    LM_CUDA(cudaGetDeviceProperties(prop, device));
    if (prop->major != 10) return LM_ERR_NO_DEVICE;   // the fatbin holds sm_100a code only
    return LM_OK;
}

// Banded filterbank as mma.sync A fragments (scaled by 1/4: the kernel produces 4 |X|^2).
// Mel tile mt = filters [8mt, 8mt+8).  Its band starts at kb (first non-zero bin, rounded down to
// 4) and is walked in steps of 16 bins = two MMA k-steps.  For step d and k-step s, lane
// (g = lane/4, tg = lane%4) holds one float4 = the A fragment (a0, a1, a2, a3) =
// (head w0, residual w0, head w1, residual w1) with w_j = fb[kb + 16d + 4tg + 2s + j][8mt + g]:
// MMA rows 0-7 carry the TF32 head (low 13 mantissa bits cleared), rows 8-15 the residual w - head
// (13 significant bits, of which the tensor core keeps 11), and the k-permutation matches the
// kernel's LDS.128 loads of the power rows.  Fills the bands of `tab` (kb, ndk, off), `melw` and the
// filterbank's non-zero count.
int pack_filterbank(const lm_config& cfg, int row_cap, lm::MelTable* tab, std::vector<float4>* melw, int* nnz) {
    const int n_freqs = cfg.n_fft / 2 + 1, n_mels = cfg.n_mels, n_mt = (n_mels + 7) / 8;
    *nnz = 0;
    for (int k = 0; k < n_freqs; ++k)
        for (int m = 0; m < n_mels; ++m) *nnz += cfg.fb[static_cast<size_t>(k) * n_mels + m] != 0.0f;
    auto fbv = [&](int k, int m) -> float {
        return (k < n_freqs && m < n_mels) ? 0.25f * cfg.fb[static_cast<size_t>(k) * n_mels + m] : 0.0f;
    };
    auto head = [](float w) -> float {
        uint32_t u;
        memcpy(&u, &w, 4);
        u &= 0xffffe000u;
        float h;
        memcpy(&h, &u, 4);
        return h;
    };
    // bins past n_freqs that a padded band reads hold finite values (zeros, the next frame's spectrum, FFT scratch)
    // and meet zero weights
    for (int mt = 0; mt < n_mt; ++mt) {
        int lo = -1, hi = -1;
        for (int k = 0; k < n_freqs; ++k)
            for (int g = 0; g < 8; ++g)
                if (fbv(k, 8 * mt + g) != 0.0f) { if (lo < 0) lo = k; hi = k; }
        int kb = 0, ndk = 0;
        if (lo >= 0) { kb = lo & ~3; ndk = (hi + 1 - kb + 15) / 16; }
        while (ndk > 0 && kb > 0 && kb + 16 * ndk > row_cap) kb -= 4;   // keep the padded band inside the row
        if (kb + 16 * ndk > row_cap) return LM_ERR_FILTERBANK;
        tab->kb[mt] = kb; tab->ndk[mt] = ndk; tab->off[mt] = static_cast<int>(melw->size() / 64);
        for (int d = 0; d < ndk; ++d)
            for (int s = 0; s < 2; ++s)
                for (int lane = 0; lane < 32; ++lane) {
                    const int g = lane >> 2, tg = lane & 3, k0 = kb + 16 * d + 4 * tg + 2 * s, m = 8 * mt + g;
                    const float w0 = fbv(k0, m), w1 = fbv(k0 + 1, m);
                    melw->push_back(make_float4(head(w0), w0 - head(w0), head(w1), w1 - head(w1)));
                }
    }
    if (melw->empty()) melw->assign(64, make_float4(0.f, 0.f, 0.f, 0.f));
    return melw->size() / 64 > static_cast<size_t>(lm::kMaxDk) ? LM_ERR_FILTERBANK : LM_OK;
}

// Longest-processing-time assignment of the n_mt mel tiles of `tab` to the 8 warps of a group (both groups use the
// same table); warps 2s and 2s+1... of one scheduler are warp % 4, balanced too.
void assign_mel_tiles(int n_mt, lm::MelTable* tab) {
    for (auto& w : tab->warp_tile)
        for (int& t : w) t = -1;
    std::vector<int> order(n_mt);
    for (int i = 0; i < n_mt; ++i) order[i] = i;
    std::sort(order.begin(), order.end(), [&](int a, int b) { return tab->ndk[a] > tab->ndk[b]; });
    int load_w[lm::kGroupWarps] = {0}, load_s[4] = {0, 0, 0, 0}, cnt_w[lm::kGroupWarps] = {0};
    for (int mt : order) {
        int best = -1;
        for (int w = 0; w < lm::kGroupWarps; ++w) {
            if (cnt_w[w] >= lm::kTileSlots) continue;
            if (best < 0) { best = w; continue; }
            const int a = load_w[w] * 64 + load_s[w & 3];
            const int b = load_w[best] * 64 + load_s[best & 3];
            // lightest warp first, then lightest scheduler
            if (a < b) best = w;
        }
        tab->warp_tile[best][cnt_w[best]++] = mt;
        load_w[best] += tab->ndk[mt] + 4;      // a tile's fixed cost (setup + epilogue) is worth ~4 steps
        load_s[best & 3] += tab->ndk[mt] + 4;
    }
}

constexpr double kTwoPi = 6.283185307179586476925286766559;

// W_nc^(k1 n2) between the two FFT stages (warp_twiddle): nc points per complex FFT, lane = s * (nc / 32) + n2
// carries point n2 of sub-FFT s.  Rows k1 = 1, 2, 3, 4, 8, ..., 28; the kernel forms the others as products.
std::vector<float2> fft_twiddles(int nc) {
    std::vector<float2> tw(32 * lm::kTwRows);
    for (int r = 0; r < lm::kTwRows; ++r) {
        const int k1 = r < 3 ? r + 1 : 4 * (r - 2);
        for (int lane = 0; lane < 32; ++lane) {
            const int n2 = lane % (nc / 32);
            const double a = kTwoPi * static_cast<double>(k1 * n2) / static_cast<double>(nc);
            tw[r * 32 + lane] = make_float2(static_cast<float>(cos(a)), static_cast<float>(-sin(a)));
        }
    }
    return tw;
}

// (cos, sin)(2 pi k / 2048), k < 512: the real-FFT untangle at n_fft = 2048
std::vector<float2> untangle_twiddles() {
    std::vector<float2> utw(512);
    for (int k = 0; k < 512; ++k) {
        const double a = kTwoPi * static_cast<double>(k) / 2048.0;
        utw[k] = make_float2(static_cast<float>(cos(a)), static_cast<float>(sin(a)));
    }
    return utw;
}

// The plan's constant tables to the device, and its scheduling counters and small-batch scratch, zeroed.
int upload_tables(lm_plan* p, const float* window, const std::vector<float2>& tw, const std::vector<float2>& utw,
                  const std::vector<float4>& melw, const lm::MelTable& tab) {
    auto up = [&](void** dst, const void* src, size_t bytes) -> int {
        LM_CUDA(cudaMalloc(dst, bytes));
        LM_CUDA(cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice));
        return LM_OK;
    };
    int rc = LM_OK;
    if ((rc = up(reinterpret_cast<void**>(&p->d_window), window, sizeof(float) * p->n_fft)) ||
        (rc = up(reinterpret_cast<void**>(&p->d_tw), tw.data(), sizeof(float2) * tw.size())) ||
        (rc = up(reinterpret_cast<void**>(&p->d_utw), utw.data(), sizeof(float2) * utw.size())) ||
        (rc = up(reinterpret_cast<void**>(&p->d_melw), melw.data(), sizeof(float4) * melw.size())) ||
        (rc = up(reinterpret_cast<void**>(&p->d_tab), &tab, sizeof(tab))))
        return rc;
    LM_CUDA(cudaMalloc(&p->d_counters, sizeof(int) * 2 * kCounters));
    LM_CUDA(cudaMemset(p->d_counters, 0, sizeof(int) * 2 * kCounters));
    LM_CUDA(cudaMalloc(&p->d_split, static_cast<size_t>(kCounters) * kMaxSplitClips * 20));
    LM_CUDA(cudaMemset(p->d_split, 0, static_cast<size_t>(kCounters) * kMaxSplitClips * 20));
    return LM_OK;
}

// lm_forward_host and lm_forward_host_pcm16: `wave` holds fp32 samples, or 16-bit PCM when pcm16.
int forward_host_impl(lm_plan* plan, const void* wave, bool pcm16, int64_t total_samples, const int64_t* offset,
                      const int32_t* length, int32_t B, const lm_aug* aug, const float* noise, float* out, int32_t normalize) {
    if (!plan || B < 0 || total_samples < 0) return LM_ERR_INVALID_ARG;
    if (B == 0) return LM_OK;
    if (!wave || !offset || !length || !out) return LM_ERR_INVALID_ARG;
    for (int i = 0; i < B; ++i)
        if (length[i] < 0 || offset[i] < 0 || offset[i] + length[i] > total_samples) return LM_ERR_INVALID_ARG;
    NvtxRange nvtx(pcm16 ? "lm_forward_host_pcm16" : "lm_forward_host");
    std::lock_guard<std::mutex> one_caller(plan->host_mu);   // the staging slots belong to the plan
    DeviceOf on(plan->device);
    if (on.err) return cuda_fail(on.err, "cudaSetDevice");
    int rc = ensure_slots(plan);
    if (rc) return rc;

    const size_t clip_elems = static_cast<size_t>(plan->n_mels) * plan->frames;
    const size_t sample_bytes = pcm16 ? sizeof(int16_t) : sizeof(float);
    // chunk so that a few chunks are in flight: ~64 MB of waveform, at least 2 SM-waves of clips
    const int auto_chunk = std::max(2 * plan->sm_count, static_cast<int>((64u << 20) / (4u * static_cast<size_t>(plan->T))));
    const int chunk = std::max(1, std::min<int>(B, plan->host_chunk_clips > 0 ? plan->host_chunk_clips : auto_chunk));
    int slot_i = 0;
    for (int c0 = 0; c0 < B && rc == LM_OK; c0 += chunk, slot_i = (slot_i + 1) % kSlots) {
        const int n = std::min(chunk, B - c0);
        HostSlot& s = plan->slots[slot_i];
        if ((rc = cudaStreamSynchronize(s.stream) == cudaSuccess ? LM_OK : cuda_fail(cudaGetLastError(), "slot sync"))) break;
        int64_t lo = INT64_MAX, hi = 0;
        for (int i = c0; i < c0 + n; ++i) {
            if (length[i] == 0) continue;
            lo = std::min(lo, offset[i]);
            hi = std::max(hi, offset[i] + length[i]);
        }
        if (lo == INT64_MAX) { lo = 0; hi = 0; }
        lo &= ~int64_t(7);   // keep 16-byte alignment of clip starts (TMA staging path; 8 PCM samples per int4)
        const size_t n_wave = static_cast<size_t>(hi - lo);
        constexpr size_t kMetaPerClip = sizeof(long long) + sizeof(lm_aug) + sizeof(int);
        if (n > s.cap_clips) {
            cudaFree(s.d_meta);
            if (s.h_meta) cudaFreeHost(s.h_meta);
            s.d_meta = nullptr; s.h_meta = nullptr; s.cap_clips = 0;
            if (cudaMalloc(&s.d_meta, kMetaPerClip * n) != cudaSuccess || cudaMallocHost(&s.h_meta, kMetaPerClip * n) != cudaSuccess) {
                rc = cuda_fail(cudaGetLastError(), "slot metadata alloc");
                break;
            }
            s.cap_clips = n;
        }
        // the blocks are laid out for the slot's capacity so that the three arrays keep their alignment
        const size_t cap = static_cast<size_t>(s.cap_clips);
        long long* h_off = reinterpret_cast<long long*>(s.h_meta);
        lm_aug* h_aug = reinterpret_cast<lm_aug*>(s.h_meta + sizeof(long long) * cap);
        int* h_len = reinterpret_cast<int*>(s.h_meta + (sizeof(long long) + sizeof(lm_aug)) * cap);
        const long long* d_off = reinterpret_cast<const long long*>(s.d_meta);
        const lm_aug* d_aug = reinterpret_cast<const lm_aug*>(s.d_meta + sizeof(long long) * cap);
        const int* d_len = reinterpret_cast<const int*>(s.d_meta + (sizeof(long long) + sizeof(lm_aug)) * cap);
        if ((rc = grow(&s.d_wave, &s.cap_wave, sample_bytes * std::max<size_t>(n_wave + 8, 16)))) break;
        if ((rc = grow(&s.d_out, &s.cap_out, clip_elems * n))) break;
        if (noise && (rc = grow(&s.d_noise, &s.cap_noise, static_cast<size_t>(plan->T) * n))) break;
        for (int i = 0; i < n; ++i) h_off[i] = length[c0 + i] ? offset[c0 + i] - lo : 0;
        memcpy(h_len, length + c0, sizeof(int) * n);
        if (aug) memcpy(h_aug, aug + c0, sizeof(lm_aug) * n);

        cudaError_t e = cudaMemcpyAsync(s.d_meta, s.h_meta, kMetaPerClip * cap, cudaMemcpyHostToDevice, s.stream);
        if (e != cudaSuccess) { rc = cuda_fail(e, "H2D copy (metadata)"); break; }
        if (n_wave)
            e = cudaMemcpyAsync(s.d_wave, static_cast<const unsigned char*>(wave) + sample_bytes * lo, sample_bytes * n_wave,
                                cudaMemcpyHostToDevice, s.stream);
        if (e == cudaSuccess && noise)
            e = cudaMemcpyAsync(s.d_noise, noise + static_cast<size_t>(c0) * plan->T, sizeof(float) * plan->T * n,
                                cudaMemcpyHostToDevice, s.stream);
        if (e != cudaSuccess) { rc = cuda_fail(e, "H2D copy"); break; }
        rc = launch(plan, {s.d_wave, pcm16, reinterpret_cast<const int64_t*>(d_off), d_len, n, aug ? d_aug : nullptr,
                           noise ? s.d_noise : nullptr}, {s.d_out}, normalize, s.stream);
        if (rc) break;
        e = cudaMemcpyAsync(out + clip_elems * c0, s.d_out, sizeof(float) * clip_elems * n, cudaMemcpyDeviceToHost, s.stream);
        if (e != cudaSuccess) { rc = cuda_fail(e, "D2H copy"); break; }
    }
    for (auto& s : plan->slots) {
        const cudaError_t e = cudaStreamSynchronize(s.stream);
        if (e != cudaSuccess && rc == LM_OK) rc = cuda_fail(e, "pipeline drain");
    }
    return rc;
}

// The polyphase taps of one rate pair and their geometry: rates divided by their gcd (o -> q), `width`, per phase the
// first kept tap k0 and 4 nt4 taps (the widest phase's ntaps, zero-padded to whole float4).  Host arithmetic only:
// lm_resampler_create uploads the tables, lm_clip_span derives the samples a clip's features read from view().
struct RsDesign {
    int o = 1, q = 1, width = 0, nt4 = 1;
    std::vector<float> taps4;   // [q][4 nt4]
    std::vector<int> k0;        // [q]
    lm::RsTaps view() const { return {nullptr, k0.data(), o, q, nt4, width}; }
};

RsDesign rs_design(int orig_freq, int new_freq) {
    RsDesign d;
    int a = orig_freq, b = new_freq;
    while (b) { const int t = a % b; a = b; b = t; }
    const int o = orig_freq / a, q = new_freq / a;
    // TA/functional/functional.py _get_sinc_resample_kernel with lowpass_filter_width = 6, rolloff = 0.99,
    // sinc_interp_hann, float64 index arithmetic, kernel rounded to float32 at the end
    const int lpw = 6;
    const double base_freq = std::min(o, q) * 0.99;
    const int width = static_cast<int>(ceil(lpw * o / base_freq));
    const int K = 2 * width + o;
    const double pi = 3.14159265358979323846;
    std::vector<float> dense(static_cast<size_t>(q) * K);
    for (int p = 0; p < q; ++p)
        for (int k = 0; k < K; ++k) {
            double t = (static_cast<double>(-p) / q + static_cast<double>(k - width) / o) * base_freq;
            t = std::min(std::max(t, -static_cast<double>(lpw)), static_cast<double>(lpw));
            const double c = cos(t * pi / lpw / 2.0);
            const double window = c * c;
            const double tp = t * pi;
            const double sinc = (tp == 0.0) ? 1.0 : sin(tp) / tp;
            dense[static_cast<size_t>(p) * K + k] = static_cast<float>(sinc * window * (base_freq / o));
        }
    // per phase keep the taps that are not negligible (|w| > 1e-12: the clamped tails are ~1e-33)
    int ntaps = 1;
    std::vector<int> k0(q);
    for (int p = 0; p < q; ++p) {
        int lo = K, hi = -1;
        for (int k = 0; k < K; ++k)
            if (fabsf(dense[static_cast<size_t>(p) * K + k]) > 1e-12f) { lo = std::min(lo, k); hi = k; }
        if (hi < 0) { lo = 0; hi = 0; }
        k0[p] = lo;
        ntaps = std::max(ntaps, hi - lo + 1);
    }
    const int row = 4 * ((ntaps + 3) / 4);
    std::vector<float> taps4(static_cast<size_t>(q) * row, 0.0f);
    for (int p = 0; p < q; ++p) {
        if (k0[p] + ntaps > K) k0[p] = std::max(0, K - ntaps);
        for (int i = 0; i < ntaps && k0[p] + i < K; ++i) taps4[static_cast<size_t>(p) * row + i] = dense[static_cast<size_t>(p) * K + k0[p] + i];
    }
    d.o = o; d.q = q; d.width = width; d.nt4 = row / 4;
    d.taps4 = std::move(taps4); d.k0 = std::move(k0);
    return d;
}

}  // namespace

extern "C" {

int lm_abi_version(void) { return LM_ABI_VERSION; }

const char* lm_strerror(int status) {
    switch (status) {
        case LM_OK: return "ok";
        case LM_ERR_INVALID_ARG: return "invalid argument";
        case LM_ERR_UNSUPPORTED: return "unsupported configuration (n_fft must be 256, 512, 1024 or 2048; hop even and <= n_fft/4; n_mels <= 256; window must be the periodic Hann window: w[n] + w[n + n_fft/2] = 1)";
        case LM_ERR_FILTERBANK: return "filterbank support too wide for the on-chip table";
        case LM_ERR_CUDA: return "CUDA runtime error (see lm_last_cuda_error)";
        case LM_ERR_NO_DEVICE: return "no usable CUDA device (an sm_100 GPU is required; there is no CPU fallback)";
        case LM_ERR_TOO_SHORT: return "target_len must exceed n_fft/2 (reflect padding)";
        default: return "unknown status";
    }
}

const char* lm_last_cuda_error(void) { return g_cuda_err; }

int lm_plan_create(const lm_config* cfg, int device, lm_plan** out_plan) {
    NvtxRange nvtx("lm_plan_create");
    if (!cfg || !out_plan || !cfg->window || !cfg->fb) return LM_ERR_INVALID_ARG;
    *out_plan = nullptr;
    int rc = validate_config(*cfg);
    cudaDeviceProp prop{};
    if (rc || (rc = check_device(device, &prop))) return rc;
    DeviceOf on(device);
    if (on.err) return cuda_fail(on.err, "cudaSetDevice");

    lm_plan* p = new (std::nothrow) lm_plan();
    if (!p) return LM_ERR_INVALID_ARG;
    auto fail = [p](int status) { free_plan(p); return status; };
    const Geometry geo = geometry(cfg->n_fft, cfg->hop);
    p->device = device;
    p->n_fft = cfg->n_fft; p->hop = cfg->hop; p->n_mels = cfg->n_mels; p->T = cfg->target_len;
    p->n_freqs = cfg->n_fft / 2 + 1;
    p->frames = 1 + cfg->target_len / cfg->hop;
    p->tile_f = geo.tile_f;
    p->n_tiles = (p->frames + p->tile_f - 1) / p->tile_f;
    p->ns = geo.ns;
    std::copy(std::begin(geo.kernels), std::end(geo.kernels), p->kernels);
    p->db_mult = cfg->db_multiplier; p->amin = cfg->amin; p->db_offset = cfg->db_offset;
    p->norm_eps = cfg->norm_eps;
    p->floor_db = cfg->db_multiplier * log10f(cfg->amin) - cfg->db_offset;
    p->sm_count = prop.multiProcessorCount;

    lm::MelTable tab{};
    std::vector<float4> melw;
    if ((rc = pack_filterbank(*cfg, geo.row_cap, &tab, &melw, &p->fb_nnz))) return fail(rc);
    assign_mel_tiles((cfg->n_mels + 7) / 8, &tab);
    p->n_dk = static_cast<int>(melw.size() / 64);
    if ((rc = upload_tables(p, cfg->window, fft_twiddles(geo.nc), untangle_twiddles(), melw, tab))) return fail(rc);

    p->smem_bytes = geo.smem_total(p->ns, p->n_dk);
    if (p->smem_bytes > prop.sharedMemPerBlockOptin) return fail(LM_ERR_FILTERBANK);
    const cudaError_t e = set_smem_limit(p->kernels, device, p->smem_bytes);
    if (e != cudaSuccess) return fail(cuda_fail(e, "cudaFuncSetAttribute(MaxDynamicSharedMemorySize)"));
    *out_plan = p;
    return LM_OK;
}

int lm_plan_destroy(lm_plan* plan) { return free_plan(plan); }

#if LM_TIMING
// debug builds only (tools/build_variants.py "timing"): per-warp phase cycle counters of the last launch
int lm_debug_timing(long long* host_out, int n) {
    cudaDeviceSynchronize();
    return cudaMemcpyFromSymbol(host_out, lm::g_timing, sizeof(long long) * n) == cudaSuccess ? LM_OK : LM_ERR_CUDA;
}
#endif

int lm_plan_frames(const lm_plan* plan) { return plan ? plan->frames : LM_ERR_INVALID_ARG; }

int lm_plan_info(const lm_plan* plan, lm_info* info) {
    if (!plan || !info) return LM_ERR_INVALID_ARG;
    info->abi_version = LM_ABI_VERSION;
    info->frames = plan->frames;
    info->n_freqs = plan->n_freqs;
    info->sm_count = plan->max_ctas > 0 ? plan->max_ctas : plan->sm_count;
    info->threads_per_cta = lm::kThreads;
    info->smem_bytes = static_cast<int32_t>(plan->smem_bytes);
    info->fb_nnz = plan->fb_nnz;
    info->tma_staging = plan->use_tma;
    info->bytes_per_clip = 4LL * plan->T + 4LL * plan->n_mels * plan->frames;
    return LM_OK;
}

int lm_plan_set(lm_plan* plan, const char* key, int value) {
    if (!plan || !key) return LM_ERR_INVALID_ARG;
    if (!strcmp(key, "tma")) { plan->use_tma = value ? 1 : 0; return LM_OK; }
    if (!strcmp(key, "host_chunk_clips")) { if (value < 0) return LM_ERR_INVALID_ARG; plan->host_chunk_clips = value; return LM_OK; }
    if (!strcmp(key, "stagger_ns")) { if (value < 0) return LM_ERR_INVALID_ARG; plan->stagger_ns = value; return LM_OK; }
    if (!strcmp(key, "max_ctas")) { if (value < 0) return LM_ERR_INVALID_ARG; plan->max_ctas = value; return LM_OK; }
    if (!strcmp(key, "split")) { if (value < 0) return LM_ERR_INVALID_ARG; plan->split_override = value; return LM_OK; }
    return LM_ERR_INVALID_ARG;
}

int64_t lm_plan_launch_count(const lm_plan* plan) { return plan ? plan->launches.load() : 0; }

int lm_forward(lm_plan* plan, const float* wave, const int64_t* offset, const int32_t* length, int32_t B,
               const lm_aug* aug, const float* noise, float* out_norm, float* out_db, float* out_melpow,
               int32_t normalize, void* cuda_stream) {
    return forward_on_device("lm_forward", Call::Plain, plan, {wave, 0, offset, length, B, aug, noise},
                             {out_norm, out_db, out_melpow}, normalize, cuda_stream);
}

int lm_forward_pcm16(lm_plan* plan, const int16_t* pcm, const int64_t* offset, const int32_t* length, int32_t B,
                     const lm_aug* aug, const float* noise, float* out_norm, int32_t normalize, void* cuda_stream) {
    return forward_on_device("lm_forward_pcm16", Call::Plain, plan, {pcm, 1, offset, length, B, aug, noise}, {out_norm},
                             normalize, cuda_stream);
}

int lm_forward_gather(lm_plan* plan, const float* wave, const int64_t* offset, const int32_t* length, int32_t B,
                      const lm_aug* aug, const float* noise, float* out_slice, float* const* peer_slices,
                      int32_t n_peers, float* mc_slice, void* cuda_stream) {
    return forward_on_device("lm_forward_gather", Call::Gather, plan, {wave, 0, offset, length, B, aug, noise},
                             {out_slice, nullptr, nullptr, peer_slices, n_peers, mc_slice}, 1, cuda_stream);
}

int lm_forward_resampled(lm_plan* plan, const lm_resampler* const* resamplers, int32_t n_resamplers, const void* wave,
                         int32_t pcm16, const int64_t* offset, const int32_t* length, const int32_t* source, int32_t B,
                         const lm_aug* aug, const float* noise, float* out_norm, int32_t normalize, void* cuda_stream) {
    return forward_on_device("lm_forward_resampled", Call::Resampled, plan,
                             {wave, pcm16, offset, length, B, aug, noise, source, resamplers, n_resamplers}, {out_norm},
                             normalize, cuda_stream);
}

int lm_clip_span(int32_t orig_freq, int32_t new_freq, int32_t target_len, int64_t length, int64_t* first, int64_t* count) {
    if (orig_freq < 1 || new_freq < 1 || target_len < 1 || length < 0 || !first || !count) return LM_ERR_INVALID_ARG;
    long long lo = 0, hi = 0;
    if (orig_freq == new_freq) {   // no resampling: the pad / centre-crop span
        lo = length > target_len ? (length - target_len) / 2 : 0;
        hi = lo + std::min<int64_t>(length, target_len);
    } else {
        // a worker asks once per item: keep each rate pair's design (per thread, so no lock is held across a fork)
        thread_local std::map<std::pair<int, int>, RsDesign> designs;
        auto it = designs.find(std::make_pair(orig_freq, new_freq));
        if (it == designs.end()) it = designs.emplace(std::make_pair(orig_freq, new_freq), rs_design(orig_freq, new_freq)).first;
        lm::rs_read_span(it->second.view(), length, target_len, &lo, &hi);
    }
    *first = lo;
    *count = hi - lo;
    return LM_OK;
}

int lm_forward_spans(lm_plan* plan, const lm_resampler* const* resamplers, int32_t n_resamplers, const void* wave,
                     int32_t pcm16, const int64_t* offset, const int64_t* first, const int32_t* stored,
                     const int32_t* length, const int32_t* source, int32_t B, const lm_aug* aug, const float* noise,
                     float* out_norm, int32_t normalize, void* cuda_stream) {
    return forward_on_device("lm_forward_spans", Call::Spans, plan,
                             {wave, pcm16, offset, length, B, aug, noise, source, resamplers, n_resamplers, first, stored},
                             {out_norm}, normalize, cuda_stream);
}

int lm_resize_finish(const float* in, int32_t B, int32_t n_mels, int32_t frames_in, int32_t frames_out,
                     const lm_aug* aug, float* out, int32_t normalize, float norm_eps, void* cuda_stream) {
    if (B < 0 || n_mels < 1 || frames_in < 1 || frames_out < 1) return LM_ERR_INVALID_ARG;
    if (B == 0) return LM_OK;
    if (!in || !out || in == out) return LM_ERR_INVALID_ARG;
    DeviceOf guard(out);
    lm::resize_finish_kernel<<<B, lm::kAuxThreads, 0, static_cast<cudaStream_t>(cuda_stream)>>>(
        in, out, aug, n_mels, frames_in, frames_out, normalize, norm_eps);
    LM_CUDA(cudaGetLastError());
    return LM_OK;
}

int lm_pcm16_roundtrip(const float* in, float* out, int64_t n, void* cuda_stream) {
    if (n < 0) return LM_ERR_INVALID_ARG;
    if (n == 0) return LM_OK;
    if (!in || !out) return LM_ERR_INVALID_ARG;
    DeviceOf guard(out);
    const int blocks = static_cast<int>(std::min<int64_t>((n + 1023) / 1024, 148 * 8));
    lm::pcm16_roundtrip_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(cuda_stream)>>>(in, out, n);
    LM_CUDA(cudaGetLastError());
    return LM_OK;
}

int lm_resampler_create(int32_t orig_freq, int32_t new_freq, int device, lm_resampler** out) {
    if (!out || orig_freq < 1 || new_freq < 1) return LM_ERR_INVALID_ARG;
    *out = nullptr;
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || device < 0 || device >= n_dev) {
        cudaGetLastError();
        return LM_ERR_NO_DEVICE;
    }
    DeviceOf on(device);
    if (on.err) return cuda_fail(on.err, "cudaSetDevice");
    const RsDesign d = rs_design(orig_freq, new_freq);
    lm_resampler* r = new (std::nothrow) lm_resampler();
    if (!r) return LM_ERR_INVALID_ARG;
    r->device = device;
    r->k0max = *std::max_element(d.k0.begin(), d.k0.end());
    {
        const size_t span = static_cast<size_t>((lm::kRsChunk + d.q - 1) / d.q + 1) * d.o + r->k0max + 4 * d.nt4 + 8;
        r->tile_smem = span * sizeof(float) <= 96 * 1024 ? span * sizeof(float) : 0;
        if (const char* e = getenv("LM_RESAMPLE_UNTILED")) { if (e[0] == '1') r->tile_smem = 0; }   // tests compare the two kernels
        if (r->tile_smem > 48 * 1024 &&
            cudaFuncSetAttribute(lm::resample_tiled_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(r->tile_smem)) != cudaSuccess) {
            cudaGetLastError();
            r->tile_smem = 0;
        }
    }
    float4* taps4 = nullptr;
    int* k0 = nullptr;
    if (cudaMalloc(&taps4, sizeof(float) * d.taps4.size()) != cudaSuccess ||
        cudaMalloc(&k0, sizeof(int) * d.q) != cudaSuccess ||
        cudaMemcpy(taps4, d.taps4.data(), sizeof(float) * d.taps4.size(), cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(k0, d.k0.data(), sizeof(int) * d.q, cudaMemcpyHostToDevice) != cudaSuccess) {
        const int rc = cuda_fail(cudaGetLastError(), "resampler tables");
        cudaFree(taps4); cudaFree(k0);
        delete r;
        return rc;
    }
    r->rs = {taps4, k0, d.o, d.q, d.nt4, d.width};
    *out = r;
    return LM_OK;
}

int lm_resampler_destroy(lm_resampler* r) {
    if (!r) return LM_OK;
    DeviceOf on(r->device);
    cudaFree(const_cast<float4*>(r->rs.taps4)); cudaFree(const_cast<int*>(r->rs.k0));
    delete r;
    return LM_OK;
}

int64_t lm_resampler_out_len(const lm_resampler* r, int64_t in_len) {
    if (!r || in_len < 0) return LM_ERR_INVALID_ARG;
    return (static_cast<int64_t>(r->rs.q) * in_len + r->rs.o - 1) / r->rs.o;   // ceil(new * len / orig)
}

int lm_resample_rows(const lm_resampler* r, const float* in, int64_t in_len, int64_t in_stride, int32_t n_rows,
                     float* out, int64_t out_stride, void* cuda_stream) {
    if (!r || in_len < 0 || n_rows < 0) return LM_ERR_INVALID_ARG;
    const int64_t n_out = lm_resampler_out_len(r, in_len);
    if (n_out == 0 || n_rows == 0) return LM_OK;
    if (!in || !out || in_stride < in_len || out_stride < n_out) return LM_ERR_INVALID_ARG;
    DeviceOf guard(out);
    const int threads = 256;
    const long long blocks = (n_out + threads - 1) / threads;
    if (blocks > 0x7fffffffLL) return LM_ERR_INVALID_ARG;
    for (int32_t r0 = 0; r0 < n_rows && r->tile_smem; r0 += 65535) {   // tiled: one input span per 1024 outputs
        const int32_t nr = std::min<int32_t>(65535, n_rows - r0);
        const long long tblocks = (n_out + lm::kRsChunk - 1) / lm::kRsChunk;
        lm::resample_tiled_kernel<<<dim3(static_cast<unsigned>(tblocks), static_cast<unsigned>(nr)), lm::kRsThreads, r->tile_smem,
                                    static_cast<cudaStream_t>(cuda_stream)>>>(
            in + static_cast<int64_t>(r0) * in_stride, in_len, in_stride, out + static_cast<int64_t>(r0) * out_stride, n_out,
            out_stride, r->rs, r->k0max);
    }
    for (int32_t r0 = 0; r0 < n_rows && !r->tile_smem; r0 += 65535) {   // grid.y limit
        const int32_t nr = std::min<int32_t>(65535, n_rows - r0);
        lm::resample_kernel<<<dim3(static_cast<unsigned>(blocks), static_cast<unsigned>(nr)), threads, 0,
                              static_cast<cudaStream_t>(cuda_stream)>>>(
            in + static_cast<int64_t>(r0) * in_stride, in_len, in_stride, out + static_cast<int64_t>(r0) * out_stride, n_out,
            out_stride, r->rs);
    }
    LM_CUDA(cudaGetLastError());
    return LM_OK;
}

int lm_resample(const lm_resampler* r, const float* in, int64_t in_len, float* out, void* cuda_stream) {
    return lm_resample_rows(r, in, in_len, in_len, 1, out, lm_resampler_out_len(r, in_len), cuda_stream);
}

int lm_amplitude_to_db(const float* in, float* out, int64_t n, float multiplier, float amin, float db_offset, void* cuda_stream) {
    if (n < 0 || !(amin > 0.f)) return LM_ERR_INVALID_ARG;
    if (n == 0) return LM_OK;
    if (!in || !out) return LM_ERR_INVALID_ARG;
    DeviceOf guard(out);
    const int blocks = static_cast<int>(std::min<int64_t>((n + 255) / 256, 148 * 8));
    lm::amplitude_to_db_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(cuda_stream)>>>(
        in, out, n, static_cast<float>(static_cast<double>(multiplier) * 0.30102999566398119521), amin, db_offset);
    LM_CUDA(cudaGetLastError());
    return LM_OK;
}

int lm_pcm16_decode(const int16_t* in, float* out, int64_t n, void* cuda_stream) {
    if (n < 0) return LM_ERR_INVALID_ARG;
    if (n == 0) return LM_OK;
    if (!in || !out || (reinterpret_cast<uintptr_t>(in) & 15u) || (reinterpret_cast<uintptr_t>(out) & 15u)) return LM_ERR_INVALID_ARG;
    DeviceOf guard(out);
    const int blocks = static_cast<int>(std::min<int64_t>((n / 8 + 255) / 256 + 1, 148 * 8));
    lm::pcm16_decode_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(cuda_stream)>>>(in, out, n);
    LM_CUDA(cudaGetLastError());
    return LM_OK;
}

int lm_forward_host(lm_plan* plan, const float* wave, int64_t total_samples, const int64_t* offset,
                    const int32_t* length, int32_t B, const lm_aug* aug, const float* noise, float* out,
                    int32_t normalize) {
    return forward_host_impl(plan, wave, false, total_samples, offset, length, B, aug, noise, out, normalize);
}

int lm_forward_host_pcm16(lm_plan* plan, const int16_t* pcm, int64_t total_samples, const int64_t* offset,
                          const int32_t* length, int32_t B, const lm_aug* aug, const float* noise, float* out,
                          int32_t normalize) {
    return forward_host_impl(plan, pcm, true, total_samples, offset, length, B, aug, noise, out, normalize);
}

}  // extern "C"
