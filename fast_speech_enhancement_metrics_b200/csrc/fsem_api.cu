// C ABI of libfsem_b200.so (see include/fsem.h): contexts, workspace planning, kernel launches,
// and the host-buffer entry points with copy/compute overlap.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <new>
#include <vector>

#include "fsem_common.cuh"
#include "fsem_pesq.cuh"
#include "fsem_stoi.cuh"
#include "fsem_lsd.cuh"
#include "fsem_sdr.cuh"
#include "fsem_sdr_tc.cuh"
#include "fsem_ingest.cuh"

using namespace fsem;

// ------------------------------------------------------------------------------------------------
namespace {

thread_local char g_err[512] = "";
std::atomic<int64_t> g_launches{0};

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define FSEM_CUDA(expr)                                                                          \
    do {                                                                                         \
        cudaError_t e__ = (expr);                                                                \
        if (e__ != cudaSuccess)                                                                  \
            return fail(FSEM_E_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__),   \
                        __FILE__, __LINE__);                                                     \
    } while (0)

#define FSEM_LAUNCHED()                                                                          \
    do {                                                                                         \
        g_launches.fetch_add(1, std::memory_order_relaxed);                                      \
        FSEM_CUDA(cudaGetLastError());                                                           \
    } while (0)

inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

// ---- optional per-kernel timing with CUDA events on the launching stream (bench.py only; not thread-safe)
enum KernelId {
    K_PESQ_FILTER = 0, K_PESQ_SPECTRUM, K_PESQ_BARK, K_STOI_RESAMPLE, K_STOI_ENERGY, K_STOI_COMPACT,
    K_STOI_TOB, K_STOI_SEGMENT, K_STOI_FINALIZE, K_PESQ_RESAMPLE, K_LSD_FRAMES, K_SDR_CORR, K_SDR_SOLVE, K_INGEST, K_STOI_MARGIN, K_COUNT
};
const char* const kKernelNames[K_COUNT] = {
    "pesq_filter_kernel", "pesq_spectrum_kernel", "pesq_bark_kernel", "stoi_resample_kernel", "stoi_energy_kernel",
    "stoi_compact_kernel", "stoi_tob_kernel", "stoi_segment_kernel", "stoi_finalize_kernel", "pesq_resample_kernel", "lsd_frames_kernel", "sdr_corr_kernel", "sdr_solve_kernel", "ingest_kernel", "stoi_margin_kernel"};
bool g_profile = false;
struct ProfRecord { int id; cudaEvent_t start, stop; };
std::vector<ProfRecord> g_prof_pending;
std::vector<cudaEvent_t> g_prof_pool;
double g_prof_ms[K_COUNT] = {0};
int64_t g_prof_launches[K_COUNT] = {0};

cudaEvent_t prof_event() {
    if (!g_prof_pool.empty()) { cudaEvent_t e = g_prof_pool.back(); g_prof_pool.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}
struct ProfScope {
    int id; cudaStream_t stream; cudaEvent_t start = nullptr;
    ProfScope(int id_, cudaStream_t s) : id(id_), stream(s) {
        if (g_profile) { start = prof_event(); cudaEventRecord(start, stream); }
    }
    ~ProfScope() {
        if (start) { cudaEvent_t stop = prof_event(); cudaEventRecord(stop, stream); g_prof_pending.push_back({id, start, stop}); }
    }
};
void prof_collect() {
    for (auto& r : g_prof_pending) {
        float ms = 0.f;
        if (cudaEventSynchronize(r.stop) == cudaSuccess && cudaEventElapsedTime(&ms, r.start, r.stop) == cudaSuccess) {
            g_prof_ms[r.id] += ms;
            g_prof_launches[r.id] += 1;
        }
        g_prof_pool.push_back(r.start);
        g_prof_pool.push_back(r.stop);
    }
    g_prof_pending.clear();
}

struct DeviceInfo {
    int device = -1;
    int sms = 0;
};

int query_device(DeviceInfo& d) {
    FSEM_CUDA(cudaGetDevice(&d.device));
    FSEM_CUDA(cudaDeviceGetAttribute(&d.sms, cudaDevAttrMultiProcessorCount, d.device));
    return FSEM_OK;
}

// Double-buffered device staging for the host entry points.
struct HostPipe {
    cudaStream_t copy = nullptr, compute = nullptr;
    cudaEvent_t copied[2] = {nullptr, nullptr}, done[2] = {nullptr, nullptr};
    void* in[2] = {nullptr, nullptr};     // clean | deg | lengths of one chunk
    size_t in_bytes = 0;
    void* ws = nullptr;
    size_t ws_bytes = 0;
    void* out = nullptr;                  // device score columns for the WHOLE batch (one D2H at the end)
    size_t out_bytes = 0;

    HostPipe() = default;
    HostPipe(const HostPipe&) = delete;
    HostPipe& operator=(const HostPipe&) = delete;
    ~HostPipe() {
        for (int i = 0; i < 2; ++i) {
            if (in[i]) cudaFree(in[i]);
            if (copied[i]) cudaEventDestroy(copied[i]);
            if (done[i]) cudaEventDestroy(done[i]);
        }
        if (ws) cudaFree(ws);
        if (out) cudaFree(out);
        if (copy) cudaStreamDestroy(copy);
        if (compute) cudaStreamDestroy(compute);
    }

    int init() {
        if (copy) return FSEM_OK;
        FSEM_CUDA(cudaStreamCreateWithFlags(&copy, cudaStreamNonBlocking));
        FSEM_CUDA(cudaStreamCreateWithFlags(&compute, cudaStreamNonBlocking));
        for (int i = 0; i < 2; ++i) {
            FSEM_CUDA(cudaEventCreateWithFlags(&copied[i], cudaEventDisableTiming));
            FSEM_CUDA(cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming));
        }
        return FSEM_OK;
    }
    int reserve(size_t in_b, size_t ws_b, size_t out_b) {
        if (in_b > in_bytes) {
            for (int i = 0; i < 2; ++i) {
                if (in[i]) cudaFree(in[i]);
                in[i] = nullptr;
                FSEM_CUDA(cudaMalloc(&in[i], in_b));
            }
            in_bytes = in_b;
        }
        if (ws_b > ws_bytes) {
            if (ws) cudaFree(ws);
            ws = nullptr;
            FSEM_CUDA(cudaMalloc(&ws, ws_b));
            ws_bytes = ws_b;
        }
        if (out_b > out_bytes) {
            if (out) cudaFree(out);
            out = nullptr;
            FSEM_CUDA(cudaMalloc(&out, out_b));
            out_bytes = out_b;
        }
        return FSEM_OK;
    }
};

// items per chunk of the host pipeline: ~128 MB of input per chunk (in the dtype that crosses PCIe), at least 1 item
int64_t host_chunk_items(int64_t batch, int64_t n, size_t es) {
    const int64_t bytes_per_item = 2 * n * (int64_t)es;
    int64_t items = (int64_t(128) << 20) / (bytes_per_item > 0 ? bytes_per_item : 1);
    if (items < 1) items = 1;
    if (items > batch) items = batch;
    return items;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
// rows of `es`-byte samples that the kernels may read four samples at a time
bool rows_vec4(const void* a, const void* b, int64_t stride, size_t es) {
    const uintptr_t m = 4 * es - 1;
    return (reinterpret_cast<uintptr_t>(a) & m) == 0 && (reinterpret_cast<uintptr_t>(b) & m) == 0 && stride % 4 == 0;
}
size_t dtype_size(int dtype) {
    return dtype == FSEM_DTYPE_F32 ? sizeof(float) : (dtype == FSEM_DTYPE_I16 || dtype == FSEM_DTYPE_F16) ? 2 : 0;
}
// run `fn(T{})` with T = the sample type of `dtype`
int launch_ingest(const void* src, int dtype, int64_t rows, int64_t n, int64_t sstride, float* dst, int64_t dstride,
                  cudaStream_t stream);

template <typename F>
int dispatch_dtype(int dtype, F&& fn) {
    switch (dtype) {
        case FSEM_DTYPE_F32: return fn(float{});
        case FSEM_DTYPE_I16: return fn(int16_t{});
        case FSEM_DTYPE_F16: return fn(__half{});
        default: return FSEM_E_INVALID;
    }
}

// Checks of a batch of (clean, deg) row pairs, in the one order every entry point uses.  Returns FSEM_E_INVALID (the
// message names `who`), kEmptyBatch for a valid empty batch, or FSEM_OK.  [n_min, n_max]: the signal lengths the entry
// point takes.  With `n_checked_when_empty` an empty batch needs a valid n too (LSD, SDR, the resampler); otherwise an
// empty batch is accepted whatever its n (PESQ, STOI, the host pipeline).
constexpr int kEmptyBatch = 1;
constexpr int64_t kMaxN = (int64_t(1) << 30) - 1;      // sample indices of the device kernels stay below 2^30
int check_batch(const char* who, const void* clean, const void* deg, int64_t batch, int64_t n, int64_t stride,
                int64_t n_min, int64_t n_max, bool n_checked_when_empty) {
    const bool n_ok = n >= n_min && n <= n_max;
    if (batch < 0 || n < 0 || stride < n || (n_checked_when_empty && !n_ok))
        return fail(FSEM_E_INVALID, "%s: bad shape batch=%lld n=%lld stride=%lld", who, (long long)batch, (long long)n,
                    (long long)stride);
    if (batch == 0) return kEmptyBatch;
    if (!clean || !deg) return fail(FSEM_E_INVALID, "%s: null input", who);
    if (!n_ok)
        return fail(FSEM_E_INVALID, "%s: n=%lld outside [%lld, %lld]", who, (long long)n, (long long)n_min,
                    (long long)n_max);
    return FSEM_OK;
}

// The general polyphase resampler (stoi_resample_kernel): rates divided by their gcd, kernel half-width, the taps
// [neu][ntaps] and their device copy.  PESQ's resample-on-ingest, STOI's general path and fsem_resampler_t use it.
struct Resampler {
    int orig = 1, neu = 1, width = 0, ntaps = 0;
    float* d_taps = nullptr;

    Resampler() = default;
    Resampler(const Resampler&) = delete;
    Resampler& operator=(const Resampler&) = delete;
    ~Resampler() { if (d_taps) cudaFree(d_taps); }

    // the design rule of the kernel; makes no CUDA call
    static int check(const char* who, int orig, int neu, int width, int ntaps, const float* taps) {
        if (orig <= 0 || neu <= 0 || width < 0 || !taps || ntaps != 2 * width + orig)
            return fail(FSEM_E_INVALID, "%s: bad resampling kernel (ntaps must be 2*width+orig)", who);
        return FSEM_OK;
    }
    // keeps a design that passed check() and copies its taps to the device
    int upload(int orig_, int neu_, int width_, int ntaps_, const float* taps) {
        orig = orig_; neu = neu_; width = width_; ntaps = ntaps_;
        FSEM_CUDA(cudaMalloc(&d_taps, sizeof(float) * neu * ntaps));
        FSEM_CUDA(cudaMemcpy(d_taps, taps, sizeof(float) * neu * ntaps, cudaMemcpyHostToDevice));
        return FSEM_OK;
    }
    // clean and deg rows of `dtype` -> fp32 rows [2, batch, out_stride] (clean rows, then deg rows); with per-item
    // lengths and a non-null `lengths_out`, also the resampled lengths
    int launch(const char* who, KernelId id, const fsem_batch_t* in, int dtype, float* out, int64_t out_stride,
               int32_t* lengths_out, cudaStream_t stream) const {
        const int64_t bps = ceil_div(stoi_resampled_len(in->n, orig, neu), 256);
        if (bps * 2 * in->batch >= (int64_t(1) << 31))
            return fail(FSEM_E_INVALID, "%s: batch x samples too large for one launch; split the batch", who);
        { ProfScope prof_(id, stream);
          dispatch_dtype(dtype, [&](auto tag) {
              using T = decltype(tag);
              stoi_resample_kernel<T><<<(unsigned)(bps * 2 * in->batch), 256, 0, stream>>>(
                  reinterpret_cast<const T*>(in->clean), reinterpret_cast<const T*>(in->deg), in->lengths, in->batch,
                  in->n, in->stride, d_taps, orig, neu, width, ntaps, out, out_stride, (int)bps);
              return FSEM_OK;
          }); }
        FSEM_LAUNCHED();
        if (in->lengths && lengths_out) {
            resampled_lengths_kernel<<<(unsigned)ceil_div(in->batch, 256), 256, 0, stream>>>(
                in->lengths, in->batch, in->n, orig, neu, lengths_out);
            FSEM_LAUNCHED();
        }
        return FSEM_OK;
    }
};

}  // namespace

// ------------------------------------------------------------------------------------------------
extern "C" int fsem_version(void) { return FSEM_VERSION; }
extern "C" const char* fsem_last_error(void) { return g_err; }
extern "C" int64_t fsem_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
extern "C" int fsem_profile_enable(int on) { g_profile = on != 0; return FSEM_OK; }
extern "C" int fsem_profile_reset(void) {
    prof_collect();
    for (int i = 0; i < K_COUNT; ++i) { g_prof_ms[i] = 0; g_prof_launches[i] = 0; }
    return FSEM_OK;
}
extern "C" int fsem_profile_read(int index, const char** name, double* total_ms, int64_t* launches) {
    if (index < 0 || index >= K_COUNT) return FSEM_E_INVALID;
    prof_collect();
    if (name) *name = kKernelNames[index];
    if (total_ms) *total_ms = g_prof_ms[index];
    if (launches) *launches = g_prof_launches[index];
    return FSEM_OK;
}

// ================================================================================================
// PESQ
// ================================================================================================
struct fsem_pesq_ctx {
    DeviceInfo dev;
    PesqFilterCoef coef;
    int warm = 640;
    PesqTables* d_tab = nullptr;
    Resampler rs;                    // resample-on-ingest to 16 kHz (base.py:19-20); 1:1 when the input is 16 kHz
    int spec_ctas_per_sm = 2;
    int filt_ctas_per_sm = 4;
    // > 0: plan the IIR time-chunk grid as for a batch of this size (fsem_graph_create scores a batch in slices and
    // keeps the chunk grid -- the only batch-dependent arithmetic of either chain -- of the whole batch, so that sliced
    // and unsliced scoring agree bit for bit)
    int64_t plan_batch_hint = 0;
    HostPipe pipe;

    ~fsem_pesq_ctx() { if (d_tab) cudaFree(d_tab); }
};

namespace {

struct PesqPlan {
    int64_t batch, n, zstride;       // n = samples per item at 16 kHz (after resample-on-ingest)
    int64_t n_in, rstride;           // input samples per item; row pitch of the resampled signals
    bool resample;
    bool tiled;                      // lane = signal (tiled kernel) vs thread = (signal, chunk) for tiny batches
    int tmax, tpitch, chunk, nchunks;   // tpitch = round4(tmax): frame pitch of the Bark / disturbance rows (16-byte tiles)
    size_t off_rs, off_rslen, off_z, off_partial, off_bark, off_dist, off_power, off_order, off_fprefix, total;
};

PesqPlan pesq_plan(const fsem_pesq_ctx* ctx, int64_t batch, int64_t n_in) {
    constexpr int quantum = 64;                        // chunk granularity: owned tiles start on an even 32-sample slot
    PesqPlan p{};
    p.batch = batch;
    p.n_in = n_in;
    p.resample = ctx->rs.orig != ctx->rs.neu;
    const int64_t n = stoi_resampled_len(n_in, ctx->rs.orig, ctx->rs.neu);
    p.rstride = round_up(n > 0 ? n : 1, 4);
    p.n = n;
    // the spectrum kernel fetches whole 1 KB half-frames with bulk copies: the last frame ends at most 255 samples
    // (the n % 256 zero padding, PESQ.py:128-130) beyond n, so a pitch of n + 256 keeps every copy inside its own row
    p.zstride = round_up((n > 0 ? n : 1) + FSEM_PESQ_HOP, 4);
    p.tmax = pesq_num_frames(n);
    if (p.tmax < 1) p.tmax = 1;
    p.tpitch = (int)round_up(p.tmax, 4);
    // Chunking of the serial IIR pass.  A warp-unit = (32 signals, one chunk) and costs chunk + warm-up sample steps;
    // all units are equal, so the kernel runs in whole "waves" of resident warps.  Pick the chunk count that minimises
    // waves x (chunk + warm-up): enough units to fill the chip, no half-empty last wave, little redundant warm-up.
    const int64_t nn = n > 0 ? n : 1;
    const int64_t plan_batch = ctx->plan_batch_hint > 0 ? ctx->plan_batch_hint : batch;
    const int64_t groups = 2 * ceil_div(plan_batch > 0 ? plan_batch : 1, 32);
    const int64_t slots = (int64_t)ctx->dev.sms * ctx->filt_ctas_per_sm * kFiltWarps;   // resident warps of the IIR pass
    const int64_t max_ch = ceil_div(nn, 256) < 1024 ? ceil_div(nn, 256) : 1024;     // chunks of at least 256 samples
    int64_t nch = 1, chunk = round_up(nn, quantum);
    double best = 1e300;
    // tiny batches cannot fill the 32 signal lanes of a warp: there a thread takes one (signal, chunk) and the time
    // axis is cut as finely as the warm-up allows
    p.tiled = plan_batch >= 16;
    if (!p.tiled) {
        chunk = round_up(ceil_div(nn, max_ch), 64);
        nch = ceil_div(nn, chunk);
    }
    for (int64_t c = 1; p.tiled && c <= max_ch; ++c) {
        const int64_t ch = round_up(ceil_div(nn, c), quantum);
        const int64_t cc = ceil_div(nn, ch);
        const int64_t waves = ceil_div(groups * cc, slots);
        const double cost = (double)waves * (double)(ch + (cc > 1 ? ctx->warm : 0));
        if (cost < best * 0.999) { best = cost; nch = cc; chunk = ch; }
    }
    p.chunk = (int)chunk;
    p.nchunks = (int)nch;
    size_t off = 0;
    p.off_rs = off;      off = align256(off + (p.resample ? sizeof(float) * 2 * batch * p.rstride : 0));
    p.off_rslen = off;   off = align256(off + (p.resample ? sizeof(int32_t) * batch : 0));
    p.off_z = off;       off = align256(off + sizeof(float) * 2 * batch * p.zstride);
    p.off_bark = off;    off = align256(off + sizeof(float) * 2 * batch * p.tpitch * kBarkRow);
    p.off_dist = off;    off = align256(off + sizeof(float) * 2 * batch * p.tpitch);
    p.off_power = off;   off = align256(off + sizeof(double) * 2 * batch);
    p.off_order = off;   off = align256(off + sizeof(int32_t) * batch);              // variable-length batches only
    p.off_fprefix = off; off = align256(off + sizeof(int64_t) * (batch + 1));
    p.off_partial = off; off = align256(off + sizeof(double) * 2 * batch * p.nchunks);
    p.total = off;
    return p;
}

}  // namespace

extern "C" int fsem_pesq_create(fsem_pesq_ctx_t** out, const fsem_pesq_design_t* d) {
    if (!out || !d) return fail(FSEM_E_INVALID, "fsem_pesq_create: null argument");
    *out = nullptr;
    // the whole design is checked before the first CUDA call
    for (int k = 0; k < 15; ++k)
        if (fabsf(d->taper[k] - (float)(k + 1) * 0.0625f) > 1e-7f)
            return fail(FSEM_E_INVALID, "fsem_pesq_create: taper must be k/16 (PESQ.py:90)");
    PesqTables h{};
    memcpy(h.hann, d->hann, sizeof(h.hann));
    double wtot = 0.0;
    for (int b = 0; b < FSEM_PESQ_NBANDS; ++b) {
        h.band_first[b] = d->band_first_bin[b];
        h.band_count[b] = d->band_num_bins[b];
        const int expect_first = b == 0 ? 0 : h.band_first[b - 1] + h.band_count[b - 1];
        if (h.band_first[b] != expect_first || h.band_count[b] < 1 || h.band_count[b] > 32 ||
            h.band_first[b] + h.band_count[b] > 256)
            return fail(FSEM_E_INVALID, "fsem_pesq_create: Bark bands must tile bins 0..255 contiguously, at most 32 bins each (band %d)", b);
        {   // the spectrum kernel gathers a band from at most 1 (bands 0..31) / 4 (bands 32..48) earlier 8-bin groups
            const int span = ((h.band_first[b] + h.band_count[b] - 1) >> 3) - (h.band_first[b] >> 3);
            if (span > (b < 32 ? kBarkPiecesLow : kBarkPiecesHigh))
                return fail(FSEM_E_INVALID, "fsem_pesq_create: Bark band %d spans %d groups of 8 bins (unsupported layout)", b, span + 1);
        }
        h.pow_dens[b] = d->pow_dens[b];
        h.thresh[b] = d->thresh[b];
        h.zw_exp[b] = d->zwicker_exp[b];
        h.width[b] = d->width_bark[b];
        h.loud_scale[b] = (float)((double)d->sl * pow(2.0 * (double)d->thresh[b], (double)d->zwicker_exp[b]));
        if (b >= 1) wtot += (double)d->width_bark[b];
    }
    h.width_total = (float)wtot;
    const bool resample = d->rs_orig != d->rs_neu;
    int rc = resample ? Resampler::check("fsem_pesq_create", d->rs_orig, d->rs_neu, d->rs_width, d->rs_ntaps, d->rs_taps)
                      : FSEM_OK;
    if (rc != FSEM_OK) return rc;

    std::unique_ptr<fsem_pesq_ctx> ctx(new (std::nothrow) fsem_pesq_ctx());
    if (!ctx) return fail(FSEM_E_INVALID, "out of host memory");
    ctx->coef.k = d->bp_direct;
    for (int s = 0; s < FSEM_BP_SECTIONS; ++s) {
        ctx->coef.c0[s] = d->bp_c0[s]; ctx->coef.c1[s] = d->bp_c1[s];
        ctx->coef.a1[s] = d->bp_a1[s]; ctx->coef.a2[s] = d->bp_a2[s];
    }
    ctx->coef.pb0 = d->pre_b[0]; ctx->coef.pb1 = d->pre_b[1]; ctx->coef.pb2 = d->pre_b[2];
    ctx->coef.pa1 = d->pre_a[0]; ctx->coef.pa2 = d->pre_a[1];
    ctx->warm = (int)round_up(d->warmup > 0 ? d->warmup : 640, 32);
    if ((rc = query_device(ctx->dev)) != FSEM_OK) return rc;
    FSEM_CUDA(cudaMalloc(&ctx->d_tab, sizeof(PesqTables)));
    FSEM_CUDA(cudaMemcpy(ctx->d_tab, &h, sizeof(h), cudaMemcpyHostToDevice));
    if (resample && (rc = ctx->rs.upload(d->rs_orig, d->rs_neu, d->rs_width, d->rs_ntaps, d->rs_taps)) != FSEM_OK)
        return rc;
    FSEM_CUDA(cudaFuncSetAttribute(pesq_spectrum_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSpecDynSmem));
    FSEM_CUDA(cudaFuncSetAttribute(pesq_bark_kernel<kBarkThreadsWide, kBarkTileWide>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bark_dyn_smem(kBarkTileWide)));
    if (bark_dyn_smem(kBarkTile) > 0)
        FSEM_CUDA(cudaFuncSetAttribute(pesq_bark_kernel<kBarkThreads, kBarkTile>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bark_dyn_smem(kBarkTile)));
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pesq_spectrum_kernel, kSpecWarps * 32, kSpecDynSmem) == cudaSuccess && occ > 0)
        ctx->spec_ctas_per_sm = occ;
    occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pesq_filter_tiled_kernel<false, float>, kFiltWarps * 32, 0) == cudaSuccess && occ > 0)
        ctx->filt_ctas_per_sm = occ;
    *out = ctx.release();
    return FSEM_OK;
}

extern "C" int fsem_pesq_destroy(fsem_pesq_ctx_t* ctx) {
    delete ctx;
    return FSEM_OK;
}

extern "C" size_t fsem_pesq_workspace_bytes(const fsem_pesq_ctx_t* ctx, int64_t batch, int64_t n) {
    if (!ctx || batch <= 0 || n <= 0) return 0;
    return pesq_plan(ctx, batch, n).total;
}

extern "C" int fsem_pesq_score_f32(fsem_pesq_ctx_t* ctx, const fsem_batch_t* in, float* mos_out,
                                   int32_t* status_out, void* workspace, size_t workspace_bytes,
                                   void* stream_v) {
    return fsem_pesq_score(ctx, in, FSEM_DTYPE_F32, mos_out, status_out, workspace, workspace_bytes, stream_v);
}

// Any ingest dtype: the first kernel (IIR pass, or the resampler when the context resamples on ingest) reads the rows
// as they are; `in->clean` / `in->deg` point at rows of `dtype`, `in->stride` counts elements.
extern "C" int fsem_pesq_score(fsem_pesq_ctx_t* ctx, const fsem_batch_t* in, int dtype, float* mos_out,
                               int32_t* status_out, void* workspace, size_t workspace_bytes, void* stream_v) {
    if (!ctx || !in || !mos_out) return fail(FSEM_E_INVALID, "fsem_pesq_score: null argument");
    if (dtype_size(dtype) == 0) return fail(FSEM_E_INVALID, "fsem_pesq_score: unknown dtype %d", dtype);
    if (int rc = check_batch("fsem_pesq_score", in->clean, in->deg, in->batch, in->n, in->stride, 0, kMaxN, false))
        return rc == kEmptyBatch ? FSEM_OK : rc;
    const PesqPlan p = pesq_plan(ctx, in->batch, in->n);
    // without per-item lengths every item has n samples: fewer than 20 frames is the reference's
    // RuntimeError from unfold (PESQ.py:169)
    if (!in->lengths && pesq_num_frames(p.n) < 20)
        return fail(FSEM_E_TOO_SHORT, "PESQ needs at least 20 frames of 512/256 samples at 16 kHz; n=%lld gives %d",
                    (long long)in->n, pesq_num_frames(p.n));
    if (!workspace || workspace_bytes < p.total)
        return fail(FSEM_E_WORKSPACE, "fsem_pesq_score: workspace %zu < %zu bytes", workspace_bytes, p.total);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
    char* ws = static_cast<char*>(workspace);
    float* z = reinterpret_cast<float*>(ws + p.off_z);
    double* partial = reinterpret_cast<double*>(ws + p.off_partial);
    float* bark = reinterpret_cast<float*>(ws + p.off_bark);
    float* dist = reinterpret_cast<float*>(ws + p.off_dist);
    double* power = reinterpret_cast<double*>(ws + p.off_power);

    fsem_batch_t rs_batch;
    if (p.resample) {   // resample-on-ingest to 16 kHz (base.py:19-20), then the pipeline runs on the workspace copy
        float* y = reinterpret_cast<float*>(ws + p.off_rs);
        int32_t* rslen = reinterpret_cast<int32_t*>(ws + p.off_rslen);
        const int rc = ctx->rs.launch("fsem_pesq_score", K_PESQ_RESAMPLE, in, dtype, y, p.rstride, rslen, stream);
        if (rc != FSEM_OK) return rc;
        rs_batch = fsem_batch_t{y, y + in->batch * p.rstride, in->lengths ? rslen : nullptr, in->batch, p.n, p.rstride};
        in = &rs_batch;
        dtype = FSEM_DTYPE_F32;                                   // the rest of the chain reads the resampled fp32 rows
    }

    // variable-length batches: length-sorted item order (IIR warps of similar signals, longest Bark CTAs first) and
    // the prefix sum of valid frames (balanced spectrum warps)
    int32_t* order = nullptr;
    int64_t* fprefix = nullptr;
    if (in->lengths) {
        order = reinterpret_cast<int32_t*>(ws + p.off_order);
        fprefix = reinterpret_cast<int64_t*>(ws + p.off_fprefix);
        pesq_order_kernel<<<1, kOrderThreads, 0, stream>>>(in->lengths, in->batch, in->n, order, fprefix);
        FSEM_LAUNCHED();
    }
    {   // kernel A: reads the rows in their own dtype (float32, int16 PCM, fp16)
        const bool vec4 = rows_vec4(in->clean, in->deg, in->stride, dtype_size(dtype));
        ProfScope prof_(K_PESQ_FILTER, stream);
        dispatch_dtype(dtype, [&](auto tag) {
            using T = decltype(tag);
            const T* c = reinterpret_cast<const T*>(in->clean);
            const T* d = reinterpret_cast<const T*>(in->deg);
            if (vec4 && p.tiled) {
                const int64_t units = 2 * ceil_div(in->batch, 32) * p.nchunks;
                const unsigned grid = (unsigned)ceil_div(units, kFiltWarps);
                if (in->lengths)
                    pesq_filter_tiled_kernel<true, T><<<grid, kFiltWarps * 32, 0, stream>>>(
                        c, d, in->lengths, order, in->batch, in->n, in->stride, p.chunk, p.nchunks, ctx->warm, ctx->coef, z,
                        p.zstride, partial);
                else
                    pesq_filter_tiled_kernel<false, T><<<grid, kFiltWarps * 32, 0, stream>>>(
                        c, d, nullptr, nullptr, in->batch, in->n, in->stride, p.chunk, p.nchunks, ctx->warm, ctx->coef, z,
                        p.zstride, partial);
            } else {
                const int64_t threads = 2 * in->batch * p.nchunks;
                const unsigned grid = (unsigned)ceil_div(threads, 128);
                if (vec4)
                    pesq_filter_kernel<true, T><<<grid, 128, 0, stream>>>(
                        c, d, in->lengths, in->batch, in->n, in->stride, p.chunk, p.nchunks, ctx->warm, ctx->coef, z,
                        p.zstride, partial);
                else
                    pesq_filter_kernel<false, T><<<grid, 128, 0, stream>>>(
                        c, d, in->lengths, in->batch, in->n, in->stride, p.chunk, p.nchunks, ctx->warm, ctx->coef, z,
                        p.zstride, partial);
            }
            return FSEM_OK;
        });
    }
    FSEM_LAUNCHED();
    {   // kernel B
        const int64_t units = in->batch * (int64_t)p.tmax;
        int64_t grid = ceil_div(units, kSpecWarps);
        const int64_t cap = (int64_t)ctx->dev.sms * ctx->spec_ctas_per_sm;
        if (grid > cap) grid = cap;
        { ProfScope prof_(K_PESQ_SPECTRUM, stream);
          pesq_spectrum_kernel<<<(unsigned)grid, kSpecWarps * 32, kSpecDynSmem, stream>>>(
              z, p.zstride, in->lengths, fprefix, in->batch, in->n, p.tmax, p.tpitch, partial, p.nchunks, ctx->d_tab, bark); }
        FSEM_LAUNCHED();
    }
    {   // kernel C
        { ProfScope prof_(K_PESQ_BARK, stream);
          if (in->batch <= ctx->dev.sms)   // cannot fill the SMs anyway: one wide CTA per item, few serial tile rounds
              pesq_bark_kernel<kBarkThreadsWide, kBarkTileWide>
                  <<<(unsigned)in->batch, kBarkThreadsWide, bark_dyn_smem(kBarkTileWide), stream>>>(
                      bark, partial, p.nchunks, in->lengths, order, in->batch, in->n, p.tpitch, ctx->d_tab, dist, mos_out,
                      status_out, power);
          else
              pesq_bark_kernel<kBarkThreads, kBarkTile>
                  <<<(unsigned)in->batch, kBarkThreads, bark_dyn_smem(kBarkTile), stream>>>(
                      bark, partial, p.nchunks, in->lengths, order, in->batch, in->n, p.tpitch, ctx->d_tab, dist, mos_out,
                      status_out, power); }
        FSEM_LAUNCHED();
    }
    return FSEM_OK;
}

extern "C" int fsem_pesq_debug_taps(fsem_pesq_ctx_t* ctx, int64_t batch, int64_t n, const void* workspace,
                                    float* bark_out, double* power_out, int64_t* frames_out, void* stream_v) {
    if (!ctx || !workspace) return fail(FSEM_E_INVALID, "fsem_pesq_debug_taps: null argument");
    const PesqPlan p = pesq_plan(ctx, batch, n);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
    const char* ws = static_cast<const char*>(workspace);
    if (frames_out) *frames_out = p.tmax;
    if (bark_out)
        for (int64_t r = 0; r < 2 * batch; ++r)                  // rows of 49 valid floats at pitch kBarkRow, tpitch frames per item
            FSEM_CUDA(cudaMemcpy2DAsync(bark_out + r * p.tmax * FSEM_PESQ_NBANDS, sizeof(float) * FSEM_PESQ_NBANDS,
                                        ws + p.off_bark + sizeof(float) * r * p.tpitch * kBarkRow, sizeof(float) * kBarkRow,
                                        sizeof(float) * FSEM_PESQ_NBANDS, (size_t)p.tmax, cudaMemcpyDeviceToDevice, stream));
    if (power_out)
        FSEM_CUDA(cudaMemcpyAsync(power_out, ws + p.off_power, sizeof(double) * 2 * batch, cudaMemcpyDeviceToDevice,
                                  stream));
    return FSEM_OK;
}

// ================================================================================================
// STOI
// ================================================================================================
struct fsem_stoi_ctx {
    DeviceInfo dev;
    Resampler rs;               // input -> 10 kHz; its rates feed the frame kernels even when they are equal
    bool fast85 = false;        // taps fit the specialised 8:5 kernel
    Resample85Taps taps85;
    StoiTables* d_tab = nullptr;
    float clip = 0.f, dyn_range = 40.f;
    int tob_ctas_per_sm = 2;
    HostPipe pipe;

    ~fsem_stoi_ctx() { if (d_tab) cudaFree(d_tab); }
};

namespace {

struct StoiPlan {
    int64_t batch, n, lmax, ystride;
    int t0max, mask_words, umax, ustride, mmax, ntiles, hops_max;
    bool resample, fused_energy;
    size_t off_hops, off_y, off_energy, off_idx, off_count, off_prefix, off_mask, off_tob, off_partial, total;
};

StoiPlan stoi_plan(const fsem_stoi_ctx* ctx, int64_t batch, int64_t n) {
    StoiPlan p{};
    p.batch = batch;
    p.n = n;
    p.resample = ctx->rs.orig != ctx->rs.neu;
    p.lmax = stoi_resampled_len(n, ctx->rs.orig, ctx->rs.neu);
    p.ystride = round_up(p.lmax > 0 ? p.lmax : 1, 4);
    p.t0max = stoi_num_frames(p.lmax);
    if (p.t0max < 1) p.t0max = 1;
    p.mask_words = (int)ceil_div(p.t0max, 32);
    p.umax = p.t0max - 2 > 0 ? p.t0max - 2 : 0;
    p.ustride = (int)round_up(p.umax > 0 ? p.umax : 1, 4);
    p.mmax = p.t0max - 31 > 0 ? p.t0max - 31 : 0;
    p.ntiles = (int)ceil_div(p.mmax > 0 ? p.mmax : 1, kSegTile);
    p.fused_energy = ctx->fast85;
    // hop energies of the fused resample kernel: whole tiles of 10 hops
    p.hops_max = (int)(ceil_div(p.lmax > 0 ? p.lmax : 1, kRs85TileOut) * kRs85Hops);
    size_t off = 0;
    p.off_hops = off;    off = align256(off + (p.fused_energy ? sizeof(double2) * batch * p.hops_max : 0));
    // the 10 kHz float32 signals: written by the resampler, or by the widening copy of 10 kHz int16 / fp16 input
    p.off_y = off;       off = align256(off + sizeof(float) * 2 * batch * p.ystride);
    p.off_energy = off;  off = align256(off + sizeof(float) * batch * p.t0max);
    p.off_idx = off;     off = align256(off + sizeof(int32_t) * batch * p.t0max);
    p.off_count = off;   off = align256(off + sizeof(int32_t) * batch);
    p.off_prefix = off;  off = align256(off + sizeof(int32_t) * (batch + 1));
    p.off_mask = off;    off = align256(off + sizeof(uint32_t) * batch * p.mask_words);
    p.off_tob = off;     off = align256(off + sizeof(float) * 2 * batch * FSEM_STOI_NBANDS * p.ustride);
    p.off_partial = off; off = align256(off + sizeof(float2) * batch * p.ntiles);
    p.total = off;
    return p;
}

}  // namespace

extern "C" int fsem_stoi_create(fsem_stoi_ctx_t** out, const fsem_stoi_design_t* d) {
    if (!out || !d) return fail(FSEM_E_INVALID, "fsem_stoi_create: null argument");
    *out = nullptr;
    if (d->orig <= 0 || d->neu <= 0) return fail(FSEM_E_INVALID, "fsem_stoi_create: bad rates");
    int rc = d->orig != d->neu ? Resampler::check("fsem_stoi_create", d->orig, d->neu, d->width, d->ntaps, d->taps)
                               : FSEM_OK;
    if (rc != FSEM_OK) return rc;
    for (int b = 0; b < FSEM_STOI_NBANDS; ++b)
        if (d->band_lo[b] < 0 || d->band_hi[b] < d->band_lo[b] || d->band_hi[b] > 256)
            return fail(FSEM_E_INVALID, "fsem_stoi_create: band %d outside bins 0..255", b);
    if (d->band_hi[FSEM_STOI_NBANDS - 1] - d->band_lo[FSEM_STOI_NBANDS - 1] > 48)
        return fail(FSEM_E_INVALID, "fsem_stoi_create: third-octave bands must be at most 48 bins wide");
    for (int b = 0; b + 1 < FSEM_STOI_NBANDS; ++b)
        if (d->band_hi[b] != d->band_lo[b + 1] || d->band_hi[b] - d->band_lo[b] > 48)
            return fail(FSEM_E_INVALID, "fsem_stoi_create: third-octave bands must be contiguous and at most 48 bins wide");
    std::unique_ptr<fsem_stoi_ctx> ctx(new (std::nothrow) fsem_stoi_ctx());
    if (!ctx) return fail(FSEM_E_INVALID, "out of host memory");
    if ((rc = query_device(ctx->dev)) != FSEM_OK) return rc;
    ctx->clip = d->clip; ctx->dyn_range = d->dyn_range;
    StoiTables h{};
    memcpy(h.window, d->window, sizeof(h.window));
    for (int b = 0; b < FSEM_STOI_NBANDS; ++b) { h.band_lo[b] = d->band_lo[b]; h.band_hi[b] = d->band_hi[b]; }
    h.clip = d->clip; h.dyn_range = d->dyn_range;
    FSEM_CUDA(cudaMalloc(&ctx->d_tab, sizeof(StoiTables)));
    FSEM_CUDA(cudaMemcpy(ctx->d_tab, &h, sizeof(h), cudaMemcpyHostToDevice));
    ctx->rs.orig = d->orig; ctx->rs.neu = d->neu;
    if (d->orig != d->neu && (rc = ctx->rs.upload(d->orig, d->neu, d->width, d->ntaps, d->taps)) != FSEM_OK) return rc;
    if (d->orig == 8 && d->neu == 5 && d->width == 10 && d->ntaps == 28) {
        ctx->fast85 = true;
        for (int p = 0; p < 5; ++p)
            for (int j = 0; j < 28; ++j) {
                ctx->taps85.h[p][j] = d->taps[p * 28 + j];
                if ((j < rs85_lo(p) || j > rs85_hi(p)) && d->taps[p * 28 + j] != 0.f) ctx->fast85 = false;
            }
    }
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, stoi_tob_kernel<true>, kTobWarps * 32, 0) == cudaSuccess && occ > 0)
        ctx->tob_ctas_per_sm = occ;
    *out = ctx.release();
    return FSEM_OK;
}

extern "C" int fsem_stoi_destroy(fsem_stoi_ctx_t* ctx) {
    delete ctx;
    return FSEM_OK;
}

extern "C" size_t fsem_stoi_workspace_bytes(const fsem_stoi_ctx_t* ctx, int64_t batch, int64_t n) {
    if (!ctx || batch <= 0 || n <= 0) return 0;
    return stoi_plan(ctx, batch, n).total;
}

extern "C" int fsem_stoi_score_f32(fsem_stoi_ctx_t* ctx, const fsem_batch_t* in, float* stoi_out,
                                   float* estoi_out, int32_t* kept_frames_out, int32_t* status_out,
                                   void* workspace, size_t workspace_bytes, void* stream_v) {
    return fsem_stoi_score(ctx, in, FSEM_DTYPE_F32, stoi_out, estoi_out, kept_frames_out, status_out, workspace,
                           workspace_bytes, stream_v);
}

// Any ingest dtype: the resampler (the first kernel whenever the input is not already 10 kHz) reads the rows as they
// are; 10 kHz int16 / fp16 rows are widened into the workspace first (the frame kernels read float32).
extern "C" int fsem_stoi_score(fsem_stoi_ctx_t* ctx, const fsem_batch_t* in, int dtype, float* stoi_out,
                               float* estoi_out, int32_t* kept_frames_out, int32_t* status_out,
                               void* workspace, size_t workspace_bytes, void* stream_v) {
    if (!ctx || !in || !stoi_out || !estoi_out) return fail(FSEM_E_INVALID, "fsem_stoi_score: null argument");
    if (dtype_size(dtype) == 0) return fail(FSEM_E_INVALID, "fsem_stoi_score: unknown dtype %d", dtype);
    if (int rc = check_batch("fsem_stoi_score", in->clean, in->deg, in->batch, in->n, in->stride, 1, kMaxN, false))
        return rc == kEmptyBatch ? FSEM_OK : rc;
    const StoiPlan p = stoi_plan(ctx, in->batch, in->n);
    if (in->batch * (int64_t)p.t0max >= (int64_t(1) << 31))
        return fail(FSEM_E_INVALID, "fsem_stoi_score: batch x frames exceeds 2^31; split the batch");
    if (!workspace || workspace_bytes < p.total)
        return fail(FSEM_E_WORKSPACE, "fsem_stoi_score: workspace %zu < %zu bytes", workspace_bytes, p.total);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
    char* ws = static_cast<char*>(workspace);
    float* y = reinterpret_cast<float*>(ws + p.off_y);
    double2* hops = reinterpret_cast<double2*>(ws + p.off_hops);
    float* energy = reinterpret_cast<float*>(ws + p.off_energy);
    int32_t* kept_idx = reinterpret_cast<int32_t*>(ws + p.off_idx);
    int32_t* kept_count = reinterpret_cast<int32_t*>(ws + p.off_count);
    int32_t* frame_prefix = reinterpret_cast<int32_t*>(ws + p.off_prefix);
    uint32_t* mask = reinterpret_cast<uint32_t*>(ws + p.off_mask);
    float* tob = reinterpret_cast<float*>(ws + p.off_tob);
    float2* partial = reinterpret_cast<float2*>(ws + p.off_partial);

    const float* c10 = in->clean;
    const float* d10 = in->deg;
    int64_t sstride = in->stride;
    if (p.resample) {
        const bool vec4 = rows_vec4(in->clean, in->deg, in->stride, dtype_size(dtype));
        if (ctx->fast85) {
            const int64_t bps = ceil_div(p.lmax, (int64_t)kRs85TileOut * kRs85TilesPerCta);
            const unsigned grid = (unsigned)(bps * 2 * in->batch);       // < 2^31: batch x frames is checked above
            { ProfScope prof_(K_STOI_RESAMPLE, stream);
              dispatch_dtype(dtype, [&](auto tag) {
                  using T = decltype(tag);
                  const T* c = reinterpret_cast<const T*>(in->clean);
                  const T* d = reinterpret_cast<const T*>(in->deg);
                  if (vec4)
                      stoi_resample85_kernel<true, T><<<grid, kRs85Threads, 0, stream>>>(
                          c, d, in->lengths, in->batch, in->n, in->stride, ctx->taps85, ctx->d_tab, y, p.ystride, hops,
                          p.hops_max, (int)bps);
                  else
                      stoi_resample85_kernel<false, T><<<grid, kRs85Threads, 0, stream>>>(
                          c, d, in->lengths, in->batch, in->n, in->stride, ctx->taps85, ctx->d_tab, y, p.ystride, hops,
                          p.hops_max, (int)bps);
                  return FSEM_OK;
              }); }
            FSEM_LAUNCHED();
        } else {
            const int rc = ctx->rs.launch("fsem_stoi_score", K_STOI_RESAMPLE, in, dtype, y, p.ystride, nullptr, stream);
            if (rc != FSEM_OK) return rc;
        }
        c10 = y;
        d10 = y + in->batch * p.ystride;
        sstride = p.ystride;
    } else if (dtype != FSEM_DTYPE_F32) {
        // already 10 kHz, but not float32: widen into the (otherwise unused) resample area of the workspace
        int rc = launch_ingest(in->clean, dtype, in->batch, in->n, in->stride, y, p.ystride, stream);
        if (rc == FSEM_OK)
            rc = launch_ingest(in->deg, dtype, in->batch, in->n, in->stride, y + in->batch * p.ystride, p.ystride, stream);
        if (rc != FSEM_OK) return rc;
        c10 = y;
        d10 = y + in->batch * p.ystride;
        sstride = p.ystride;
    }
    if (p.fused_energy) {
        const int64_t threads = in->batch * (int64_t)p.t0max;
        { ProfScope prof_(K_STOI_ENERGY, stream);
          stoi_energy_from_hops_kernel<<<(unsigned)ceil_div(threads, 256), 256, 0, stream>>>(
              hops, p.hops_max, in->lengths, in->batch, in->n, p.t0max, energy); }
        FSEM_LAUNCHED();
    } else {
        const int64_t warps = in->batch * (int64_t)p.t0max;
        { ProfScope prof_(K_STOI_ENERGY, stream);
          stoi_energy_kernel<<<(unsigned)ceil_div(warps * 32, 256), 256, 0, stream>>>(
            c10, sstride, in->lengths, in->batch, in->n, ctx->rs.orig, ctx->rs.neu, p.t0max, ctx->d_tab, energy); }
        FSEM_LAUNCHED();
    }
    {
        { ProfScope prof_(K_STOI_COMPACT, stream);
          stoi_compact_kernel<<<(unsigned)ceil_div(in->batch * 32, 128), 128, 0, stream>>>(
              energy, in->lengths, in->batch, in->n, ctx->rs.orig, ctx->rs.neu, p.t0max, p.mask_words, ctx->dyn_range,
              kept_idx, kept_count, mask); }
        FSEM_LAUNCHED();
    }
    if (p.umax > 0) {
        { ProfScope prof_(K_STOI_COMPACT, stream);
          stoi_prefix_kernel<<<1, 1024, 0, stream>>>(kept_count, in->batch, frame_prefix); }
        FSEM_LAUNCHED();
        const int64_t units = in->batch * (int64_t)p.umax;          // upper bound of the real frame count
        int64_t grid = ceil_div(units, kTobWarps);
        const int64_t cap = (int64_t)ctx->dev.sms * ctx->tob_ctas_per_sm;
        if (grid > cap) grid = cap;
        const bool vec2 = (reinterpret_cast<uintptr_t>(c10) & 7u) == 0 && (reinterpret_cast<uintptr_t>(d10) & 7u) == 0 &&
                          sstride % 2 == 0;
        { ProfScope prof_(K_STOI_TOB, stream);
          if (vec2)
              stoi_tob_kernel<true><<<(unsigned)grid, kTobWarps * 32, 0, stream>>>(
                  c10, d10, sstride, in->batch, p.t0max, p.umax, p.ustride, kept_idx, frame_prefix, ctx->d_tab, tob);
          else
              stoi_tob_kernel<false><<<(unsigned)grid, kTobWarps * 32, 0, stream>>>(
                  c10, d10, sstride, in->batch, p.t0max, p.umax, p.ustride, kept_idx, frame_prefix, ctx->d_tab, tob); }
        FSEM_LAUNCHED();
    }
    {
        { ProfScope prof_(K_STOI_SEGMENT, stream);
          stoi_segment_kernel<<<(unsigned)(in->batch * ceil_div(p.ntiles, kSegTilesPerCta)), kSegThreads, 0, stream>>>(
              tob, in->batch, p.ustride, p.ntiles, kept_count, ctx->clip, partial); }
        FSEM_LAUNCHED();
        { ProfScope prof_(K_STOI_FINALIZE, stream);
          stoi_finalize_kernel<<<(unsigned)ceil_div(in->batch, 128), 128, 0, stream>>>(
              partial, in->batch, p.ntiles, kept_count, stoi_out, estoi_out, kept_frames_out, status_out); }
        FSEM_LAUNCHED();
    }
    return FSEM_OK;
}

extern "C" int fsem_stoi_debug_taps(fsem_stoi_ctx_t* ctx, int64_t batch, int64_t n, const void* workspace,
                                    uint32_t* mask_out, float* tob_out, float* resampled_out, int64_t* dims_out,
                                    void* stream_v) {
    if (!ctx || !workspace) return fail(FSEM_E_INVALID, "fsem_stoi_debug_taps: null argument");
    const StoiPlan p = stoi_plan(ctx, batch, n);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
    const char* ws = static_cast<const char*>(workspace);
    if (dims_out) {
        dims_out[0] = p.mask_words;
        dims_out[1] = p.ustride;
        dims_out[2] = p.resample ? p.ystride : 0;
    }
    if (mask_out)
        FSEM_CUDA(cudaMemcpyAsync(mask_out, ws + p.off_mask, sizeof(uint32_t) * batch * p.mask_words,
                                  cudaMemcpyDeviceToDevice, stream));
    if (tob_out)
        FSEM_CUDA(cudaMemcpyAsync(tob_out, ws + p.off_tob, sizeof(float) * 2 * batch * FSEM_STOI_NBANDS * p.ustride,
                                  cudaMemcpyDeviceToDevice, stream));
    if (resampled_out && p.resample)
        FSEM_CUDA(cudaMemcpyAsync(resampled_out, ws + p.off_y, sizeof(float) * 2 * batch * p.ystride,
                                  cudaMemcpyDeviceToDevice, stream));
    return FSEM_OK;
}

extern "C" int fsem_stoi_mask_margin(fsem_stoi_ctx_t* ctx, int64_t batch, int64_t n, const int32_t* lengths,
                                     const void* workspace, float* margin_out, void* stream_v) {
    if (!ctx || !workspace || !margin_out) return fail(FSEM_E_INVALID, "fsem_stoi_mask_margin: null argument");
    if (batch <= 0 || n <= 0) return fail(FSEM_E_INVALID, "fsem_stoi_mask_margin: bad shape");
    const StoiPlan p = stoi_plan(ctx, batch, n);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
    const float* energy = reinterpret_cast<const float*>(static_cast<const char*>(workspace) + p.off_energy);
    { ProfScope prof_(K_STOI_MARGIN, stream);
      stoi_margin_kernel<<<(unsigned)ceil_div(batch * 32, 128), 128, 0, stream>>>(
          energy, lengths, batch, n, ctx->rs.orig, ctx->rs.neu, p.t0max, ctx->dyn_range, margin_out); }
    FSEM_LAUNCHED();
    return FSEM_OK;
}

// ================================================================================================
// Host entry points.  One pipeline serves PESQ only, STOI only and PESQ + STOI on one upload (SURVEY.md 8f rank 1:
// callers of the reference always score both metrics on the same pair of tensors, README.md:29-30,
// benchmark_metrics.py:22,24; with host tensors the host->device copy dominates, so every chunk is copied ONCE and
// all selected kernel chains run on it), for every ingest dtype (SURVEY.md 8f rank 2).
// ================================================================================================
namespace {

// device rows of `dtype` -> device fp32 rows on `stream`
int launch_ingest(const void* src, int dtype, int64_t rows, int64_t n, int64_t sstride, float* dst, int64_t dstride,
                  cudaStream_t stream) {
    if (rows <= 0 || n <= 0) return FSEM_OK;
    if (dtype == FSEM_DTYPE_F32) {
        FSEM_CUDA(cudaMemcpy2DAsync(dst, dstride * sizeof(float), src, sstride * sizeof(float), n * sizeof(float), rows,
                                    cudaMemcpyDeviceToDevice, stream));
        return FSEM_OK;
    }
    const bool vec = aligned16(src) && aligned16(dst) && sstride % 8 == 0 && dstride % 4 == 0;
    const int64_t groups = rows * ceil_div(n, 8);
    int64_t grid = ceil_div(groups, 256);
    if (grid > (1 << 20)) grid = 1 << 20;
    { ProfScope prof_(K_INGEST, stream);
      if (dtype == FSEM_DTYPE_I16) {
          const int16_t* s = static_cast<const int16_t*>(src);
          if (vec) ingest_kernel<int16_t, true><<<(unsigned)grid, 256, 0, stream>>>(s, sstride, dst, dstride, rows, n);
          else ingest_kernel<int16_t, false><<<(unsigned)grid, 256, 0, stream>>>(s, sstride, dst, dstride, rows, n);
      } else {
          const __half* s = static_cast<const __half*>(src);
          if (vec) ingest_kernel<__half, true><<<(unsigned)grid, 256, 0, stream>>>(s, sstride, dst, dstride, rows, n);
          else ingest_kernel<__half, false><<<(unsigned)grid, 256, 0, stream>>>(s, sstride, dst, dstride, rows, n);
      } }
    FSEM_LAUNCHED();
    return FSEM_OK;
}

int score_host_any(const char* who, fsem_pesq_ctx* pctx, fsem_stoi_ctx* sctx, const void* clean, const void* deg,
                   int dtype, const int32_t* lengths, int64_t batch, int64_t n, int64_t stride, float* mos_out,
                   int32_t* pesq_status_out, float* stoi_out, float* estoi_out, int32_t* kept_frames_out,
                   int32_t* stoi_status_out) {
    if ((!pctx && !sctx) || !clean || !deg || (pctx && !mos_out) || (sctx && (!stoi_out || !estoi_out)))
        return fail(FSEM_E_INVALID, "%s: null argument", who);
    const size_t es = dtype_size(dtype);
    if (es == 0) return fail(FSEM_E_INVALID, "%s: unknown dtype %d", who, dtype);
    if (int rc = check_batch(who, clean, deg, batch, n, stride, 0, INT64_MAX, false))
        return rc == kEmptyBatch ? FSEM_OK : rc;
    if (pctx && !lengths && pesq_num_frames(pesq_plan(pctx, 1, n).n) < 20)
        return fail(FSEM_E_TOO_SHORT, "PESQ needs at least 20 frames of 512/256 samples at 16 kHz; n=%lld is too short",
                    (long long)n);
    HostPipe& P = pctx ? pctx->pipe : sctx->pipe;
    int rc = P.init();
    if (rc != FSEM_OK) return rc;
    // staged rows as uploaded: 16-byte aligned pitch; the first kernel of either chain reads them in their own dtype
    // (no widening pass: a 2-byte batch is read from HBM at 2 bytes per sample as well)
    const int64_t rstride = round_up(n, 16 / (int64_t)es);
    const int64_t per = host_chunk_items(batch, n, es);
    const size_t raw_sig = align256(es * per * rstride);
    const size_t in_bytes = 2 * raw_sig + align256(sizeof(int32_t) * per);
    const size_t ws_pesq = pctx ? align256(fsem_pesq_workspace_bytes(pctx, per, n)) : 0;
    const size_t ws_stoi = sctx ? align256(fsem_stoi_workspace_bytes(sctx, per, n)) : 0;
    const size_t col = align256(sizeof(float) * batch);
    rc = P.reserve(in_bytes, ws_pesq + ws_stoi, 6 * col);
    if (rc != FSEM_OK) return rc;
    char* const ob = static_cast<char*>(P.out);
    char* const wsb = static_cast<char*>(P.ws);
    const char* h_clean = static_cast<const char*>(clean);
    const char* h_deg = static_cast<const char*>(deg);
    auto upload = [&](void* dst, const char* src, int64_t cnt) -> cudaError_t {
        if (stride == n && rstride == n)
            return cudaMemcpyAsync(dst, src, es * n * cnt, cudaMemcpyHostToDevice, P.copy);
        return cudaMemcpy2DAsync(dst, rstride * es, src, stride * es, n * es, cnt, cudaMemcpyHostToDevice, P.copy);
    };
    // Everything that touches the caller's host buffers or the staging slots runs inside `run`; whatever it returns,
    // both streams are drained before this function does, so that no async copy still references memory the caller
    // may free or reuse after an error return.
    auto run = [&]() -> int {
    int64_t done_chunks = 0;
    for (int64_t i0 = 0; i0 < batch; i0 += per, ++done_chunks) {
        const int slot = (int)(done_chunks & 1);
        const int64_t cnt = (batch - i0 < per) ? (batch - i0) : per;
        char* base = static_cast<char*>(P.in[slot]);
        int32_t* d_len = reinterpret_cast<int32_t*>(base + 2 * raw_sig);
        if (done_chunks >= 2) FSEM_CUDA(cudaStreamWaitEvent(P.copy, P.done[slot], 0));   // staging slot free again
        FSEM_CUDA(upload(base, h_clean + (size_t)i0 * stride * es, cnt));
        FSEM_CUDA(upload(base + raw_sig, h_deg + (size_t)i0 * stride * es, cnt));
        if (lengths)
            FSEM_CUDA(cudaMemcpyAsync(d_len, lengths + i0, sizeof(int32_t) * cnt, cudaMemcpyHostToDevice, P.copy));
        FSEM_CUDA(cudaEventRecord(P.copied[slot], P.copy));
        FSEM_CUDA(cudaStreamWaitEvent(P.compute, P.copied[slot], 0));
        fsem_batch_t dev{reinterpret_cast<const float*>(base), reinterpret_cast<const float*>(base + raw_sig),
                         lengths ? d_len : nullptr, cnt, n, rstride};
        if (rc == FSEM_OK && pctx && sctx)
            rc = fsem_pesq_stoi_score(pctx, sctx, &dev, dtype, reinterpret_cast<float*>(ob) + i0,
                                          reinterpret_cast<int32_t*>(ob + col) + i0,
                                          reinterpret_cast<float*>(ob + 2 * col) + i0,
                                          reinterpret_cast<float*>(ob + 3 * col) + i0,
                                          reinterpret_cast<int32_t*>(ob + 4 * col) + i0,
                                          reinterpret_cast<int32_t*>(ob + 5 * col) + i0, wsb, ws_pesq, wsb + ws_pesq,
                                          ws_stoi, P.compute);
        else if (rc == FSEM_OK && pctx)
            rc = fsem_pesq_score(pctx, &dev, dtype, reinterpret_cast<float*>(ob) + i0,
                                 reinterpret_cast<int32_t*>(ob + col) + i0, wsb, ws_pesq, P.compute);
        else if (rc == FSEM_OK && sctx)
            rc = fsem_stoi_score(sctx, &dev, dtype, reinterpret_cast<float*>(ob + 2 * col) + i0,
                                     reinterpret_cast<float*>(ob + 3 * col) + i0,
                                     reinterpret_cast<int32_t*>(ob + 4 * col) + i0,
                                     reinterpret_cast<int32_t*>(ob + 5 * col) + i0, wsb + ws_pesq, ws_stoi, P.compute);
        if (rc != FSEM_OK) return rc;
        FSEM_CUDA(cudaEventRecord(P.done[slot], P.compute));
    }
    // one read-back of the score columns (a per-chunk copy into pageable memory would stall the pipeline)
    const size_t nb = sizeof(float) * batch;
    auto readback = [&](void* dst, size_t column) -> cudaError_t {
        return dst ? cudaMemcpyAsync(dst, ob + column * col, nb, cudaMemcpyDeviceToHost, P.compute) : cudaSuccess;
    };
    if (pctx) {
        FSEM_CUDA(readback(mos_out, 0));
        FSEM_CUDA(readback(pesq_status_out, 1));
    }
    if (sctx) {
        FSEM_CUDA(readback(stoi_out, 2));
        FSEM_CUDA(readback(estoi_out, 3));
        FSEM_CUDA(readback(kept_frames_out, 4));
        FSEM_CUDA(readback(stoi_status_out, 5));
    }
    return FSEM_OK;
    };
    rc = run();
    const cudaError_t e_copy = cudaStreamSynchronize(P.copy);
    const cudaError_t e_comp = cudaStreamSynchronize(P.compute);
    if (rc != FSEM_OK) return rc;                                    // g_err already holds the first failure
    if (e_copy != cudaSuccess || e_comp != cudaSuccess)
        return fail(FSEM_E_CUDA, "%s: %s", who, cudaGetErrorString(e_copy != cudaSuccess ? e_copy : e_comp));
    return FSEM_OK;
}

}  // namespace

extern "C" int fsem_ingest_f32(const void* src, int dtype, int64_t rows, int64_t n, int64_t src_stride, float* dst,
                               int64_t dst_stride, void* stream) {
    if (!src || !dst) return fail(FSEM_E_INVALID, "fsem_ingest_f32: null argument");
    if (dtype_size(dtype) == 0) return fail(FSEM_E_INVALID, "fsem_ingest_f32: unknown dtype %d", dtype);
    if (dst_stride < n) return fail(FSEM_E_INVALID, "fsem_ingest_f32: dst_stride %lld < n", (long long)dst_stride);
    if (int rc = check_batch("fsem_ingest_f32", src, dst, rows, n, src_stride, 0, INT64_MAX, false))
        return rc == kEmptyBatch ? FSEM_OK : rc;
    return launch_ingest(src, dtype, rows, n, src_stride, dst, dst_stride, static_cast<cudaStream_t>(stream));
}

extern "C" int fsem_score_host(fsem_pesq_ctx_t* pesq, fsem_stoi_ctx_t* stoi, const void* clean, const void* deg, int dtype,
                               const int32_t* lengths, int64_t batch, int64_t n, int64_t stride, float* mos_out,
                               int32_t* pesq_status_out, float* stoi_out, float* estoi_out, int32_t* kept_frames_out,
                               int32_t* stoi_status_out) {
    return score_host_any("fsem_score_host", pesq, stoi, clean, deg, dtype, lengths, batch, n, stride, mos_out,
                          pesq_status_out, stoi_out, estoi_out, kept_frames_out, stoi_status_out);
}

extern "C" int fsem_pesq_score_host_f32(fsem_pesq_ctx_t* ctx, const fsem_batch_t* in, float* mos_out,
                                        int32_t* status_out) {
    if (!ctx || !in) return fail(FSEM_E_INVALID, "fsem_pesq_score_host_f32: null argument");
    return score_host_any("fsem_pesq_score_host_f32", ctx, nullptr, in->clean, in->deg, FSEM_DTYPE_F32, in->lengths,
                          in->batch, in->n, in->stride, mos_out, status_out, nullptr, nullptr, nullptr, nullptr);
}

extern "C" int fsem_stoi_score_host_f32(fsem_stoi_ctx_t* ctx, const fsem_batch_t* in, float* stoi_out,
                                        float* estoi_out, int32_t* kept_frames_out, int32_t* status_out) {
    if (!ctx || !in) return fail(FSEM_E_INVALID, "fsem_stoi_score_host_f32: null argument");
    return score_host_any("fsem_stoi_score_host_f32", nullptr, ctx, in->clean, in->deg, FSEM_DTYPE_F32, in->lengths,
                          in->batch, in->n, in->stride, nullptr, nullptr, stoi_out, estoi_out, kept_frames_out,
                          status_out);
}

extern "C" int fsem_pesq_stoi_score_host_f32(fsem_pesq_ctx_t* pctx, fsem_stoi_ctx_t* sctx, const fsem_batch_t* in,
                                             float* mos_out, int32_t* pesq_status_out, float* stoi_out,
                                             float* estoi_out, int32_t* kept_frames_out, int32_t* stoi_status_out) {
    if (!pctx || !sctx || !in) return fail(FSEM_E_INVALID, "fsem_pesq_stoi_score_host_f32: null argument");
    return score_host_any("fsem_pesq_stoi_score_host_f32", pctx, sctx, in->clean, in->deg, FSEM_DTYPE_F32, in->lengths,
                          in->batch, in->n, in->stride, mos_out, pesq_status_out, stoi_out, estoi_out, kept_frames_out,
                          stoi_status_out);
}

// ================================================================================================
// Resample-on-ingest as a building block (BaseMetric.prepare_audio, fast_se_metrics/base.py:13,19-20): the
// general polyphase kernel behind a small context that owns the device copy of the taps.  PESQ and STOI run the
// same kernel inside their own chains; LSD and SDR call this first.
// ================================================================================================
struct fsem_resampler : Resampler {};

extern "C" int fsem_resampler_create(fsem_resampler_t** out, int32_t orig, int32_t neu, int32_t width, int32_t ntaps,
                                     const float* taps) {
    if (!out) return fail(FSEM_E_INVALID, "fsem_resampler_create: null argument");
    *out = nullptr;
    int rc = Resampler::check("fsem_resampler_create", orig, neu, width, ntaps, taps);
    if (rc != FSEM_OK) return rc;
    std::unique_ptr<fsem_resampler> r(new (std::nothrow) fsem_resampler());
    if (!r) return fail(FSEM_E_INVALID, "out of host memory");
    if ((rc = r->upload(orig, neu, width, ntaps, taps)) != FSEM_OK) return rc;
    *out = r.release();
    return FSEM_OK;
}

extern "C" int fsem_resampler_destroy(fsem_resampler_t* r) {
    delete r;
    return FSEM_OK;
}

extern "C" int64_t fsem_resampled_len(const fsem_resampler_t* r, int64_t n) {
    if (!r || n < 0) return 0;
    return stoi_resampled_len(n, r->orig, r->neu);
}

extern "C" int fsem_resample_f32(fsem_resampler_t* r, const fsem_batch_t* in, float* out, int64_t out_stride,
                                 int32_t* lengths_out, void* stream_v) {
    if (!r || !in || !out) return fail(FSEM_E_INVALID, "fsem_resample_f32: null argument");
    if (int rc = check_batch("fsem_resample_f32", in->clean, in->deg, in->batch, in->n, in->stride, 1, kMaxN, true))
        return rc == kEmptyBatch ? FSEM_OK : rc;
    const int64_t L = stoi_resampled_len(in->n, r->orig, r->neu);
    if (out_stride < L) return fail(FSEM_E_INVALID, "fsem_resample_f32: out_stride %lld < resampled length %lld",
                                    (long long)out_stride, (long long)L);
    if (in->lengths && !lengths_out) return fail(FSEM_E_INVALID, "fsem_resample_f32: lengths given but lengths_out is null");
    return r->launch("fsem_resample_f32", K_PESQ_RESAMPLE, in, FSEM_DTYPE_F32, out, out_stride, lengths_out,
                     static_cast<cudaStream_t>(stream_v));
}

// ================================================================================================
// LSD (SURVEY.md 8f rank 3): log-spectral distance on the same packed FFT (fast_se_metrics/LSD.py:6-52)
// ================================================================================================
struct fsem_lsd_ctx {
    DeviceInfo dev;
    float* d_hann = nullptr;
    int ctas_per_sm = 2;

    ~fsem_lsd_ctx() { if (d_hann) cudaFree(d_hann); }
};

namespace {
struct LsdPlan { int tmax; size_t off_alpha, off_frames, total; };
LsdPlan lsd_plan(int64_t batch, int64_t n) {
    LsdPlan p{};
    p.tmax = lsd_num_frames(n);
    size_t off = 0;
    p.off_alpha = off;  off = align256(off + sizeof(float) * batch);
    p.off_frames = off; off = align256(off + sizeof(float) * batch * p.tmax);
    p.total = off;
    return p;
}
}  // namespace

extern "C" int fsem_lsd_create(fsem_lsd_ctx_t** out, const float* hann512) {
    if (!out || !hann512) return fail(FSEM_E_INVALID, "fsem_lsd_create: null argument");
    *out = nullptr;
    std::unique_ptr<fsem_lsd_ctx> ctx(new (std::nothrow) fsem_lsd_ctx());
    if (!ctx) return fail(FSEM_E_INVALID, "out of host memory");
    const int rc = query_device(ctx->dev);
    if (rc != FSEM_OK) return rc;
    FSEM_CUDA(cudaMalloc(&ctx->d_hann, sizeof(float) * 512));
    FSEM_CUDA(cudaMemcpy(ctx->d_hann, hann512, sizeof(float) * 512, cudaMemcpyHostToDevice));
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, lsd_frames_kernel<true>, kLsdWarps * 32, 0) == cudaSuccess && occ > 0)
        ctx->ctas_per_sm = occ;
    *out = ctx.release();
    return FSEM_OK;
}

extern "C" int fsem_lsd_destroy(fsem_lsd_ctx_t* ctx) {
    delete ctx;
    return FSEM_OK;
}

extern "C" size_t fsem_lsd_workspace_bytes(const fsem_lsd_ctx_t* ctx, int64_t batch, int64_t n) {
    if (!ctx || batch <= 0 || n <= 0) return 0;
    return lsd_plan(batch, n).total;
}

extern "C" int fsem_lsd_score_f32(fsem_lsd_ctx_t* ctx, const fsem_batch_t* in, float* lsd_out, void* workspace,
                                  size_t workspace_bytes, void* stream_v) {
    if (!ctx || !in || !lsd_out) return fail(FSEM_E_INVALID, "fsem_lsd_score_f32: null argument");
    if (int rc = check_batch("fsem_lsd_score_f32", in->clean, in->deg, in->batch, in->n, in->stride, 1, kMaxN, true))
        return rc == kEmptyBatch ? FSEM_OK : rc;
    const LsdPlan p = lsd_plan(in->batch, in->n);
    if (!workspace || workspace_bytes < p.total)
        return fail(FSEM_E_WORKSPACE, "fsem_lsd_score_f32: workspace %zu < %zu bytes", workspace_bytes, p.total);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
    char* ws = static_cast<char*>(workspace);
    float* alpha = reinterpret_cast<float*>(ws + p.off_alpha);
    float* frames = reinterpret_cast<float*>(ws + p.off_frames);
    lsd_scale_kernel<<<(unsigned)in->batch, 256, 0, stream>>>(in->clean, in->deg, in->lengths, in->batch, in->n,
                                                             in->stride, alpha);
    FSEM_LAUNCHED();
    const int64_t units = in->batch * (int64_t)p.tmax;
    int64_t grid = ceil_div(units, kLsdWarps);
    const int64_t cap = (int64_t)ctx->dev.sms * ctx->ctas_per_sm;
    if (grid > cap) grid = cap;
    const bool vec2 = (reinterpret_cast<uintptr_t>(in->clean) & 7u) == 0 && (reinterpret_cast<uintptr_t>(in->deg) & 7u) == 0 &&
                      in->stride % 2 == 0;
    { ProfScope prof_(K_LSD_FRAMES, stream);
      if (vec2)
          lsd_frames_kernel<true><<<(unsigned)grid, kLsdWarps * 32, 0, stream>>>(
              in->clean, in->deg, in->lengths, in->batch, in->n, in->stride, p.tmax, ctx->d_hann, alpha, frames);
      else
          lsd_frames_kernel<false><<<(unsigned)grid, kLsdWarps * 32, 0, stream>>>(
              in->clean, in->deg, in->lengths, in->batch, in->n, in->stride, p.tmax, ctx->d_hann, alpha, frames); }
    FSEM_LAUNCHED();
    lsd_finalize_kernel<<<(unsigned)ceil_div(in->batch, 128), 128, 0, stream>>>(frames, in->lengths, in->batch, in->n,
                                                                               p.tmax, lsd_out);
    FSEM_LAUNCHED();
    return FSEM_OK;
}

// ------------------------------------------------------------------------------------------------
// Device entry point for BOTH metrics: the two kernel chains back to back on `stream`, each reading the input itself
// (SURVEY.md 8f rank 1 is delivered as "single upload": the host pipeline copies every chunk once and calls this).
extern "C" int fsem_pesq_stoi_score(fsem_pesq_ctx_t* pctx, fsem_stoi_ctx_t* sctx, const fsem_batch_t* in, int dtype,
                                    float* mos_out, int32_t* pesq_status_out, float* stoi_out, float* estoi_out,
                                    int32_t* kept_frames_out, int32_t* stoi_status_out, void* ws_pesq,
                                    size_t ws_pesq_bytes, void* ws_stoi, size_t ws_stoi_bytes, void* stream) {
    if (!pctx || !sctx) return fail(FSEM_E_INVALID, "fsem_pesq_stoi_score: null context");
    int rc = fsem_pesq_score(pctx, in, dtype, mos_out, pesq_status_out, ws_pesq, ws_pesq_bytes, stream);
    if (rc == FSEM_OK)
        rc = fsem_stoi_score(sctx, in, dtype, stoi_out, estoi_out, kept_frames_out, stoi_status_out, ws_stoi,
                             ws_stoi_bytes, stream);
    return rc;
}

extern "C" int fsem_pesq_stoi_score_f32(fsem_pesq_ctx_t* pctx, fsem_stoi_ctx_t* sctx, const fsem_batch_t* in,
                                        float* mos_out, int32_t* pesq_status_out, float* stoi_out, float* estoi_out,
                                        int32_t* kept_frames_out, int32_t* stoi_status_out, void* ws_pesq,
                                        size_t ws_pesq_bytes, void* ws_stoi, size_t ws_stoi_bytes, void* stream) {
    return fsem_pesq_stoi_score(pctx, sctx, in, FSEM_DTYPE_F32, mos_out, pesq_status_out, stoi_out, estoi_out,
                                kept_frames_out, stoi_status_out, ws_pesq, ws_pesq_bytes, ws_stoi, ws_stoi_bytes, stream);
}

// ------------------------------------------------------------------------------------------------
// Captured scoring: one CUDA graph; the batch is cut into slices and every slice's PESQ chain and STOI chain is a
// parallel branch (include/fsem.h).
struct fsem_graph {
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    void* ws = nullptr;                 // workspaces of all branches (owned)
    int kernel_nodes = 0;
    int slices = 0;
    int device = -1;
};

namespace {
void graph_free(fsem_graph* g) {
    if (!g) return;
    if (g->exec) cudaGraphExecDestroy(g->exec);
    if (g->graph) cudaGraphDestroy(g->graph);
    if (g->ws) cudaFree(g->ws);
    delete g;
}
constexpr int kGraphMaxSlices = 16;
}  // namespace

extern "C" int fsem_graph_create(fsem_graph_t** out, fsem_pesq_ctx_t* pctx, fsem_stoi_ctx_t* sctx, const fsem_batch_t* in,
                                 int dtype, float* mos_out, int32_t* pesq_status_out, float* stoi_out, float* estoi_out,
                                 int32_t* kept_frames_out, int32_t* stoi_status_out, int slices) {
    if (!out) return fail(FSEM_E_INVALID, "fsem_graph_create: null output");
    *out = nullptr;
    if (!pctx && !sctx) return fail(FSEM_E_INVALID, "fsem_graph_create: no metric selected");
    if (!in || in->batch <= 0) return fail(FSEM_E_INVALID, "fsem_graph_create: empty batch");
    if ((pctx && !mos_out) || (sctx && (!stoi_out || !estoi_out)))
        return fail(FSEM_E_INVALID, "fsem_graph_create: null output column");
    const size_t es = dtype_size(dtype);
    if (es == 0) return fail(FSEM_E_INVALID, "fsem_graph_create: unknown dtype %d", dtype);
    // measured on B200 (profiles/r02_config_sweep.json, by_slices): two branches already fill the chip, cutting the batch
    // further gains <= 1 % at 8192 x 10 s and loses below that -- the library's own choice is one slice
    if (slices <= 0) slices = 1;
    if (slices > kGraphMaxSlices) slices = kGraphMaxSlices;
    if (slices > in->batch) slices = (int)in->batch;
    fsem_graph* g = new (std::nothrow) fsem_graph();
    if (!g) return fail(FSEM_E_INVALID, "fsem_graph_create: out of host memory");
    g->slices = slices;
    // slice s = items [b0[s], b0[s + 1]): contiguous, sizes differ by at most one
    int64_t b0[kGraphMaxSlices + 1];
    for (int s = 0; s <= slices; ++s) b0[s] = in->batch * s / slices;
    if (pctx) pctx->plan_batch_hint = in->batch;                      // one IIR chunk grid for every slice
    size_t ws_off[2 * kGraphMaxSlices + 1];
    ws_off[0] = 0;
    for (int s = 0; s < slices; ++s) {
        const int64_t nb = b0[s + 1] - b0[s];
        ws_off[2 * s + 1] = ws_off[2 * s] + (pctx ? align256(fsem_pesq_workspace_bytes(pctx, nb, in->n)) : 0);
        ws_off[2 * s + 2] = ws_off[2 * s + 1] + (sctx ? align256(fsem_stoi_workspace_bytes(sctx, nb, in->n)) : 0);
    }
    const int nbranch = (pctx ? slices : 0) + (sctx ? slices : 0);
    cudaStream_t main_s = nullptr;
    std::vector<cudaStream_t> side(nbranch > 1 ? nbranch - 1 : 0, nullptr);
    std::vector<cudaEvent_t> join(side.size(), nullptr);
    cudaEvent_t fork_e = nullptr;
    int rc = FSEM_OK;
    cudaError_t e = cudaGetDevice(&g->device);
    if (e == cudaSuccess) e = cudaMalloc(&g->ws, ws_off[2 * slices] > 0 ? ws_off[2 * slices] : 256);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&main_s, cudaStreamNonBlocking);
    for (size_t i = 0; i < side.size() && e == cudaSuccess; ++i) {
        e = cudaStreamCreateWithFlags(&side[i], cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&join[i], cudaEventDisableTiming);
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&fork_e, cudaEventDisableTiming);
    const bool profile_was = g_profile;
    g_profile = false;                                     // event pairs of the per-kernel profiler do not belong in a graph
    const int64_t launches_before = g_launches.load(std::memory_order_relaxed);
    bool capturing = false;
    if (e == cudaSuccess) {
        e = cudaStreamBeginCapture(main_s, cudaStreamCaptureModeThreadLocal);
        capturing = (e == cudaSuccess);
    }
    if (capturing) {
        if (!side.empty()) e = cudaEventRecord(fork_e, main_s);
        for (size_t i = 0; i < side.size() && e == cudaSuccess; ++i) e = cudaStreamWaitEvent(side[i], fork_e, 0);
        // branch k runs on the main stream (k = 0) or on side[k - 1]; PESQ branches first: they are the longer chains
        int k = 0;
        auto stream_of = [&](int idx) { return idx == 0 ? main_s : side[idx - 1]; };
        const char* cb = reinterpret_cast<const char*>(in->clean);
        const char* db = reinterpret_cast<const char*>(in->deg);
        char* wsb = static_cast<char*>(g->ws);
        for (int pass = 0; pass < 2 && e == cudaSuccess && rc == FSEM_OK; ++pass) {
            if ((pass == 0 && !pctx) || (pass == 1 && !sctx)) continue;
            for (int s = 0; s < slices && rc == FSEM_OK; ++s, ++k) {
                const int64_t i0 = b0[s], nb = b0[s + 1] - b0[s];
                const fsem_batch_t sub{reinterpret_cast<const float*>(cb + (size_t)i0 * in->stride * es),
                                       reinterpret_cast<const float*>(db + (size_t)i0 * in->stride * es),
                                       in->lengths ? in->lengths + i0 : nullptr, nb, in->n, in->stride};
                if (pass == 0)
                    rc = fsem_pesq_score(pctx, &sub, dtype, mos_out + i0, pesq_status_out ? pesq_status_out + i0 : nullptr,
                                         wsb + ws_off[2 * s], ws_off[2 * s + 1] - ws_off[2 * s], stream_of(k));
                else
                    rc = fsem_stoi_score(sctx, &sub, dtype, stoi_out + i0, estoi_out + i0,
                                         kept_frames_out ? kept_frames_out + i0 : nullptr,
                                         stoi_status_out ? stoi_status_out + i0 : nullptr, wsb + ws_off[2 * s + 1],
                                         ws_off[2 * s + 2] - ws_off[2 * s + 1], stream_of(k));
            }
        }
        // join every side stream (also on the error path: the capture must be closed with all streams rejoined)
        for (size_t i = 0; i < side.size(); ++i) {
            cudaError_t j = cudaEventRecord(join[i], side[i]);
            if (j == cudaSuccess) j = cudaStreamWaitEvent(main_s, join[i], 0);
            if (e == cudaSuccess && rc == FSEM_OK) e = j;
        }
        cudaError_t end = cudaStreamEndCapture(main_s, &g->graph);
        if (e == cudaSuccess) e = end;
    }
    if (pctx) pctx->plan_batch_hint = 0;
    g_profile = profile_was;
    if (e == cudaSuccess && rc == FSEM_OK) {
        g->kernel_nodes = (int)(g_launches.load(std::memory_order_relaxed) - launches_before);
        e = cudaGraphInstantiate(&g->exec, g->graph, 0);
    }
    g_launches.store(launches_before, std::memory_order_relaxed);   // captured, not launched
    if (main_s) cudaStreamDestroy(main_s);
    for (size_t i = 0; i < side.size(); ++i) {
        if (side[i]) cudaStreamDestroy(side[i]);
        if (join[i]) cudaEventDestroy(join[i]);
    }
    if (fork_e) cudaEventDestroy(fork_e);
    if (rc != FSEM_OK) { graph_free(g); cudaGetLastError(); return rc; }   // message already set by the score call
    if (e != cudaSuccess) {
        graph_free(g);
        cudaGetLastError();
        return fail(FSEM_E_CUDA, "fsem_graph_create: %s", cudaGetErrorString(e));
    }
    *out = g;
    return FSEM_OK;
}

extern "C" int fsem_graph_launch(fsem_graph_t* g, void* stream) {
    if (!g || !g->exec) return fail(FSEM_E_INVALID, "fsem_graph_launch: null graph");
    FSEM_CUDA(cudaGraphLaunch(g->exec, static_cast<cudaStream_t>(stream)));
    g_launches.fetch_add(g->kernel_nodes, std::memory_order_relaxed);
    return FSEM_OK;
}

extern "C" int fsem_graph_nodes(const fsem_graph_t* g) { return g ? g->kernel_nodes : 0; }
extern "C" int fsem_graph_slices(const fsem_graph_t* g) { return g ? g->slices : 0; }

extern "C" int fsem_graph_destroy(fsem_graph_t* g) {
    graph_free(g);
    return FSEM_OK;
}

// ================================================================================================
// SDR (SURVEY.md 8f rank 3): fast_se_metrics/SDR.py:52-97
// ================================================================================================
namespace {
// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
typedef CUresult (*TensorMapEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                      const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                      CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
TensorMapEncodeFn tensor_map_encoder() {
    static TensorMapEncodeFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return reinterpret_cast<TensorMapEncodeFn>(p);
    }();
    return fn;
}
// [item][row m][sample t] view of a [batch, stride] float buffer with rows of 128 samples that overlap (dim 0 is
// kTcMapDim0 wide): address = base + 4 t + 512 m + 4 stride item.  Boxes are box0 x 16 x 1.
bool make_sdr_tensor_map(CUtensorMap* map, const float* base, int64_t batch, int64_t n, int64_t stride, int box0) {
    TensorMapEncodeFn enc = tensor_map_encoder();
    if (!enc) return false;
    const int64_t rows = (n - kTcMapDim0) / kTcM + 1;             // rows whose widest box stays inside the item's n samples
    if (rows < kTcK) return false;
    const cuuint64_t gdim[3] = {(cuuint64_t)kTcMapDim0, (cuuint64_t)rows, (cuuint64_t)batch};
    const cuuint64_t gstride[2] = {(cuuint64_t)kTcM * sizeof(float), (cuuint64_t)stride * sizeof(float)};
    const cuuint32_t box[3] = {(cuuint32_t)box0, (cuuint32_t)kTcK, 1u};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), gdim, gstride, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
}  // namespace

namespace {
struct SdrPlan { int nsuper; size_t off_energy, off_partial, total; };
SdrPlan sdr_plan(int64_t batch, int64_t n) {
    SdrPlan p{};
    p.nsuper = (int)ceil_div(n > 0 ? n : 1, (int64_t)kSdrSuper * kSdrTile);
    size_t off = 0;
    p.off_energy = off;  off = align256(off + sizeof(double) * 2 * batch);
    p.off_partial = off; off = align256(off + sizeof(double) * batch * p.nsuper * 2 * kSdrLags);
    p.total = off;
    return p;
}
}  // namespace

extern "C" size_t fsem_sdr_workspace_bytes(int64_t batch, int64_t n) {
    if (batch <= 0 || n <= 0) return 0;
    return sdr_plan(batch, n).total;
}

extern "C" int fsem_sdr_score_f32(const fsem_batch_t* in, float* sdr_out, void* workspace, size_t workspace_bytes,
                                  void* stream_v) {
    if (!in || !sdr_out) return fail(FSEM_E_INVALID, "fsem_sdr_score_f32: null argument");
    if (int rc = check_batch("fsem_sdr_score_f32", in->clean, in->deg, in->batch, in->n, in->stride, 1, kMaxN, true))
        return rc == kEmptyBatch ? FSEM_OK : rc;
    if (in->batch > 65535) return fail(FSEM_E_INVALID, "fsem_sdr_score_f32: batch > 65535; split the batch");
    const SdrPlan p = sdr_plan(in->batch, in->n);
    if (!workspace || workspace_bytes < p.total)
        return fail(FSEM_E_WORKSPACE, "fsem_sdr_score_f32: workspace %zu < %zu bytes", workspace_bytes, p.total);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
    char* ws = static_cast<char*>(workspace);
    double* energy = reinterpret_cast<double*>(ws + p.off_energy);
    double* partial = reinterpret_cast<double*>(ws + p.off_partial);
    sdr_norm_kernel<<<(unsigned)(2 * in->batch), 256, 0, stream>>>(in->clean, in->deg, in->lengths, in->batch, in->n,
                                                                  in->stride, energy);
    FSEM_LAUNCHED();
    // correlation lags: tensor cores (tcgen05, fsem_sdr_tc.cuh) by default; FSEM_SDR_SIMT=1 selects the round-1 SIMT
    // kernel (kept for A/B measurements)
    static const bool simt = [] { const char* e = getenv("FSEM_SDR_SIMT"); return e && e[0] == '1'; }();
    int nsuper = p.nsuper;
    if (simt) {
        ProfScope prof_(K_SDR_CORR, stream);
        sdr_corr_kernel<<<dim3((unsigned)p.nsuper, (unsigned)in->batch), kSdrThreads, 0, stream>>>(
            in->clean, in->deg, in->lengths, in->batch, in->n, in->stride, p.nsuper, partial);
    } else {
        FSEM_CUDA(cudaFuncSetAttribute(sdr_corr_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTcDynSmem));
        // TMA tensor maps over the two signal buffers as [item][row of 128 samples, overlapping][sample]; they need
        // 16-byte aligned rows.  Otherwise (and for the last one or two k-steps of every item) the kernel reads global
        // memory directly.
        CUtensorMap map_a{}, map_bc{}, map_bd{};
        static const bool no_tma = [] { const char* e = getenv("FSEM_SDR_NO_TMA"); return e && e[0] == '1'; }();
        int use_tma = !no_tma && rows_vec4(in->clean, in->deg, in->stride, sizeof(float)) && in->n >= kTcMapDim0 ? 1 : 0;
        if (use_tma) {
            use_tma = make_sdr_tensor_map(&map_a, in->clean, in->batch, in->n, in->stride, kTcBoxA) &&
                      make_sdr_tensor_map(&map_bc, in->clean, in->batch, in->n, in->stride, kTcBoxB) &&
                      make_sdr_tensor_map(&map_bd, in->deg, in->batch, in->n, in->stride, kTcBoxB) ? 1 : 0;
        }
        nsuper = 1;
        ProfScope prof_(K_SDR_CORR, stream);
        sdr_corr_tc_kernel<<<(unsigned)(4 * in->batch), kTcThreads, kTcDynSmem, stream>>>(
            in->clean, in->deg, in->lengths, in->batch, in->n, in->stride, use_tma, map_a, map_bc, map_bd, partial);
    }
    FSEM_LAUNCHED();
    { ProfScope prof_(K_SDR_SOLVE, stream);
      sdr_solve_kernel<<<(unsigned)in->batch, kSdrSolveThreads, 0, stream>>>(partial, nsuper, energy, in->batch, sdr_out); }
    FSEM_LAUNCHED();
    return FSEM_OK;
}
