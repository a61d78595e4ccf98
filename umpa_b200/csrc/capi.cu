// capi.cu -- extern "C" boundary of libumpa_b200.so (see include/umpa_b200.h for the
// reference interface each entry point replaces).
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <chrono>
#include <memory>
#include <mutex>
#include <string>
#include <thread>

#include "common.cuh"

static thread_local char g_err[1024] = "";

void umpa_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

// Device-block cache: models are typically created once per projection with identical shapes
// (the reference's constructor is free, so callers do that).  Freed frame/scratch blocks are
// kept and handed to the next model instead of paying cudaMalloc/cudaFree (and their implicit
// device synchronisation) per model.  Bounded by UMPA_POOL_GB (default 64).
namespace {
struct PoolBlock { void *p; size_t bytes; int dev; };
std::mutex g_pool_mu;
std::vector<PoolBlock> g_pool;
size_t g_pool_bytes = 0;
// Cap of the cache: UMPA_POOL_GB, else a quarter of the device memory (so that the caller's own allocator --
// PyTorch's, another library's -- is not starved by idle blocks); umpa_pool_trim() empties it on demand.
size_t pool_cap()
{
    if (const char *e = getenv("UMPA_POOL_GB")) return (size_t)(atof(e) * (double)(1ull << 30));
    static size_t cap = 0;
    if (!cap) {
        size_t fr = 0, tot = 0;
        cap = cudaMemGetInfo(&fr, &tot) == cudaSuccess && tot ? tot / 4 : (size_t)32 << 30;
    }
    return cap;
}
}  // namespace

size_t pool_trim()
{
    std::lock_guard<std::mutex> lk(g_pool_mu);
    int cur = 0;
    cudaGetDevice(&cur);
    size_t freed = 0;
    for (auto &b : g_pool) { cudaSetDevice(b.dev); cudaFree(b.p); freed += b.bytes; }
    cudaSetDevice(cur);
    g_pool.clear(); g_pool_bytes = 0;
    return freed;
}

cudaError_t pool_malloc(void **p, size_t bytes)
{
    int dev = 0;
    cudaGetDevice(&dev);
    {
        std::lock_guard<std::mutex> lk(g_pool_mu);
        for (size_t n = 0; n < g_pool.size(); n++)
            if (g_pool[n].bytes == bytes && g_pool[n].dev == dev) {
                *p = g_pool[n].p;
                g_pool_bytes -= bytes;
                g_pool.erase(g_pool.begin() + n);
                return cudaSuccess;
            }
    }
    cudaError_t e = cudaMalloc(p, bytes);
    if (e != cudaSuccess) {                 // out of memory: drop the cache and retry once
        cudaGetLastError();
        pool_trim();
        e = cudaMalloc(p, bytes);
    }
    return e;
}

void pool_free(void *p, size_t bytes)
{
    if (!p) return;
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lk(g_pool_mu);
    if (bytes == 0 || g_pool_bytes + bytes > pool_cap()) { cudaFree(p); return; }
    g_pool.push_back({p, bytes, dev});
    g_pool_bytes += bytes;
}

// Pinned host chunks (16 KB) for the per-model constants, kept for the life of the process.
namespace {
constexpr size_t PIN_CHUNK = 16 * 1024;
std::mutex g_pin_mu;
std::vector<void *> g_pin_free;
// one set of non-blocking streams per device, shared by the models of the process
struct DevStreams { int dev; cudaStream_t s[3]; };
std::mutex g_stream_mu;
std::vector<DevStreams> g_streams;
}  // namespace

void *pinned_small_take(size_t bytes, bool *own)
{
    void *p = nullptr;
    if (bytes <= PIN_CHUNK) {
        *own = false;
        std::lock_guard<std::mutex> lk(g_pin_mu);
        if (!g_pin_free.empty()) { p = g_pin_free.back(); g_pin_free.pop_back(); return p; }
        return cudaHostAlloc(&p, PIN_CHUNK, cudaHostAllocDefault) == cudaSuccess ? p : nullptr;
    }
    *own = true;
    return cudaHostAlloc(&p, bytes, cudaHostAllocDefault) == cudaSuccess ? p : nullptr;
}

void pinned_small_give(void *p, bool own)
{
    if (!p) return;
    if (own) { cudaFreeHost(p); return; }
    std::lock_guard<std::mutex> lk(g_pin_mu);
    g_pin_free.push_back(p);
}

int scratch_reserve(umpa_model *m, Scratch &s, size_t bytes)
{
    if (s.bytes >= bytes && s.p) return UMPA_OK;
    if (s.p) {
        // kernels queued earlier (on any stream this model used) may still read the block
        if (m->last_ev_set) cudaEventSynchronize(m->last_ev);
        pool_free(s.p, s.bytes); m->dev_bytes -= (int64_t)s.bytes; s.p = nullptr; s.bytes = 0;
    }
    cudaError_t e = pool_malloc(&s.p, bytes);
    if (e != cudaSuccess) {
        umpa_set_error("cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
        s.p = nullptr;
        return UMPA_ERR_CUDA;
    }
    s.bytes = bytes;
    m->dev_bytes += (int64_t)bytes;
    return UMPA_OK;
}

namespace {

// Every entry point that takes a model runs on the model's device, whatever device is current in the calling
// thread (multi-GPU PyTorch code switches devices freely; __del__ may run under any of them), and restores it.
struct DeviceGuard {
    int prev = -1;
    bool switched = false;
    explicit DeviceGuard(const umpa_model *m)
    {
        if (m && cudaGetDevice(&prev) == cudaSuccess && prev != m->device) switched = cudaSetDevice(m->device) == cudaSuccess;
    }
    ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
};

// All launches of a model share its scratch (tables, aux images, constants, result buffer), so they are ordered:
// a call first makes its stream(s) wait for the event the previous call recorded on ITS stream, whichever that
// was -- match_device() on a torch stream followed by match() on the library's own streams, or two
// match_device() calls on different torch streams, no longer race -- and records its own at the end.
int order_after_last(umpa_model *m, cudaStream_t st)
{
    if (m->last_ev_set) UMPA_CUDA(cudaStreamWaitEvent(st, m->last_ev, 0));
    return UMPA_OK;
}
int record_last(umpa_model *m, cudaStream_t st)
{
    if (!m->last_ev) UMPA_CUDA(cudaEventCreateWithFlags(&m->last_ev, cudaEventDisableTiming));
    UMPA_CUDA(cudaEventRecord(m->last_ev, st));
    m->last_ev_set = true;
    return UMPA_OK;
}

// 400 * (A^T A)^-1 A^T for the quadratic basis [1,i,j,i^2,ij,j^2] on the 4x4 grid {-1..2}^2
// (i = row).  The entries are integers (UMPA/lib/Optim.cpp:169-174 lists them); they are
// derived here rather than typed in.
void quad_matrix(double *Q /*6x16*/)
{
    double A[16][6], N[6][12];
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++) {
            const double u = i - 1., v = j - 1.;
            const double row[6] = {1., u, v, u * u, u * v, v * v};
            memcpy(A[4 * i + j], row, sizeof(row));
        }
    for (int r = 0; r < 6; r++)
        for (int c = 0; c < 6; c++) {
            double s = 0.;
            for (int n = 0; n < 16; n++) s += A[n][r] * A[n][c];
            N[r][c] = s;
            N[r][6 + c] = (r == c) ? 1. : 0.;
        }
    for (int p = 0; p < 6; p++) {
        int best = p;
        for (int r = p + 1; r < 6; r++)
            if (fabs(N[r][p]) > fabs(N[best][p])) best = r;
        if (best != p)
            for (int c = 0; c < 12; c++) std::swap(N[p][c], N[best][c]);
        const double d = N[p][p];
        for (int c = 0; c < 12; c++) N[p][c] /= d;
        for (int r = 0; r < 6; r++)
            if (r != p) {
                const double f = N[r][p];
                for (int c = 0; c < 12; c++) N[r][c] -= f * N[p][c];
            }
    }
    for (int r = 0; r < 6; r++)
        for (int n = 0; n < 16; n++) {
            double s = 0.;
            for (int c = 0; c < 6; c++) s += N[r][6 + c] * A[n][c];
            Q[16 * r + n] = std::round(400. * s);
        }
}

// Arena layout (byte offsets; every array 256 B aligned).  The first part is fixed, the rest scales with Na.
constexpr size_t ARENA_QUAD = 0;                                             // 96 doubles
constexpr size_t ARENA_WIN = 1024;                                           // UMPA_MAX_K^2 doubles
constexpr size_t ARENA_G = ARENA_WIN + ((UMPA_MAX_K * UMPA_MAX_K * 8 + 255) & ~(size_t)255);
constexpr size_t ARENA_CONSTS = ARENA_G + 256;                               // 3 doubles
constexpr size_t ARENA_FIXED = ARENA_CONSTS + 256;
size_t arena_a256(size_t n) { return (n + 255) & ~(size_t)255; }

int arena_carve(umpa_model *m)
{
    const size_t Na = (size_t)m->Na;
    const size_t per[] = {2 * Na * 4, 2 * Na * 4,            // dim, pos
                          Na * 8, Na * 8, Na * 8,            // frame pointer tables
                          Na * 4, Na * 4, 2 * Na * 8,        // mean_s, mean_r, means64
                          2 * Na * 64 * 8};                  // partial sums (SUM_BLOCKS = 64)
    size_t need = ARENA_FIXED;
    for (size_t b : per) need += arena_a256(b);
    need = (need + 65535) & ~(size_t)65535;                  // few distinct sizes -> the cache hits
    UMPA_CUDA(pool_malloc((void **)&m->arena, need));
    m->arena_bytes = need;
    m->d_quad = (double *)(m->arena + ARENA_QUAD);
    m->d_consts = (double *)(m->arena + ARENA_CONSTS);
    char *p = m->arena + ARENA_FIXED;
    auto take = [&](size_t b) { char *r = p; p += arena_a256(b); return r; };
    m->d_dim = (int *)take(per[0]); m->d_pos = (int *)take(per[1]);
    m->d_sam_ptrs = (const double **)take(per[2]); m->d_ref_ptrs = (const double **)take(per[3]);
    m->d_mask_ptrs = (const double **)take(per[4]);
    m->d_mean_s = (float *)take(per[5]); m->d_mean_r = (float *)take(per[6]);
    m->d_means64 = (double *)take(per[7]); m->d_partials = (double *)take(per[8]);
    return UMPA_OK;
}

// window bookkeeping: copy, separability test (w == r c^T / total), device copies
int install_window(umpa_model *m, int Nw, const double *win)
{
    if (Nw < 0) { umpa_set_error("Nw must be non-negative."); return UMPA_ERR_ARG; }   // Model.cpp:242
    const int K = 2 * Nw + 1;
    m->Nw = Nw; m->K = K;
    m->win.assign(win, win + K * K);
    std::vector<double> r(K, 0.), c(K, 0.);
    double tot = 0., wmax = 0.;
    for (int a = 0; a < K; a++)
        for (int b = 0; b < K; b++) {
            r[a] += win[a * K + b]; c[b] += win[a * K + b]; tot += win[a * K + b];
            wmax = std::max(wmax, fabs(win[a * K + b]));
        }
    m->win_sum = tot;
    bool sep = tot != 0. && K <= UMPA_MAX_K;
    double asym = 0.;
    if (sep)
        for (int a = 0; a < K; a++) {
            asym = std::max(asym, fabs(r[a] - c[a]));
            for (int b = 0; b < K; b++)
                if (fabs(win[a * K + b] - r[a] * c[b] / tot) > 1e-13 * wmax) sep = false;
        }
    if (sep && asym > 1e-13 * fabs(tot)) sep = false;      // need the same factor on both axes
    m->separable = sep;
    m->g.assign(K, 0.);
    std::vector<float> gf(K, 0.f);
    if (sep)
        for (int a = 0; a < K; a++) { m->g[a] = r[a] / sqrt(fabs(tot)) * (tot < 0 ? -1. : 1.); gf[a] = (float)m->g[a]; }
    // g (x) g = r r^T / tot = win.  Its float copy sums to win_sum only to FP32 accuracy; the
    // walk divides by the FP64 sum of the *float* factor products where it matters (see table_path.cu).
    if (m->win_own) { cudaFree(m->d_win); cudaFree(m->d_g); m->win_own = false; }
    if (K <= UMPA_MAX_K) {                       // the arena holds a window of up to UMPA_MAX_K^2
        m->d_win = (double *)(m->arena + ARENA_WIN);
        m->d_g = (float *)(m->arena + ARENA_G);
    } else {
        m->d_win = nullptr; m->d_g = nullptr;
        UMPA_CUDA(cudaMalloc(&m->d_win, K * K * sizeof(double)));
        UMPA_CUDA(cudaMalloc(&m->d_g, K * sizeof(float)));
        m->win_own = true;
    }
    UMPA_CUDA(cudaMemcpy(m->d_win, win, K * K * sizeof(double), cudaMemcpyHostToDevice));
    UMPA_CUDA(cudaMemcpy(m->d_g, gf.data(), K * sizeof(float), cudaMemcpyHostToDevice));
    if (sep) {
        // the table path filters with the FP32 factor: use ITS exact sum as "sum of window"
        double gs = 0.;
        for (int a = 0; a < K; a++) gs += (double)gf[a];
        m->win_sum = gs * gs;
    }
    m->moments_valid = false;
    return UMPA_OK;
}

int make_roi(const umpa_model *m, const int32_t roi[6], const double uv0[2], RoiView *v)
{
    if (!roi) { umpa_set_error("roi is NULL"); return UMPA_ERR_ARG; }
    if (roi[2] < 1 || roi[5] < 1) { umpa_set_error("ROI steps must be >= 1"); return UMPA_ERR_ARG; }
    v->off0 = m->padding + roi[0]; v->step0 = roi[2];
    v->off1 = m->padding + roi[3]; v->step1 = roi[5];
    v->N0 = 1 + (roi[1] - roi[0] - 1) / roi[2];                 // model.pyx:414-415
    v->N1 = 1 + (roi[4] - roi[3] - 1) / roi[5];
    if (roi[1] <= roi[0]) v->N0 = 0;
    if (roi[4] <= roi[3]) v->N1 = 0;
    v->uv0[0] = uv0 ? uv0[0] : 0.; v->uv0[1] = uv0 ? uv0[1] : 0.;
    v->abc = nullptr; v->cover = nullptr; v->cover_threshold = 0.;
    v->dirty = nullptr; v->dirty_want = 0;
    return UMPA_OK;
}

// every pixel the ROI can touch must lie inside every frame the reference would read
int check_roi_bounds(const umpa_model *m, const RoiView &v)
{
    if (v.N0 <= 0 || v.N1 <= 0) return UMPA_OK;
    if (!m->uniform) return UMPA_OK;       // ragged frames: the reach test (Model.cpp:430-433) guards per frame
    const int reach = m->padding;          // max_shift + Nw + safe_crop
    const int i_lo = v.off0, i_hi = v.off0 + (v.N0 - 1) * v.step0;
    const int j_lo = v.off1, j_hi = v.off1 + (v.N1 - 1) * v.step1;
    if (i_lo - reach < 0 || i_hi + reach > m->H || j_lo - reach < 0 || j_hi + reach > m->W) {
        umpa_set_error("ROI rows [%d,%d] cols [%d,%d] (raw) reach outside the %dx%d frames (padding %d)",
                       i_lo, i_hi, j_lo, j_hi, m->H, m->W, reach);
        return UMPA_ERR_ARG;
    }
    return UMPA_OK;
}

void free_frames(umpa_model *m)
{
    const size_t b64 = m->stack_elems * sizeof(double);
    const size_t b32 = (size_t)m->Na * m->H * m->pitch * sizeof(float);
    pool_free(m->d_sam64, b64); pool_free(m->d_ref64, b64); pool_free(m->d_mask64, b64);
    pool_free(m->d_sam32, b32); pool_free(m->d_ref32, b32);
    m->h_sam.clear(); m->h_ref.clear(); m->h_mask.clear();
    m->h_sam_f.clear(); m->h_ref_f.clear(); m->h_mask_f.clear();
    m->host_f32 = false;
    m->maskbad_valid = false; m->mask_mode = 0;
    m->host_pending = false; m->fp64_missing = false;
    m->d_sam64 = m->d_ref64 = m->d_mask64 = nullptr;
    m->d_sam32 = m->d_ref32 = nullptr;
    m->frames_set = false;
}

int zero_outputs(const umpa_outputs &o, size_t n, cudaStream_t st)
{
    if (o.f) UMPA_CUDA(cudaMemsetAsync(o.f, 0, n * sizeof(double), st));
    if (o.T) UMPA_CUDA(cudaMemsetAsync(o.T, 0, n * sizeof(double), st));
    if (o.dx) UMPA_CUDA(cudaMemsetAsync(o.dx, 0, n * sizeof(double), st));
    if (o.dy) UMPA_CUDA(cudaMemsetAsync(o.dy, 0, n * sizeof(double), st));
    if (o.df) UMPA_CUDA(cudaMemsetAsync(o.df, 0, n * sizeof(double), st));
    if (o.err) UMPA_CUDA(cudaMemsetAsync(o.err, 0, n * sizeof(int32_t), st));
    if (o.ncalls) UMPA_CUDA(cudaMemsetAsync(o.ncalls, 0, n * sizeof(int32_t), st));
    if (o.debug_d) UMPA_CUDA(cudaMemsetAsync(o.debug_d, 0, 25 * n * sizeof(double), st));
    if (o.debug_a) UMPA_CUDA(cudaMemsetAsync(o.debug_a, 0, 16 * n * sizeof(double), st));
    return UMPA_OK;
}

// Centring constant of host frame f (sample frames 0..Na-1, then reference frames; hoststage.cu): the same value
// whether the frame then goes up in one piece, in bands, or partly converted.
double host_frame_mean(const umpa_model *m, int f)
{
    const int k = f < m->Na ? f : f - m->Na, fh = m->dim[2 * k], fw = m->dim[2 * k + 1];
    if (m->host_f32) return host_sampled_mean_f32(f < m->Na ? m->h_sam_f[k] : m->h_ref_f[k], fh, fw, table_row_step(fh));
    return host_sampled_mean(f < m->Na ? m->h_sam[k] : m->h_ref[k], fh, fw, table_row_step(fh));
}

// the constants of all 2 Na frames, by host threads
void host_means(const umpa_model *m, std::vector<double> &mu)
{
    const int Na = m->Na;
    mu.assign(2 * Na, 0.);
    std::atomic<int> next{0};
    auto work = [&]() {
        for (;;) {
            const int f = next.fetch_add(1);
            if (f >= 2 * Na) break;
            mu[f] = host_frame_mean(m, f);
        }
    };
    size_t samples = 0;                          // what the threads share: small jobs are not worth a thread start
    for (int k = 0; k < Na; k++) samples += (size_t)2 * ((m->dim[2 * k] + table_row_step(m->dim[2 * k]) - 1) / table_row_step(m->dim[2 * k])) * m->dim[2 * k + 1];
    const int want = (int)std::min<size_t>(8, samples / 1000000 + 1);
    const int nt = std::max(1, std::min(want, std::min(2 * Na, (int)std::thread::hardware_concurrency() - 1)));
    std::vector<std::thread> pool;
    for (int t = 1; t < nt; t++) pool.emplace_back(work);
    work();
    for (auto &t : pool) t.join();
}

__global__ void widen_kernel(double *dst, const float *src, size_t n)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) dst[i] = (double)src[i];
}

int widen_stack(double *dst, const float *src, size_t n, cudaStream_t st)
{
    widen_kernel<<<(unsigned)std::min<size_t>((n + 255) / 256, 148 * 16), 256, 0, st>>>(dst, src, n);
    UMPA_CUDA(cudaGetLastError());
    return UMPA_OK;
}

// Deferred host frames (umpa_set_frames on_device = 2): bring the FP64 stacks (and, if they are not
// there yet, the centred FP32 stacks) to the device now, on `st`.
int ensure_resident(umpa_model *m, cudaStream_t st)
{
    if (!m->host_pending && !m->fp64_missing) return UMPA_OK;
    double *dsts[3] = {m->d_sam64, m->d_ref64, m->d_mask64};
    float *tmp = nullptr;                        // float32 host frames: one stack at a time through a device buffer
    const size_t tmp_bytes = m->stack_elems * sizeof(float);
    if (m->host_f32) {
        UMPA_CUDA(pool_malloc((void **)&tmp, tmp_bytes));
        const std::vector<const float *> *srcs[3] = {&m->h_sam_f, &m->h_ref_f, &m->h_mask_f};
        for (int a = 0; a < 3; a++) {
            if (srcs[a]->empty()) continue;
            for (int k = 0; k < (int)srcs[a]->size(); k++) {
                const size_t n = (size_t)m->dim[2 * k] * m->dim[2 * k + 1];
                cudaError_t e = cudaMemcpyAsync(tmp + m->frame_off[k], (*srcs[a])[k], n * sizeof(float), cudaMemcpyHostToDevice, st);
                if (e != cudaSuccess) { cudaStreamSynchronize(st); pool_free(tmp, tmp_bytes); UMPA_CUDA(e); }
            }
            int rc = widen_stack(dsts[a], tmp, m->stack_elems, st);
            if (rc) { cudaStreamSynchronize(st); pool_free(tmp, tmp_bytes); return rc; }
        }
    } else {
        const std::vector<const double *> *srcs[3] = {&m->h_sam, &m->h_ref, &m->h_mask};
        for (int a = 0; a < 3; a++)
            for (int k = 0; k < (int)srcs[a]->size(); k++) {
                const size_t n = (size_t)m->dim[2 * k] * m->dim[2 * k + 1];
                UMPA_CUDA(cudaMemcpyAsync(dsts[a] + m->frame_off[k], (*srcs[a])[k], n * sizeof(double), cudaMemcpyHostToDevice, st));
            }
    }
    if (m->host_pending && (m->uniform || !m->masked)) {
        std::vector<double> mu;
        host_means(m, mu);
        int rc = table_alloc32(m);
        if (!rc) rc = table_set_means(m, mu.data(), st);
        if (!rc) rc = table_center_rows(m, 0, m->H, st);
        if (rc) { if (tmp) { cudaStreamSynchronize(st); pool_free(tmp, tmp_bytes); } return rc; }
    }
    cudaError_t se = cudaStreamSynchronize(st);
    if (tmp) pool_free(tmp, tmp_bytes);
    UMPA_CUDA(se);
    m->host_pending = false; m->fp64_missing = false;
    return UMPA_OK;
}

// the table paths read the centred FP32 stacks only
int ensure_fp32(umpa_model *m, cudaStream_t st) { return m->host_pending ? ensure_resident(m, st) : UMPA_OK; }

int ensure_streams(umpa_model *m)
{
    if (m->s_comp) return UMPA_OK;
    std::lock_guard<std::mutex> lk(g_stream_mu);
    for (auto &d : g_streams)
        if (d.dev == m->device) { m->s_copy = d.s[0]; m->s_comp = d.s[1]; m->s_out = d.s[2]; return UMPA_OK; }
    DevStreams d{m->device, {nullptr, nullptr, nullptr}};
    for (auto &st : d.s) UMPA_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    g_streams.push_back(d);
    m->s_copy = d.s[0]; m->s_comp = d.s[1]; m->s_out = d.s[2];
    return UMPA_OK;
}

// path selection + launch for one (sub-)ROI; everything is resident (or being streamed in by the caller)
int match_view(umpa_model *m, const RoiView &v, const umpa_outputs &out, cudaStream_t st, bool streaming = false)
{
    const size_t n = (size_t)v.N0 * v.N1;
    int rc;
    if (v.cover) { if ((rc = zero_outputs(out, n, st))) return rc; }
    else if (out.df && m->kind != UMPA_DF) UMPA_CUDA(cudaMemsetAsync(out.df, 0, n * sizeof(double), st));
    std::string why;
    bool use_table = false;
    if (m->path_opt != UMPA_PATH_LAZY && (m->masked || !m->uniform) && table_eligible(m, v, nullptr, true)) {
        // masks / ragged frames: table kernels on the pixels where they are exact, FP64 lazy evaluation elsewhere
        if ((rc = ensure_resident(m, st))) return rc;
        m->last_path = UMPA_PATH_MIXED;
        return mixed_match(m, v, out, st);
    }
    if (m->path_opt != UMPA_PATH_LAZY) {
        use_table = table_eligible(m, v, &why);
        if (!use_table && m->path_opt == UMPA_PATH_TABLE) {
            umpa_set_error("table path requested but not eligible: %s", why.c_str());
            return UMPA_ERR_UNSUPPORTED;
        }
    }
    if (use_table) {
        m->last_path = UMPA_PATH_TABLE;
        if (!streaming && (rc = ensure_fp32(m, st))) return rc;
        return table_match(m, v, out, st);
    }
    m->last_path = UMPA_PATH_LAZY;
    if ((rc = ensure_resident(m, st))) return rc;
    return lazy_match(m, v, out, st);
}

umpa_outputs offset_outputs(const umpa_outputs &o, size_t px)
{
    umpa_outputs r = o;
    if (r.f) r.f += px;
    if (r.T) r.T += px;
    if (r.dx) r.dx += px;
    if (r.dy) r.dy += px;
    if (r.df) r.df += px;
    if (r.err) r.err += px;
    if (r.ncalls) r.ncalls += px;
    if (r.debug_d) r.debug_d += 25 * px;
    if (r.debug_a) r.debug_a += 16 * px;
    return r;
}

// device -> host copies of `n` pixels of every requested map, asynchronous on `st`
int download_outputs(const umpa_outputs &host, const umpa_outputs &dev, size_t n, cudaStream_t st)
{
    auto back = [&](void *dst, const void *src, size_t bytes) -> cudaError_t {
        return (dst && src) ? cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st) : cudaSuccess;
    };
    UMPA_CUDA(back(host.f, dev.f, n * sizeof(double)));
    UMPA_CUDA(back(host.T, dev.T, n * sizeof(double)));
    UMPA_CUDA(back(host.dx, dev.dx, n * sizeof(double)));
    UMPA_CUDA(back(host.dy, dev.dy, n * sizeof(double)));
    UMPA_CUDA(back(host.df, dev.df, n * sizeof(double)));
    UMPA_CUDA(back(host.err, dev.err, n * sizeof(int32_t)));
    UMPA_CUDA(back(host.ncalls, dev.ncalls, n * sizeof(int32_t)));
    UMPA_CUDA(back(host.debug_d, dev.debug_d, 25 * n * sizeof(double)));
    UMPA_CUDA(back(host.debug_a, dev.debug_a, 16 * n * sizeof(double)));
    return UMPA_OK;
}

// Pinned FP32 staging for the rows the host converts (grow-only, shared by all models of the process).
// Pinning is slow (~0.3 ms per MB: config 2 needs ~0.8 GB), so it never happens inside a call: the first call that
// wants a bigger buffer than there is starts a builder thread and goes by plain DMA itself (no host conversion);
// the builder allocates page-aligned memory, touches it (no CUDA involved: most of the cost of pinning is faulting the
// pages in), registers it with CUDA in ONE piece (a 2-D copy must not span two registrations) and publishes it for the
// calls that follow.  UMPA_STAGE_SYNC=1 pins inside the call instead (tests, benchmarks of
// the steady state from the first call on).
struct HostStage {
    std::mutex mu;                  // held by a pipelined match for its whole duration; the builder publishes under it
    float *p = nullptr;
    size_t bytes = 0;
    bool registered = false;        // p came from the builder (aligned_alloc + cudaHostRegister), not from cudaHostAlloc
    std::atomic<bool> building{false};
} g_stage;

void stage_release_locked()
{
    if (!g_stage.p) return;
    if (g_stage.registered) { cudaHostUnregister(g_stage.p); free(g_stage.p); }
    else cudaFreeHost(g_stage.p);
    g_stage.p = nullptr; g_stage.bytes = 0; g_stage.registered = false;
}

void stage_builder(size_t bytes, int device)
{
    cudaSetDevice(device);
    bytes = (bytes + 4095) & ~(size_t)4095;
    char *q = (char *)aligned_alloc(4096, bytes);
    bool ok = q != nullptr;
    if (ok) {
        for (size_t o = 0; o < bytes; o += 4096) q[o] = 0;                // fault the pages in (first touch on this thread)
        ok = cudaHostRegister(q, bytes, cudaHostRegisterPortable) == cudaSuccess;
        if (!ok) { cudaGetLastError(); free(q); }
    }
    if (ok) {
        std::lock_guard<std::mutex> lk(g_stage.mu);                      // (waits for a match that is using the old buffer)
        if (g_stage.bytes < bytes) {
            stage_release_locked();
            g_stage.p = (float *)q; g_stage.bytes = bytes; g_stage.registered = true;
        } else {
            cudaHostUnregister(q);
            free(q);
        }
    }
    g_stage.building.store(false);
}

// Measured rates of the two sides of the pipelined upload (this process, exponential average): how
// fast the host threads convert while the DMA engine runs, and how fast the DMA engine moves FP64
// rows.  They set the share of rows the host converts in the next call, so the split follows the
// machine (cores and memory bandwidth left by other ranks / the caller) instead of a guess.
struct HostRates {
    std::mutex mu;
    double conv_gbs = 0., dma_gbs = 0.;          // while both run (0 = not measured yet)
    double dma_alone_gbs = 0.;                   // DMA engine with no conversion running (probed once)
} g_rates;

// do [lo, hi) lie inside one CUDA allocation (pinned host block)?  cuMemGetAddressRange through the runtime's
// driver entry point; "no" when it cannot be told.
bool same_allocation(const void *lo, const void *hi)
{
    typedef int (*RangeFn)(unsigned long long *, size_t *, unsigned long long);
    static RangeFn fn = []() -> RangeFn {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess) return nullptr;
        return (RangeFn)p;
    }();
    if (!fn) return false;
    unsigned long long base = 0;
    size_t size = 0;
    if (fn(&base, &size, (unsigned long long)(uintptr_t)lo) != 0) { cudaGetLastError(); return false; }
    return (unsigned long long)(uintptr_t)hi <= base + size;
}

// Byte distance between consecutive host frames (frame_bytes each) when they are equally spaced, without overlap,
// inside ONE pinned allocation -- a 2-D copy must not span two -- and 0 otherwise.
size_t frame_spacing(const std::vector<const void *> &f, size_t frame_bytes)
{
    if (f.size() < 2) return frame_bytes;
    const ptrdiff_t d = (const char *)f[1] - (const char *)f[0];
    if (d < (ptrdiff_t)frame_bytes) return 0;
    for (size_t k = 2; k < f.size(); k++)
        if ((const char *)f[k] - (const char *)f[k - 1] != d) return 0;
    return same_allocation(f[0], (const char *)f.back() + frame_bytes) ? (size_t)d : 0;
}

// Host -> device copy, on `st`, of rows [y0, y1) of Na frames, `width` bytes of each row.  Host frame k starts at
// src[k], or at src[0] + k * sstride when the frames lie in one pinned block (sstride > 0, see frame_spacing); it holds
// rows sy, sy + 1, ... spitch bytes apart.  Device frame k starts at dst + k * dstride, rows dpitch bytes apart.
// One 2-D copy covers all frames when the source is one block, the rows are contiguous on both sides and both strides
// are legal cudaMemcpy2D pitches (cudaDevAttrMaxPitch = 2^31 - 1 bytes); otherwise one copy per frame, a 2-D one
// when the rows are not contiguous.
cudaError_t upload_rows(void *dst, size_t dstride, size_t dpitch, const void *const *src, size_t sstride, size_t spitch,
                        int sy, size_t width, int Na, int y0, int y1, cudaStream_t st)
{
    const size_t max_pitch = ((size_t)1 << 31) - 1, rows = (size_t)(y1 - y0), soff = (size_t)(y0 - sy) * spitch;
    const bool packed = spitch == width && dpitch == width;
    char *d = (char *)dst + (size_t)y0 * dpitch;
    if (sstride > 0 && packed && sstride <= max_pitch && dstride <= max_pitch)
        return cudaMemcpy2DAsync(d, dstride, (const char *)src[0] + soff, sstride, rows * width, Na, cudaMemcpyHostToDevice, st);
    for (int k = 0; k < Na; k++, d += dstride) {
        const char *s = (sstride > 0 ? (const char *)src[0] + k * sstride : (const char *)src[k]) + soff;
        const cudaError_t e = packed ? cudaMemcpyAsync(d, s, rows * width, cudaMemcpyHostToDevice, st)
                                     : cudaMemcpy2DAsync(d, dpitch, s, spitch, width, rows, cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

int host_threads()
{
    if (const char *e = getenv("UMPA_HOST_THREADS")) return std::max(0, atoi(e));
    // default: leave a few cores to the caller; processes launched side by side (one rank per GPU:
    // torchrun exports LOCAL_WORLD_SIZE) share the box's cores
    int hw = (int)std::thread::hardware_concurrency(), ranks = 1;
    if (const char *e = getenv("LOCAL_WORLD_SIZE")) ranks = std::max(1, atoi(e));
    return std::max(0, std::min(12, hw / ranks - (ranks > 1 ? 2 : 4)));
}

// Row bands of a pipelined match: equal slices of the N0 output rows, the last one halved twice so that little
// work is left when the final rows arrive (kernels and download hide behind the upload).  UMPA_BANDS overrides.
std::vector<int> band_edges(int N0)
{
    std::vector<int> edge;
    int nu = std::max(1, std::min(10, N0 / 128));
    if (const char *e = getenv("UMPA_BANDS")) nu = std::max(1, std::min(N0, atoi(e)));
    const int rows_per = (N0 + nu - 1) / nu;
    for (int r = 0; r < N0; r += rows_per) edge.push_back(r);
    edge.push_back(N0);
    for (int split = 0; split < 2 && nu > 1; split++) {
        const int lo = edge[edge.size() - 2], hi = edge.back();
        if (hi - lo < 64) break;
        edge.insert(edge.end() - 1, lo + (hi - lo + 1) / 2);
    }
    return edge;
}

// The pipelined host-to-host match.  Frames still in host memory go up in row bands on a copy stream
// while the kernels of the previous band run and the maps of the band before that go back to the host.
// Band b needs input rows below off0 + step0*(r1-1) + padding only, so its kernels start as soon as
// those rows have landed.  Each band's new rows arrive in two parts, split at row Yc of every frame:
//  * direct rows (< Yc) cross PCIe in the frames' own element type.  Float64 rows land in the FP64 stacks
//    and are centred into the FP32 stacks (center_frames); float32 rows, half the bytes, land in the FP32
//    stacks and are centred where they lie (center_inplace).
//  * staged rows (>= Yc) are centred to FP32 by host threads into pinned staging (same arithmetic as
//    center_frames: FP64 subtract, one rounding) while the DMA engine is busy with the direct rows, and
//    then cross at FP32 size straight into the FP32 stacks.
// PCIe is the critical path (1.68 GB of FP64 for config 2 against ~4 ms of kernels), so for float64 frames
// the host threads shorten it by staging the lower rows; they also take the centring constants from the
// sampled rows.
// Pixels are independent: the result is the one the unpipelined path gives for the same constants.
int streamed_match(umpa_model *m, const RoiView &v, const umpa_outputs &dev, const umpa_outputs &host)
{
    const int Na = m->Na, H = m->H, W = m->W, pitch = m->pitch;
    const bool f32 = m->host_f32;
    const std::vector<int> edge = band_edges(v.N0);     // band b = output rows [edge[b], edge[b+1])
    const int nb = (int)edge.size() - 1;
    std::vector<int> need(nb);                  // band b needs input rows [0, need[b])
    for (int b = 0; b < nb; b++)
        need[b] = b == nb - 1 ? H : std::min(H, v.off0 + v.step0 * (edge[b + 1] - 1) + m->padding + 1);

    // direct rows: host stacks (sample, reference) -> FP64 stacks (float64 frames) or FP32 stacks (float32 frames)
    std::vector<const void *> src[2];
    if (f32) { src[0].assign(m->h_sam_f.begin(), m->h_sam_f.end()); src[1].assign(m->h_ref_f.begin(), m->h_ref_f.end()); }
    else { src[0].assign(m->h_sam.begin(), m->h_sam.end()); src[1].assign(m->h_ref.begin(), m->h_ref.end()); }
    void *const ddst[2] = {f32 ? (void *)m->d_sam32 : m->d_sam64, f32 ? (void *)m->d_ref32 : m->d_ref64};
    const size_t rowb = (size_t)W * (f32 ? sizeof(float) : sizeof(double));    // bytes of a host row
    const size_t drow = f32 ? (size_t)pitch * sizeof(float) : rowb;            // ... and of its device row
    const size_t srow = (size_t)pitch * sizeof(float);                          // a staged row, on both sides
    const size_t sstride[2] = {frame_spacing(src[0], (size_t)H * rowb), frame_spacing(src[1], (size_t)H * rowb)};
    cudaPointerAttributes pa{};
    const bool pinned = cudaPointerGetAttributes(&pa, src[0][0]) == cudaSuccess && pa.type != cudaMemoryTypeUnregistered;
    cudaGetLastError();

    // route: nthr host threads stage rows [Yc, H) of every frame.  Pageable frames would crawl through the driver's
    // own staging (measured: 80 ms for config 2 in float32), so the host stages all of their rows.
    int nthr = nb > 1 ? host_threads() : 0;
    int Yc = H;
    if (nthr > 0) {
        double x;                                       // share of the rows the host stages
        if (f32) {
            x = pinned ? 0. : 1.;                       // pinned float32 rows go up as they are, at the full DMA rate
        } else {
            // Which share x of the rows should the host convert?  Per input byte a converted row costs the
            // host memory system 2 bytes of traffic (read, write FP32, DMA read of the FP32) against 1 for a
            // row that goes up as FP64, and PCIe half a byte against one.  With M = B_conc + 1.5 R_conc the
            // memory bandwidth this process got while both sides ran, and B_alone the DMA rate with nobody
            // converting:   PCIe time (1 - x/2) D / B_alone  ==  memory time (1 + x) D / M
            //           =>  x = (M - B_alone) / (M/2 + B_alone).
            // On an idle host (B_conc = B_alone = B) this is the CPU balance x = 1 / (B/R + 1/2); when several
            // ranks saturate the host memory (measured: 2 ranks on one 24-vCPU box, DMA 53 -> 40 GB/s,
            // conversion 73 -> 36 GB/s) it backs off, down to plain DMA.
            double Ba, Bc, Rc;
            {
                std::lock_guard<std::mutex> lk(g_rates.mu);
                if (pinned && g_rates.dma_alone_gbs == 0.) {       // once per process: ~128 MB of real rows, nobody converting
                    const int pr = std::max(1, std::min(H, (int)(((size_t)128 << 20) / ((size_t)Na * rowb))));
                    cudaEvent_t e0 = nullptr, e1 = nullptr;
                    cudaEventCreate(&e0); cudaEventCreate(&e1);
                    cudaEventRecord(e0, m->s_copy);
                    upload_rows(m->d_sam64, (size_t)H * rowb, rowb, src[0].data(), sstride[0], rowb, 0, rowb, Na, 0, pr, m->s_copy);
                    cudaEventRecord(e1, m->s_copy);
                    float ms = 0.f;
                    if (cudaEventSynchronize(e1) == cudaSuccess && cudaEventElapsedTime(&ms, e0, e1) == cudaSuccess && ms > 0.f)
                        g_rates.dma_alone_gbs = (double)Na * pr * rowb / (ms * 1e-3) / 1e9;
                    cudaEventDestroy(e0); cudaEventDestroy(e1);
                    cudaGetLastError();
                }
                Ba = g_rates.dma_alone_gbs > 0. ? g_rates.dma_alone_gbs : 55.;
                Bc = g_rates.dma_gbs > 0. ? g_rates.dma_gbs : Ba;
                Rc = g_rates.conv_gbs > 0. ? g_rates.conv_gbs : std::min(85., 6.5 * nthr);
            }
            const double Mem = Bc + 1.5 * Rc;
            x = (Mem - Ba) / (.5 * Mem + Ba);
            if (x < .15) x = 0.;                               // not worth the threads
            x = std::min(x, .9);
            if (!pinned) x = 1.;
            if (const char *e = getenv("UMPA_HOST_FRAC")) x = atof(e);
            x = std::max(0., std::min(1., x));
        }
        Yc = H - (int)(x * H);
        if (Yc >= H) nthr = 0;
    }
    int HC = H - Yc;                            // staged rows per frame
    std::unique_lock<std::mutex> stage_lock(g_stage.mu, std::defer_lock);
    if (nthr > 0) {
        stage_lock.lock();
        const size_t want = (size_t)2 * Na * HC * srow;
        if (g_stage.bytes < want) {
            // room for every split the rate model may pick later (all rows when the frames are pageable)
            const size_t want_max = (size_t)2 * Na * H * srow;
            if (getenv("UMPA_STAGE_SYNC")) {
                stage_release_locked();
                if (cudaHostAlloc((void **)&g_stage.p, want_max, cudaHostAllocDefault) == cudaSuccess) g_stage.bytes = want_max;
                else cudaGetLastError();
            } else if (!g_stage.building.exchange(true)) {
                std::thread(stage_builder, want_max, m->device).detach();
            }
        }
        if (g_stage.bytes < want) {              // not pinned (yet): this call goes by plain DMA
            nthr = 0; Yc = H; HC = 0;
            stage_lock.unlock();
        }
    }

    // ---- host workers: constants first, then staging jobs in the order the bands need them ----
    struct Job { int band, stack, frame, y0, y1; };
    std::vector<Job> jobs;
    std::vector<int> cy0(nb, 0), cy1(nb, 0);    // staged rows that band b waits for: [cy0, cy1)
    {
        int hi = Yc;
        for (int b = 0; b < nb && nthr > 0; b++) {
            cy0[b] = hi; cy1[b] = std::max(hi, need[b]);
            hi = cy1[b];
            for (int k = 0; k < Na && cy1[b] > cy0[b]; k++)
                for (int a = 0; a < 2; a++) jobs.push_back({b, a, k, cy0[b], cy1[b]});
        }
    }
    std::vector<double> mu(2 * Na, 0.);      // centring constants (host_sampled_mean of every frame)
    std::unique_ptr<std::atomic<int>[]> left(new std::atomic<int>[nb]);
    for (int b = 0; b < nb; b++) left[b].store(nthr > 0 && cy1[b] > cy0[b] ? 2 * Na : 0);
    std::atomic<int> next_mean{0}, means_done{0}, next_job{0};
    std::atomic<bool> abort_flag{false};
    using clk = std::chrono::steady_clock;
    std::vector<clk::time_point> conv_t0(std::max(nthr, 1)), conv_t1(std::max(nthr, 1));
    auto worker = [&](int wid) {
        for (;;) {
            const int f = next_mean.fetch_add(1);
            if (f >= 2 * Na) break;
            mu[f] = host_frame_mean(m, f);
        }
        means_done.fetch_add(1, std::memory_order_acq_rel);
        while (means_done.load(std::memory_order_acquire) < nthr) std::this_thread::yield();
        conv_t0[wid] = conv_t1[wid] = clk::now();
        for (;;) {
            const int j = next_job.fetch_add(1);
            if (j >= (int)jobs.size() || abort_flag.load()) break;
            const Job &q = jobs[j];
            float *dst = g_stage.p + ((size_t)(q.stack * Na + q.frame) * HC + (q.y0 - Yc)) * pitch;
            const double c = mu[q.stack * Na + q.frame];
            const void *s = src[q.stack][q.frame];
            if (f32) host_center_rows_f32(dst, (const float *)s + (size_t)q.y0 * W, q.y1 - q.y0, W, pitch, c);
            else host_center_rows(dst, (const double *)s + (size_t)q.y0 * W, q.y1 - q.y0, W, pitch, c);
            left[q.band].fetch_sub(1, std::memory_order_acq_rel);
            conv_t1[wid] = clk::now();
        }
    };
    std::vector<std::thread> pool;
    for (int t = 0; t < nthr; t++) pool.emplace_back(worker, t);

    std::vector<cudaEvent_t> ev(2 * nb, nullptr);
    cudaEvent_t rate_ev[2] = {nullptr, nullptr}; // around the first band's FP64 rows: the DMA rate
    int rc = UMPA_OK;
    auto fail = [&](int code) {
        abort_flag.store(true);
        for (auto &t : pool) t.join();
        cudaStreamSynchronize(m->s_copy); cudaStreamSynchronize(m->s_comp); cudaStreamSynchronize(m->s_out);
        for (auto e : ev) if (e) cudaEventDestroy(e);
        for (auto e : rate_ev) if (e) cudaEventDestroy(e);
        return code;
    };
#define ST_CUDA(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { \
        umpa_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); return fail(UMPA_ERR_CUDA); } } while (0)
    for (auto &e : ev) ST_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    const bool trace = getenv("UMPA_STREAM_TRACE") != nullptr;     // timeline of the three streams on stderr
    std::vector<cudaEvent_t> tev;                // trace only: start, then per band: copy, comp, out
    auto mark = [&](cudaStream_t st) {
        if (!trace) return;
        cudaEvent_t e = nullptr;
        cudaEventCreate(&e);
        cudaEventRecord(e, st);
        tev.push_back(e);
    };
    if (trace) { cudaStreamSynchronize(m->s_copy); cudaStreamSynchronize(m->s_comp); }
    mark(m->s_copy);

    size_t rate_bytes = 0;
    if (nthr > 0) { cudaEventCreate(&rate_ev[0]); cudaEventCreate(&rate_ev[1]); cudaEventRecord(rate_ev[0], m->s_copy); }
    int up_hi = 0;                              // rows [0, up_hi) are on the device and centred
    bool have_means = false;
    int launches = 0;
    for (int b = 0; b < nb; b++) {
        const int r0 = edge[b], r1 = edge[b + 1];
        const int hi = std::max(up_hi, need[b]);
        const int d1 = std::min(hi, Yc), s0 = std::max(up_hi, Yc);     // direct rows [up_hi, d1), staged rows [s0, hi)
        if (d1 > up_hi) {
            for (int a = 0; a < 2; a++)
                ST_CUDA(upload_rows(ddst[a], (size_t)H * drow, drow, src[a].data(), sstride[a], rowb, 0, rowb, Na, up_hi, d1, m->s_copy));
            if (b == 0 && rate_ev[1]) { cudaEventRecord(rate_ev[1], m->s_copy); rate_bytes = (size_t)2 * Na * (d1 - up_hi) * rowb; }
        }
        if (!have_means) {                       // the first direct rows are on their way; now the constants
            if (nthr > 0) while (means_done.load(std::memory_order_acquire) < nthr) std::this_thread::yield();
            else host_means(m, mu);
            if ((rc = table_set_means(m, mu.data(), m->s_comp))) return fail(rc);
            have_means = true;
        }
        if (hi > s0) {
            while (left[b].load(std::memory_order_acquire) > 0) std::this_thread::yield();
            for (int a = 0; a < 2; a++) {
                const void *stage = g_stage.p + (size_t)a * Na * HC * pitch;     // stack a: frame k holds rows [Yc, H)
                ST_CUDA(upload_rows(a ? m->d_ref32 : m->d_sam32, (size_t)H * srow, srow, &stage, (size_t)HC * srow, srow, Yc, srow,
                                    Na, s0, hi, m->s_copy));
            }
        }
        ST_CUDA(cudaEventRecord(ev[2 * b], m->s_copy));
        mark(m->s_copy);
        ST_CUDA(cudaStreamWaitEvent(m->s_comp, ev[2 * b], 0));
        const int c1 = std::max(up_hi, d1);
        if ((rc = f32 ? table_center_rows_inplace(m, up_hi, c1, m->s_comp) : table_center_rows(m, up_hi, c1, m->s_comp))) return fail(rc);
        up_hi = hi;
        RoiView vb = v;
        vb.off0 = v.off0 + v.step0 * r0; vb.N0 = r1 - r0;
        const size_t px0 = (size_t)r0 * v.N1;
        if (v.abc) vb.abc = v.abc + 3 * px0;
        if (v.cover) vb.cover = v.cover + px0;
        const umpa_outputs db = offset_outputs(dev, px0);
        m->last_launches = 0;
        if ((rc = match_view(m, vb, db, m->s_comp, true))) return fail(rc);
        launches += m->last_launches;
        ST_CUDA(cudaEventRecord(ev[2 * b + 1], m->s_comp));
        mark(m->s_comp);
        ST_CUDA(cudaStreamWaitEvent(m->s_out, ev[2 * b + 1], 0));
        if ((rc = download_outputs(offset_outputs(host, px0), db, (size_t)(r1 - r0) * v.N1, m->s_out))) return fail(rc);
        mark(m->s_out);
    }
    m->last_launches = launches;
    for (auto &t : pool) t.join();
    pool.clear();
    ST_CUDA(cudaStreamSynchronize(m->s_out));
    ST_CUDA(cudaStreamSynchronize(m->s_comp));
    ST_CUDA(cudaStreamSynchronize(m->s_copy));
#undef ST_CUDA
    if (trace) {
        fprintf(stderr, "[umpa stream] %s frames, %d bands, %d host threads stage rows >= %d of %d\n",
                f32 ? "float32" : "float64", nb, nthr, Yc, H);
        for (int b = 0; b < nb; b++) {
            float tc = 0.f, tk = 0.f, to = 0.f;
            cudaEventElapsedTime(&tc, tev[0], tev[1 + 3 * b]);
            cudaEventElapsedTime(&tk, tev[0], tev[2 + 3 * b]);
            cudaEventElapsedTime(&to, tev[0], tev[3 + 3 * b]);
            fprintf(stderr, "[umpa stream] band %2d: uploaded %.2f  computed %.2f  downloaded %.2f ms\n", b, tc, tk, to);
        }
        for (auto e : tev) cudaEventDestroy(e);
    }
    for (auto e : ev) if (e) cudaEventDestroy(e);
    m->host_pending = false;
    m->fp64_missing = f32 || Yc < H;            // no FP64 copy of these rows on the device: ensure_resident makes one on demand
    if (nthr > 0 && !jobs.empty() && !f32) {    // update the measured rates
        clk::time_point a = conv_t0[0], z = conv_t1[0];
        for (int t = 1; t < nthr; t++) { a = std::min(a, conv_t0[t]); z = std::max(z, conv_t1[t]); }
        const double secs = std::chrono::duration<double>(z - a).count();
        const double conv = secs > 0. ? (double)2 * Na * HC * rowb / secs / 1e9 : 0.;
        float ms = 0.f;
        double dma = 0.;
        if (rate_bytes && cudaEventElapsedTime(&ms, rate_ev[0], rate_ev[1]) == cudaSuccess && ms > 0.f) dma = rate_bytes / (ms * 1e-3) / 1e9;
        std::lock_guard<std::mutex> lk(g_rates.mu);
        if (conv > 0.) g_rates.conv_gbs = g_rates.conv_gbs > 0. ? .5 * (g_rates.conv_gbs + conv) : conv;
        if (dma > 0.) g_rates.dma_gbs = g_rates.dma_gbs > 0. ? .5 * (g_rates.dma_gbs + dma) : dma;
        if (trace) fprintf(stderr, "[umpa stream] host conversion %.1f GB/s, DMA %.1f GB/s (averages %.1f / %.1f, DMA alone %.1f)\n",
                           conv, dma, g_rates.conv_gbs, g_rates.dma_gbs, g_rates.dma_alone_gbs);
    }
    for (auto e : rate_ev) if (e) cudaEventDestroy(e);
    m->stream_bands = nb; m->stream_threads = nthr; m->stream_host_rows = HC;
    return UMPA_OK;
}

}  // namespace

extern "C" {

const char *umpa_last_error(void) { return g_err; }
const char *umpa_version(void) { return "umpa_b200 0.1 (sm_100a)"; }

int umpa_create(umpa_model **out, int kind, int Na, const int32_t *dim, const int32_t *pos, int Nw,
                const double *win, int max_shift, int padding)
{
    if (!out || !dim || !win) { umpa_set_error("umpa_create: NULL argument"); return UMPA_ERR_ARG; }
    if (kind < UMPA_NODF || kind > UMPA_DFKERNEL) { umpa_set_error("umpa_create: unknown model kind %d", kind); return UMPA_ERR_ARG; }
    if (Na < 1) { umpa_set_error("umpa_create: Na must be >= 1"); return UMPA_ERR_ARG; }
    if (max_shift < 1 || padding < 0) { umpa_set_error("umpa_create: bad max_shift/padding"); return UMPA_ERR_ARG; }
    umpa_model *m = new (std::nothrow) umpa_model();
    if (!m) { umpa_set_error("out of host memory"); return UMPA_ERR_ARG; }
    m->kind = kind; m->Na = Na; m->max_shift = max_shift; m->padding = padding;
    cudaError_t e = cudaGetDevice(&m->device);
    if (e != cudaSuccess) { umpa_set_error("no CUDA device: %s", cudaGetErrorString(e)); delete m; return UMPA_ERR_CUDA; }
    cudaDeviceGetAttribute(&m->sm_count, cudaDevAttrMultiProcessorCount, m->device);
    m->dim.assign(dim, dim + 2 * Na);
    if (pos) m->pos.assign(pos, pos + 2 * Na); else m->pos.assign(2 * Na, 0);
    m->uniform = true;
    for (int k = 0; k < Na; k++) {
        if (m->dim[2 * k] < 1 || m->dim[2 * k + 1] < 1) { umpa_set_error("frame %d has an empty shape", k); delete m; return UMPA_ERR_ARG; }
        if (m->pos[2 * k] < 0 || m->pos[2 * k + 1] < 0) {
            umpa_set_error("Negative frame positions (entries in pos_list) are not allowed.");   // model.pyx:274-276
            delete m; return UMPA_ERR_ARG;
        }
        if (m->dim[2 * k] != m->dim[0] || m->dim[2 * k + 1] != m->dim[1] || m->pos[2 * k] || m->pos[2 * k + 1]) m->uniform = false;
    }
    m->H = m->dim[0]; m->W = m->dim[1];
    if (!m->uniform) {                          // canvas: the rectangle circumscribing all frames (model.pyx:531-549)
        m->H = m->W = 0;
        for (int k = 0; k < Na; k++) {
            m->H = std::max(m->H, m->pos[2 * k] + m->dim[2 * k]);
            m->W = std::max(m->W, m->pos[2 * k + 1] + m->dim[2 * k + 1]);
        }
    }
    int rc = arena_carve(m);
    if (rc) { umpa_destroy(m); return rc; }
    if ((rc = install_window(m, Nw, win))) { umpa_destroy(m); return rc; }
    double Q[96];
    quad_matrix(Q);
    cudaMemcpy(m->d_dim, m->dim.data(), 2 * Na * sizeof(int), cudaMemcpyHostToDevice);
    cudaMemcpy(m->d_pos, m->pos.data(), 2 * Na * sizeof(int), cudaMemcpyHostToDevice);
    cudaMemcpy(m->d_quad, Q, sizeof(Q), cudaMemcpyHostToDevice);
    *out = m;
    return UMPA_OK;
}

void umpa_destroy(umpa_model *m)
{
    if (!m) return;
    DeviceGuard dg(m);
    cudaDeviceSynchronize();      // (the model's device) blocks go back to the cache: nothing of this model may still be running
    free_frames(m);
    for (Scratch *s : {&m->filtA, &m->filtB, &m->auxS, &m->auxR, &m->tabX, &m->outbuf, &m->maskbad, &m->dirty, &m->maskbits, &m->maskflags, &m->maskwin, &m->fmImgS, &m->fmImgR, &m->fmS, &m->fmR, &m->fmA})
        if (s->p) pool_free(s->p, s->bytes);
    pinned_small_give(m->h_small, m->h_small_own);       // (the streams are shared per device and stay)
    if (m->win_own) { cudaFree(m->d_win); cudaFree(m->d_g); }
    if (m->arena) pool_free(m->arena, m->arena_bytes);
    for (int i = 0; i < 5; i++)
        if (m->ev[i]) cudaEventDestroy(m->ev[i]);
    if (m->last_ev) cudaEventDestroy(m->last_ev);
    delete m;
}

// device stacks + pointer tables for a new set of frames (shared by the float64 and float32 entry points)
static int alloc_frames(umpa_model *m, bool has_mask)
{
    if (m->last_ev_set) cudaEventSynchronize(m->last_ev);      // a match still in flight reads the old stacks
    free_frames(m);
    const int Na = m->Na;
    m->frame_off.assign(Na, 0);
    size_t total = 0;
    for (int k = 0; k < Na; k++) { m->frame_off[k] = total; total += (size_t)m->dim[2 * k] * m->dim[2 * k + 1]; }
    m->stack_elems = total;
    m->masked = has_mask;
    double **dsts[3] = {&m->d_sam64, &m->d_ref64, &m->d_mask64};
    const double ***ptrs[3] = {&m->d_sam_ptrs, &m->d_ref_ptrs, &m->d_mask_ptrs};
    for (int a = 0; a < 3; a++) {
        if (a == 2 && !has_mask) continue;
        UMPA_CUDA(pool_malloc((void **)dsts[a], total * sizeof(double)));
        std::vector<const double *> hp(Na);
        for (int k = 0; k < Na; k++) hp[k] = *dsts[a] + m->frame_off[k];
        UMPA_CUDA(cudaMemcpy((void *)*ptrs[a], hp.data(), Na * sizeof(double *), cudaMemcpyHostToDevice));
    }
    m->dev_bytes += (int64_t)(total * sizeof(double) * (has_mask ? 3 : 2));
    int rc = table_alloc32(m);
    if (rc) return rc;
    m->frames_set = true;
    return UMPA_OK;
}

int umpa_set_frames(umpa_model *m, const double *const *sam, const double *const *ref, const double *const *mask,
                    int on_device, void *stream)
{
    if (!m || !sam || !ref) { umpa_set_error("umpa_set_frames: NULL argument"); return UMPA_ERR_ARG; }
    if (on_device < 0 || on_device > 2) { umpa_set_error("umpa_set_frames: on_device must be 0, 1 or 2"); return UMPA_ERR_ARG; }
    DeviceGuard dg(m);
    cudaStream_t st = (cudaStream_t)stream;
    const int Na = m->Na;
    const double *const *srcs[3] = {sam, ref, mask};
    for (int a = 0; a < 3; a++)
        for (int k = 0; srcs[a] && k < Na; k++)
            if (!srcs[a][k]) { umpa_set_error("umpa_set_frames: frame %d is NULL", k); return UMPA_ERR_ARG; }
    int rc = alloc_frames(m, mask != nullptr);
    if (rc) return rc;
    if (on_device == 2) {                       // keep the host pointers; the first match uploads
        m->h_sam.assign(sam, sam + Na);
        m->h_ref.assign(ref, ref + Na);
        if (mask) m->h_mask.assign(mask, mask + Na);
        m->host_pending = true;
        return UMPA_OK;
    }
    const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    double *dsts[3] = {m->d_sam64, m->d_ref64, m->d_mask64};
    for (int a = 0; a < 3; a++)
        for (int k = 0; srcs[a] && k < Na; k++) {
            const size_t n = (size_t)m->dim[2 * k] * m->dim[2 * k + 1];
            UMPA_CUDA(cudaMemcpyAsync(dsts[a] + m->frame_off[k], srcs[a][k], n * sizeof(double), kind, st));
        }
    if ((rc = table_prepare_frames(m, st))) return rc;
    UMPA_CUDA(cudaStreamSynchronize(st));
    return UMPA_OK;
}

int umpa_set_frames_f32(umpa_model *m, const float *const *sam, const float *const *ref, const float *const *mask)
{
    if (!m || !sam || !ref) { umpa_set_error("umpa_set_frames_f32: NULL argument"); return UMPA_ERR_ARG; }
    DeviceGuard dg(m);
    const int Na = m->Na;
    const float *const *srcs[3] = {sam, ref, mask};
    for (int a = 0; a < 3; a++)
        for (int k = 0; srcs[a] && k < Na; k++)
            if (!srcs[a][k]) { umpa_set_error("umpa_set_frames_f32: frame %d is NULL", k); return UMPA_ERR_ARG; }
    int rc = alloc_frames(m, mask != nullptr);
    if (rc) return rc;
    m->h_sam_f.assign(sam, sam + Na);
    m->h_ref_f.assign(ref, ref + Na);
    if (mask) m->h_mask_f.assign(mask, mask + Na);
    m->host_f32 = true;
    m->host_pending = true;                     // the first match / cost / min uploads (umpa_set_frames, on_device = 2)
    return UMPA_OK;
}

int umpa_set_window(umpa_model *m, int Nw, const double *win)
{
    if (!m || !win) { umpa_set_error("umpa_set_window: NULL argument"); return UMPA_ERR_ARG; }
    DeviceGuard dg(m);
    if (m->last_ev_set) cudaEventSynchronize(m->last_ev);      // a match in flight still reads the old window
    return install_window(m, Nw, win);
}

int umpa_set_option(umpa_model *m, int option, int value)
{
    if (!m) { umpa_set_error("NULL model"); return UMPA_ERR_ARG; }
    switch (option) {
        case UMPA_OPT_SUBPX_FUNC: m->subpx = value; return UMPA_OK;
        case UMPA_OPT_REFERENCE_SHIFT: m->refshift = value ? 1 : 0; return UMPA_OK;
        case UMPA_OPT_PATH:
            if (value < UMPA_PATH_AUTO || value > UMPA_PATH_LAZY) { umpa_set_error("unknown path %d", value); return UMPA_ERR_ARG; }
            m->path_opt = value; return UMPA_OK;
    }
    umpa_set_error("unknown option %d", option);
    return UMPA_ERR_ARG;
}

int umpa_get_option(const umpa_model *m, int option, int *value)
{
    if (!m || !value) { umpa_set_error("NULL argument"); return UMPA_ERR_ARG; }
    switch (option) {
        case UMPA_OPT_SUBPX_FUNC: *value = m->subpx; return UMPA_OK;
        case UMPA_OPT_REFERENCE_SHIFT: *value = m->refshift; return UMPA_OK;
        case UMPA_OPT_PATH: *value = m->path_opt; return UMPA_OK;
    }
    umpa_set_error("unknown option %d", option);
    return UMPA_ERR_ARG;
}

int umpa_match(umpa_model *m, const int32_t roi[6], const double uv0[2], const double *abc, const double *cover,
               double cover_threshold, const umpa_outputs *out, void *stream)
{
    if (!m || !out) { umpa_set_error("umpa_match: NULL argument"); return UMPA_ERR_ARG; }
    if (!m->frames_set) { umpa_set_error("umpa_match: frames were not set"); return UMPA_ERR_STATE; }
    DeviceGuard dg(m);
    cudaStream_t st = (cudaStream_t)stream;
    RoiView v;
    int rc = make_roi(m, roi, uv0, &v);
    if (rc) return rc;
    m->last_launches = 0;
    m->ev_valid = false;
    if (v.N0 <= 0 || v.N1 <= 0) { m->last_path = 0; return UMPA_OK; }
    if ((rc = check_roi_bounds(m, v))) return rc;
    v.abc = abc; v.cover = cover; v.cover_threshold = cover_threshold;
    if (m->kind == UMPA_DFKERNEL && !abc) { umpa_set_error("abc array has to be provided"); return UMPA_ERR_ARG; }   // model.pyx:973-974
    if ((rc = order_after_last(m, st))) return rc;
    rc = match_view(m, v, *out, st);
    const int rr = record_last(m, st);             // also after a failure: whatever was queued still uses the scratch
    return rc ? rc : rr;
}

int umpa_match_host(umpa_model *m, const int32_t roi[6], const double uv0[2], const double *abc, const double *cover,
                    double cover_threshold, const umpa_outputs *out)
{
    if (!m || !out) { umpa_set_error("umpa_match_host: NULL argument"); return UMPA_ERR_ARG; }
    if (!m->frames_set) { umpa_set_error("umpa_match_host: frames were not set"); return UMPA_ERR_STATE; }
    DeviceGuard dg(m);
    RoiView v;
    int rc = make_roi(m, roi, uv0, &v);
    if (rc) return rc;
    m->last_launches = 0;
    m->ev_valid = false;
    if (v.N0 <= 0 || v.N1 <= 0) { m->last_path = 0; return UMPA_OK; }
    if ((rc = check_roi_bounds(m, v))) return rc;
    if (m->kind == UMPA_DFKERNEL && !abc) { umpa_set_error("abc array has to be provided"); return UMPA_ERR_ARG; }
    if ((rc = ensure_streams(m))) return rc;
    // the library's streams are shared by the models of the process and non-blocking: order them after this
    // model's last launch (e.g. a match_device() still running on a torch stream)
    for (cudaStream_t s : {m->s_copy, m->s_comp, m->s_out})
        if ((rc = order_after_last(m, s))) return rc;
    const size_t n = (size_t)v.N0 * v.N1;
    // one device block: f,T,dx,dy,df | debug_d | debug_a | abc | cover | err,ncalls
    const size_t nd = 5 * n + (out->debug_d ? 25 * n : 0) + (out->debug_a ? 16 * n : 0) + (abc ? 3 * n : 0) + (cover ? n : 0);
    if ((rc = scratch_reserve(m, m->outbuf, nd * sizeof(double) + 2 * n * sizeof(int32_t)))) return rc;
    double *p = (double *)m->outbuf.p;
    umpa_outputs d{};
    d.f = p; p += n; d.T = p; p += n; d.dx = p; p += n; d.dy = p; p += n; d.df = p; p += n;
    if (out->debug_d) { d.debug_d = p; p += 25 * n; }
    if (out->debug_a) { d.debug_a = p; p += 16 * n; }
    double *d_abc = nullptr, *d_cover = nullptr;
    if (abc) { d_abc = p; p += 3 * n; }
    if (cover) { d_cover = p; p += n; }
    d.err = (int32_t *)p; d.ncalls = d.err + n;
    if (abc) UMPA_CUDA(cudaMemcpyAsync(d_abc, abc, 3 * n * sizeof(double), cudaMemcpyHostToDevice, m->s_comp));
    if (cover) UMPA_CUDA(cudaMemcpyAsync(d_cover, cover, n * sizeof(double), cudaMemcpyHostToDevice, m->s_comp));
    v.abc = d_abc; v.cover = d_cover; v.cover_threshold = cover_threshold;

    // frames still on the host and the table path applies: pipeline upload / kernels / download
    if (m->host_pending && m->path_opt != UMPA_PATH_LAZY && !getenv("UMPA_NO_STREAMING") && table_eligible(m, v, nullptr)) {
        rc = streamed_match(m, v, d, *out);
        record_last(m, m->s_comp);                 // (it returns with its three streams drained)
        return rc;
    }
    rc = match_view(m, v, d, m->s_comp);
    if (!rc) rc = download_outputs(*out, d, n, m->s_comp);
    record_last(m, m->s_comp);
    cudaError_t e = cudaStreamSynchronize(m->s_comp);
    if (rc) return rc;
    if (e != cudaSuccess) { umpa_set_error("match failed on the device: %s", cudaGetErrorString(e)); return UMPA_ERR_CUDA; }
    return UMPA_OK;
}

int umpa_cost(umpa_model *m, int i, int j, int si, int sj, const double abc[3], double values[3], int *status)
{
    if (!m || !values) { umpa_set_error("umpa_cost: NULL argument"); return UMPA_ERR_ARG; }
    if (!m->frames_set) { umpa_set_error("umpa_cost: frames were not set"); return UMPA_ERR_STATE; }
    DeviceGuard dg(m);
    if (m->last_ev_set) cudaEventSynchronize(m->last_ev);
    if (int rc = ensure_resident(m, nullptr)) return rc;
    return lazy_cost(m, i, j, si, sj, abc, values, status);
}

int umpa_min(umpa_model *m, int i, int j, double *values, double uv[2], double dbg_d[25], double dbg_a[16],
             int *ncalls, int *ok)
{
    if (!m || !values || !uv) { umpa_set_error("umpa_min: NULL argument"); return UMPA_ERR_ARG; }
    if (!m->frames_set) { umpa_set_error("umpa_min: frames were not set"); return UMPA_ERR_STATE; }
    DeviceGuard dg(m);
    if (m->last_ev_set) cudaEventSynchronize(m->last_ev);
    if (int rc = ensure_resident(m, nullptr)) return rc;
    return lazy_min(m, i, j, values, uv, dbg_d, dbg_a, ncalls, ok);
}

int umpa_coverage(umpa_model *m, const int32_t roi[6], double *out, int on_device, void *stream)
{
    if (!m || !out) { umpa_set_error("umpa_coverage: NULL argument"); return UMPA_ERR_ARG; }
    if (!m->frames_set) { umpa_set_error("umpa_coverage: frames were not set"); return UMPA_ERR_STATE; }
    DeviceGuard dg(m);
    cudaStream_t st = (cudaStream_t)stream;
    RoiView v;
    int rc = make_roi(m, roi, nullptr, &v);
    if (rc) return rc;
    if ((rc = order_after_last(m, st))) return rc;
    if (m->masked && (rc = ensure_resident(m, st))) return rc;      // only the masked coverage reads frame data
    if (v.N0 <= 0 || v.N1 <= 0) return UMPA_OK;
    const size_t n = (size_t)v.N0 * v.N1;
    if (on_device) {
        rc = coverage_map(m, v, out, st);
        record_last(m, st);
        return rc;
    }
    double *d = nullptr;
    UMPA_CUDA(cudaMalloc(&d, n * sizeof(double)));
    rc = coverage_map(m, v, d, st);
    cudaError_t e = cudaSuccess;
    if (rc == UMPA_OK) {
        e = cudaMemcpyAsync(out, d, n * sizeof(double), cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    }
    cudaFree(d);
    if (e != cudaSuccess) { umpa_set_error("coverage failed: %s", cudaGetErrorString(e)); return UMPA_ERR_CUDA; }
    return rc;
}

int umpa_last_match_info(const umpa_model *m, int *path, int *kernel_launches)
{
    if (!m) { umpa_set_error("NULL model"); return UMPA_ERR_ARG; }
    if (path) *path = m->last_path;
    if (kernel_launches) *kernel_launches = m->last_launches;
    return UMPA_OK;
}

int umpa_last_stream_info(const umpa_model *m, int *bands, int *host_threads, int *host_rows)
{
    if (!m) { umpa_set_error("NULL model"); return UMPA_ERR_ARG; }
    if (bands) *bands = m->stream_bands;
    if (host_threads) *host_threads = m->stream_threads;
    if (host_rows) *host_rows = m->stream_host_rows;
    return UMPA_OK;
}

int umpa_set_profiling(umpa_model *m, int enable)
{
    if (!m) { umpa_set_error("NULL model"); return UMPA_ERR_ARG; }
    m->profiling = enable != 0;
    return UMPA_OK;
}

int umpa_last_stage_ms(umpa_model *m, float *ms, int n)
{
    if (!m || !ms) { umpa_set_error("NULL argument"); return UMPA_ERR_ARG; }
    if (!m->ev_valid) return 0;
    DeviceGuard dg(m);
    if (cudaEventSynchronize(m->ev[4]) != cudaSuccess) return 0;
    int k = 0;
    for (; k < 4 && k < n; k++) cudaEventElapsedTime(&ms[k], m->ev[k], m->ev[k + 1]);
    return k;
}

int64_t umpa_device_bytes(const umpa_model *m) { return m ? m->dev_bytes : 0; }

int64_t umpa_pool_trim(void) { return (int64_t)pool_trim(); }

}  // extern "C"

// ---------------------------------------------------------------------------------------
// FP32 FMA peak probe: dependent-free FFMA chains on every SM, timed with CUDA events.
// bench.py uses it as the measured denominator of the FP32-FMA roofline (SURVEY.md 8d).
namespace {
__global__ void __launch_bounds__(256) ffma_probe_kernel(float *sink, int iters, float x, float y)
{
    float a[16];
#pragma unroll
    for (int i = 0; i < 16; i++) a[i] = threadIdx.x * 1e-3f + i;
    for (int n = 0; n < iters; n++) {
#pragma unroll
        for (int u = 0; u < 8; u++)
#pragma unroll
            for (int i = 0; i < 16; i++) a[i] = fmaf(a[i], x, y);
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 16; i++) s += a[i];
    if (s == 123.456f) sink[0] = s;      // never true; keeps the chains alive
}
}  // namespace

extern "C" UMPA_API int umpa_fma_peak(double *tflops, int *sm_count)
{
    if (!tflops) { umpa_set_error("NULL argument"); return UMPA_ERR_ARG; }
    int dev = 0, sms = 0;
    UMPA_CUDA(cudaGetDevice(&dev));
    UMPA_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    float *sink = nullptr;
    UMPA_CUDA(cudaMalloc(&sink, sizeof(float)));
    cudaEvent_t e0, e1;
    UMPA_CUDA(cudaEventCreate(&e0));
    UMPA_CUDA(cudaEventCreate(&e1));
    const int iters = 4096, blocks = sms * 8, threads = 256;
    double best = 0.;
    for (int rep = 0; rep < 5; rep++) {
        UMPA_CUDA(cudaEventRecord(e0));
        ffma_probe_kernel<<<blocks, threads>>>(sink, iters, 0.999f, 1e-3f);
        UMPA_CUDA(cudaEventRecord(e1));
        UMPA_CUDA(cudaEventSynchronize(e1));
        float ms = 0.f;
        UMPA_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        const double flop = 2. * 16 * 8 * (double)iters * blocks * threads;
        if (rep > 0) best = std::max(best, flop / (ms * 1e-3) / 1e12);
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(sink);
    *tflops = best;
    if (sm_count) *sm_count = sms;
    return UMPA_OK;
}
