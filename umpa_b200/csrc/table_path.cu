// table_path.cu -- the fast CUDA path for .match(): UMPAModelNoDF / UMPAModelDF here, UMPAModelDFKernel
// through kernel_path.cu; masked models and ragged frames through mixed_match (bottom of this file).
//
// What the reference computes per pixel p and integer shift s (UMPA/lib/Model.cpp:359-509,
// 631-862; reference window moves: ia = i + shift, Model.cpp:415-421 / 695-701):
//     t1 = sum_k sum_u w(u) S_k(p+u)^2              t3 = sum_k sum_u w(u) R_k(p+s+u)^2
//     t5 = sum_k sum_u w(u) R_k(p+s+u) S_k(p+u)
//  DF: m_k = sum_u w R_k(p+s+u) / sum w,  t2 = sum_k m_k^2,  t6 = sum_k m_k sum_u w R_k(p+s+u),
//      t4 = sum_k m_k sum_u w S_k(p+u)
// and then a closed-form solve.  The reference evaluates this ~17 times per pixel with
// two (2Nw+1)^2 x Na gather loops each.  Here the same numbers come from an algebraic
// regrouping that removes the (2Nw+1)^2 factor from the shift-dependent work:
//   * the window sum is linear, so  t5(p,s) = [ w (*) C_s ](p)  with the UNWINDOWED
//     frame correlation  C_s(q) = sum_k R_k(q+s) S_k(q)  -- Na FMAs per (q,s) -- followed by
//     ONE separable Hamming filter per shift (2(2Nw+1) FMAs per (p,s));
//   * t4(p,s) = sum_k a_k(p+s) b_k(p) / sum w  with the per-frame filtered images
//     a_k = w (*) R_k, b_k = w (*) S_k  -- again Na FMAs per (p,s);
//   * t1 depends on p only, t2/t3/t6 on p+s only: they are images, computed once.
// Frames are stored centred in FP32 (x' = x - c_k, c_k = mean of the frame's sampled rows, FP64); the
// uncentred sums are rebuilt in FP64 from the centred ones plus four cheap cross images,
// so FP32 cancellation scales with the speckle variance instead of the mean squared.
// assign_coordinates = 'ref' swaps the roles of the stacks and negates the shift (TableEval<RS>).
// The per-pixel solve, the reference's integer walk (Optim.cpp:233-479) and the spline
// refinement run in FP64 on those tables (walk.cuh).
//
// Kernels (all sm_100a CUDA-core kernels; the path is a stencil/correlation, no GEMM):
//   frame_partial_sums / finish_means / center_frames   upload-time conversion
//   moments_kernel     a_k, b_k stacks + aux images                (HBM bound)
//   shift_table_kernel C_s + filter -> cross table;  a_k,b_k -> mean table (FP32 FMA / smem bound)
//   table_walk_kernel  FP64 solve + walk + spline per pixel
//   mask_rows_kernel / dirty_kernel / dirty_rect_kernel   which pixels of a masked / ragged model the
//                      table kernels may own (the rest goes to lazy_path.cu)
#include <cuda.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "shift_table.cuh"
#include "walk.cuh"

namespace {

using namespace shift_table;

// ------------------------------------------------------------------ frame conversion

constexpr int SUM_BLOCKS = 64;

// Centring constants.  Any constant close to the frame mean works (the identities that rebuild
// the uncentred sums hold for every c_k, d_k; only the FP32 cancellation depends on how close
// they are), so they are defined as the mean over the rows y = 0, step, 2 step, ... : those
// rows can be uploaded ahead of the rest (umpa_match_host pipelines the upload in row bands)
// and the result does not depend on how the upload was split.
// grid (SUM_BLOCKS, 2*Na): partial sums of the sampled rows of one FP64 frame (fixed order).
// Frames are addressed through the per-frame pointer / shape tables (they may be ragged).
__global__ void frame_partial_sums(const double *const *sam, const double *const *ref, const int *dim, int Na,
                                   double *partials)
{
    const int f = blockIdx.y, k = f < Na ? f : f - Na;
    const double *src = f < Na ? sam[k] : ref[k];
    const int H = dim[2 * k], W = dim[2 * k + 1], row_step = max(1, H / 32);     // table_row_step
    const int nrows = (H + row_step - 1) / row_step;
    double s = 0.;
    for (int r = blockIdx.x; r < nrows; r += SUM_BLOCKS) {
        const double *row = src + (size_t)r * row_step * W;
        for (int x = threadIdx.x; x < W; x += blockDim.x) {
            const double v = row[x];
            s += isfinite(v) ? v : 0.;             // a NaN / Inf pixel stays a local defect (hoststage.cu: finite_or_zero)
        }
    }
    __shared__ double red[256];
    red[threadIdx.x] = s;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) partials[(size_t)f * SUM_BLOCKS + blockIdx.x] = red[0];
}

// one block: constants of all 2*Na frames, then sum c_k d_k, sum c_k^2, sum d_k^2
__global__ void finish_means(const double *partials, const int *dim, int Na, double *means64, float *mean_s,
                             float *mean_r, double *consts)
{
    for (int f = threadIdx.x; f < 2 * Na; f += blockDim.x) {
        const int k = f < Na ? f : f - Na, H = dim[2 * k], W = dim[2 * k + 1], rs = max(1, H / 32);
        double s = 0.;
        for (int b = 0; b < SUM_BLOCKS; b++) s += partials[(size_t)f * SUM_BLOCKS + b];
        const double mu = s / ((double)((H + rs - 1) / rs) * W);
        means64[f] = mu;
        if (f < Na) mean_s[f] = (float)mu; else mean_r[f - Na] = (float)mu;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double cd = 0., cc = 0., dd = 0.;
        for (int k = 0; k < Na; k++) {
            const double d = means64[k], c = means64[Na + k];
            cd += c * d; cc += c * c; dd += d * d;
        }
        consts[0] = cd; consts[1] = cc; consts[2] = dd;
    }
}

// grid (ceil(pitch/256), y1-y0, 2*Na): rows [y0, y1) of the FP32 stacks, x' = (float)(x - c).
// The FP32 stacks live on the common canvas (H x pitch per frame): frame k covers rows
// [pos_k, pos_k + dim_k); outside its footprint the canvas holds the centred value of 0, so that a
// window that does not touch the frame contributes exactly nothing to the uncentred sums.
__global__ void center_frames(const double *const *sam, const double *const *ref, const int *dim, const int *pos,
                              const double *means64, int Na, int H, int pitch, int y0, float *sam32, float *ref32)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = y0 + blockIdx.y, f = blockIdx.z;
    if (x >= pitch) return;
    const bool is_s = f < Na;
    const int k = is_s ? f : f - Na;
    const int ly = y - pos[2 * k], lx = x - pos[2 * k + 1], fh = dim[2 * k], fw = dim[2 * k + 1];
    const double *src = is_s ? sam[k] : ref[k];
    float *dst = (is_s ? sam32 : ref32) + ((size_t)k * H + y) * pitch;
    const double v = (ly >= 0 && ly < fh && lx >= 0 && lx < fw) ? src[(size_t)ly * fw + lx] : 0.;
    dst[x] = (float)(v - means64[f]);
}

// float32 host frames (umpa_set_frames_f32) are copied raw into the FP32 stacks and centred where they lie:
// the same value as center_frames gives for the widened frame -- (float)((double)x - c) -- and (float)(0 - c)
// in the pitch padding.  Equal frames at position 0 only (the pipelined path).  grid (ceil(pitch/256), rows, 2*Na)
__global__ void center_inplace(const double *means64, int Na, int H, int W, int pitch, int y0, float *sam32, float *ref32)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = y0 + blockIdx.y, f = blockIdx.z;
    if (x >= pitch) return;
    float *row = (f < Na ? sam32 + ((size_t)f * H + y) * pitch : ref32 + ((size_t)(f - Na) * H + y) * pitch);
    const double v = x < W ? (double)row[x] : 0.;
    row[x] = (float)(v - means64[f]);
}

// ------------------------------------------------------------------ moments

// The aux images hold, per raw pixel q, everything of a cost evaluation that depends on ONE window position
// only, already rebuilt from the centred FP32 sums in FP64 (T3 = w (*) sum R'^2, P3 = sum c_k a'_k,
// U = sum d_k a'_k, M2 = sum a'_k^2, and T1, P1, V for the sample):
//     t3 = T3 + 2 P3 + sw sum c_k^2                  t1 = T1 + 2 P1 + sw sum d_k^2
//     t2 = M2/sw^2 + 2 P3/sw + sum c_k^2             (sum_k m_k^2, Model.cpp:770)
//     rden = 1/(t2 t3 - (sw t2)^2)  (DF: the determinant of the 2x2 solve, Model.cpp:849)  or 1/t3 (NoDF)
//     linq = U + sw sum c_k d_k
// so that an evaluation is one 32-byte gather + the two table entries, ~15 FP64 operations and no division.
struct __align__(16) AuxS { double t1, V; };
struct __align__(32) AuxR { double t3, t2, rden, linq; };

struct MomentsParams {
    const float *sam, *ref;      // centred stacks [Na][H][pitch]
    float *fa, *fb;              // filtered stacks a_k (from ref), b_k (from sam); nullptr for NoDF
    AuxS *auxS;                  // [H][pitch]: what a cost evaluation needs of the sample stack at a pixel
    AuxR *auxR;                  // [H][pitch]: ... and of the reference stack (see the structs above)
    const float *g;              // 1-D window factor, K
    const float *mean_s, *mean_r;
    const double *consts;        // device: sum_k c_k d_k, sum_k c_k^2, sum_k d_k^2
    double sw, inv_sw, inv_sw2;  // sum of the (FP32) window and its inverses
    int kind;
    int Na, Nw, H, W, pitch;
    int ty0, tx0;                // first tile (in tile units) of the bounding box
};

constexpr int MO_TH = 16, MO_TW = 64, MO_NT = 256, MO_FB = 2;     // MO_FB: frames per TMA box

// One block filters a 16 x 64 tile of every frame of both stacks with the separable window and
// accumulates the aux images.  Per frame:
//   * both raw tiles (with their Nw halo) arrive by TMA into a two-stage ring (box start 16 B aligned:
//     LPAD >= Nw columns are loaded left of the tile; zero fill outside the frame);
//   * row pass: an item is 4 consecutive outputs of one extended row, float4 in / float4 out, result to
//     a shared row buffer (the 8 lanes of a quarter warp cover one 128 B line: conflict free).  The raw
//     float4s an item loads anyway also feed the per-pixel sums of squares (each raw float4 is owned by exactly
//     one item: its first load, and for the items at the right edge their last one);
//   * column pass: the first four warps own the reference stack, the last four the sample stack; a thread owns
//     TWO vertically adjacent float4 of its stack's output tile, so the K+1 row-buffer lines they need are read
//     once (3 LDS.128 per output float4 instead of 5 for Nw = 2).  Its filtered values a'_k (or b'_k) go to the
//     filtered stacks and feed the aux accumulators of its own stack -- T3, P3, U, M2 belong to the reference,
//     T1, P1, V to the sample, so no thread needs the other stack's values.
// The sums of squares are filtered once at the end, as an extra "frame".
template <int NW>
__global__ void __launch_bounds__(MO_NT, 3)
moments_kernel(const __grid_constant__ CUtensorMap mapR, const __grid_constant__ CUtensorMap mapS, MomentsParams p)
{
    constexpr int K = 2 * NW + 1, ER = MO_TH + 2 * NW;
    constexpr int LPAD = (NW + 3) & ~3;                 // columns left of the tile in the TMA box
    constexpr int BW = MO_TW + 2 * LPAD, OFF = LPAD - NW;
    constexpr int NL4 = (OFF + 4 + 2 * NW + 3) / 4;     // float4 loads of one row-pass item
    constexpr int FR = ER * BW;                         // floats per raw frame tile (dense inside a TMA box)
    constexpr int RAW = ((MO_FB * FR * 4 + 127) & ~127) / 4; // floats per stack and ring stage: MO_FB frames (128 B multiple)
    constexpr int S4 = MO_TW / 4;                       // output strips per row
    constexpr int NROW = 2 * ER * S4;
    constexpr int RIT = (NROW + MO_NT - 1) / MO_NT;
    static_assert(S4 + NL4 - 1 == BW / 4, "the row-pass items of a row load every raw float4 of it");
    static_assert(MO_NT == 2 * (MO_TH / 2) * S4, "one thread per stack, row pair and strip");
    extern __shared__ __align__(128) float sm[];
    float *raw = sm;                                    // [2 stages][2 stacks][RAW]
    float *rowbuf = sm + 4 * RAW;                       // [2 stacks][ER][MO_TW]
    __shared__ uint64_t full_bar[2];
    const int tid = threadIdx.x;
    const int y0 = (blockIdx.y + p.ty0) * MO_TH, x0 = (blockIdx.x + p.tx0) * MO_TW;
    const size_t fstride = (size_t)p.H * p.pitch;
    float g[K];
#pragma unroll
    for (int v = 0; v < K; v++) g[v] = __ldg(p.g + v);

    if (tid == 0) {
        mbar_init(&full_bar[0], 1); mbar_init(&full_bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
    }
    __syncthreads();
    const int nbox = (p.Na + MO_FB - 1) / MO_FB;
    auto request = [&](int b) {                         // thread 0: frames [b MO_FB, +MO_FB) of both stacks -> stage b & 1
        float *dst = raw + (b & 1) * 2 * RAW;           // (one box per stack: a TMA box costs the same whatever its depth)
        mbar_expect_tx(&full_bar[b & 1], 2u * MO_FB * FR * sizeof(float));
        tma_load_3d(dst, &mapR, x0 - LPAD, y0 - NW, b * MO_FB, &full_bar[b & 1]);
        tma_load_3d(dst + RAW, &mapS, x0 - LPAD, y0 - NW, b * MO_FB, &full_bar[b & 1]);
    };
    if (tid == 0) { request(0); if (nbox > 1) request(1); }

    // sums of squares of the raw float4s this thread's row-pass items own: [item][first load | last load]
    float sq[RIT][2][4];
#pragma unroll
    for (int n = 0; n < RIT; n++)
#pragma unroll
        for (int h = 0; h < 2; h++)
#pragma unroll
            for (int x = 0; x < 4; x++) sq[n][h][x] = 0.f;

    // row pass of the two tiles at `in` (reference) and `in + RAW` (sample) -> rowbuf; SQ: also accumulate the squares
    auto row_pass = [&](const float *in, auto accumulate) {
        constexpr bool SQ = decltype(accumulate)::value;
#pragma unroll
        for (int n = 0; n < RIT; n++) {
            const int it = tid + n * MO_NT;
            if (it < NROW) {
                const int st = it / (ER * S4), rem = it - st * (ER * S4);
                const int er = rem / S4, c4 = rem - er * S4;
                const float *src = in + st * RAW + er * BW + 4 * c4;
                float r[4 * NL4];
#pragma unroll
                for (int v = 0; v < NL4; v++) {
                    const float4 t = *reinterpret_cast<const float4 *>(src + 4 * v);
                    r[4 * v] = t.x; r[4 * v + 1] = t.y; r[4 * v + 2] = t.z; r[4 * v + 3] = t.w;
                }
                if (SQ) {
#pragma unroll
                    for (int x = 0; x < 4; x++) sq[n][0][x] = fmaf(r[x], r[x], sq[n][0][x]);
                    if (NL4 > 1 && c4 >= S4 - (NL4 - 1)) {
#pragma unroll
                        for (int x = 0; x < 4; x++) sq[n][1][x] = fmaf(r[4 * (NL4 - 1) + x], r[4 * (NL4 - 1) + x], sq[n][1][x]);
                    }
                }
                float o[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int v = 0; v < K; v++)
#pragma unroll
                    for (int x = 0; x < 4; x++) o[x] = fmaf(g[v], r[OFF + x + v], o[x]);
                *reinterpret_cast<float4 *>(rowbuf + (st * ER + er) * MO_TW + 4 * c4) = make_float4(o[0], o[1], o[2], o[3]);
            }
        }
    };
    // column pass of this thread's two float4 (output rows 2 og, 2 og + 1, strip oc4) of its stack
    const int ost = tid >> 7, og = (tid & 127) / S4, oc4 = tid & (S4 - 1);
    auto col_pass = [&](float (&o)[2][4]) {
#pragma unroll
        for (int i = 0; i < 2; i++)
#pragma unroll
            for (int x = 0; x < 4; x++) o[i][x] = 0.f;
        const float *src = rowbuf + (ost * ER + 2 * og) * MO_TW + 4 * oc4;
#pragma unroll
        for (int u = 0; u <= K; u++) {
            const float4 t = *reinterpret_cast<const float4 *>(src + u * MO_TW);
            if (u < K) {
                o[0][0] = fmaf(g[u], t.x, o[0][0]); o[0][1] = fmaf(g[u], t.y, o[0][1]);
                o[0][2] = fmaf(g[u], t.z, o[0][2]); o[0][3] = fmaf(g[u], t.w, o[0][3]);
            }
            if (u > 0) {
                o[1][0] = fmaf(g[u - 1], t.x, o[1][0]); o[1][1] = fmaf(g[u - 1], t.y, o[1][1]);
                o[1][2] = fmaf(g[u - 1], t.z, o[1][2]); o[1][3] = fmaf(g[u - 1], t.w, o[1][3]);
            }
        }
    };

    // aux accumulators of this thread's stack: sum x^2 (M2), sum cA x (P3 | P1), sum cB x (U | V), with x = a'_k and
    // (cA, cB) = (c_k, d_k) for the reference stack, x = b'_k and (cA, cB) = (d_k, c_k) for the sample stack
    float a1[2][4], a2[2][4], a3[2][4];
#pragma unroll
    for (int i = 0; i < 2; i++)
#pragma unroll
        for (int x = 0; x < 4; x++) a1[i][x] = a2[i][x] = a3[i][x] = 0.f;
    const int oy = y0 + 2 * og, ox = x0 + 4 * oc4;
    const bool in0 = oy < p.H && ox < p.pitch, in1 = oy + 1 < p.H && ox < p.pitch;
    const size_t opix = (size_t)oy * p.pitch + ox;
    float *fdst = ost ? p.fb : p.fa;

    for (int k = 0; k < p.Na; k++) {
        const int box = k / MO_FB, fr = k - box * MO_FB;
        if (fr == 0) mbar_wait(&full_bar[box & 1], (box >> 1) & 1);
        const float *in = raw + (box & 1) * 2 * RAW + fr * FR;
        row_pass(in, std::true_type{});
        __syncthreads();                                 // row buffer complete; after a box's last frame its stage is consumed
        if (tid == 0 && (fr == MO_FB - 1 || k == p.Na - 1) && box + 2 < nbox) request(box + 2);
        float o[2][4];
        col_pass(o);
        const float ck = __ldg(p.mean_r + k), dk = __ldg(p.mean_s + k);
        const float cA = ost ? dk : ck, cB = ost ? ck : dk;
#pragma unroll
        for (int i = 0; i < 2; i++)
#pragma unroll
            for (int x = 0; x < 4; x++) {
                a1[i][x] = fmaf(o[i][x], o[i][x], a1[i][x]);
                a2[i][x] = fmaf(cA, o[i][x], a2[i][x]);
                a3[i][x] = fmaf(cB, o[i][x], a3[i][x]);
            }
        if (fdst) {
            if (in0) *reinterpret_cast<float4 *>(fdst + k * fstride + opix) = make_float4(o[0][0], o[0][1], o[0][2], o[0][3]);
            if (in1) *reinterpret_cast<float4 *>(fdst + k * fstride + opix + p.pitch) = make_float4(o[1][0], o[1][1], o[1][2], o[1][3]);
        }
        __syncthreads();                                 // row buffer free for the next frame
    }
    // the sums of squares as one more frame: T3 = w (*) sum_k R'^2, T1 = w (*) sum_k S'^2
#pragma unroll
    for (int n = 0; n < RIT; n++) {
        const int it = tid + n * MO_NT;
        if (it < NROW) {
            const int st = it / (ER * S4), rem = it - st * (ER * S4);
            const int er = rem / S4, c4 = rem - er * S4;
            float *dst = raw + st * RAW + er * BW + 4 * c4;
            *reinterpret_cast<float4 *>(dst) = make_float4(sq[n][0][0], sq[n][0][1], sq[n][0][2], sq[n][0][3]);
            if (NL4 > 1 && c4 >= S4 - (NL4 - 1))
                *reinterpret_cast<float4 *>(dst + 4 * (NL4 - 1)) = make_float4(sq[n][1][0], sq[n][1][1], sq[n][1][2], sq[n][1][3]);
        }
    }
    __syncthreads();
    row_pass(raw, std::false_type{});
    __syncthreads();
    float q[2][4];
    col_pass(q);
    const double cd = __ldg(p.consts), cc = __ldg(p.consts + 1), dd = __ldg(p.consts + 2);
#pragma unroll
    for (int i = 0; i < 2; i++) {
        if (!(i ? in1 : in0)) continue;
#pragma unroll
        for (int x = 0; x < 4; x++) {
            if (ost == 0) {                              // reference: q = T3, a1 = M2, a2 = P3, a3 = U
                AuxR r;
                r.t3 = (double)q[i][x] + 2. * (double)a2[i][x] + p.sw * cc;
                r.t2 = (double)a1[i][x] * p.inv_sw2 + 2. * (double)a2[i][x] * p.inv_sw + cc;
                const double t6 = p.sw * r.t2;
                r.rden = 1. / (p.kind == UMPA_DF ? r.t2 * r.t3 - t6 * t6 : r.t3);
                r.linq = (double)a3[i][x] + p.sw * cd;
                p.auxR[opix + i * p.pitch + x] = r;
            } else {                                     // sample: q = T1, a2 = P1, a3 = V
                p.auxS[opix + i * p.pitch + x] = AuxS{(double)q[i][x] + 2. * (double)a2[i][x] + p.sw * dd, (double)a3[i][x]};
            }
        }
    }
}

template <int NW> size_t moments_smem()
{
    constexpr int ER = MO_TH + 2 * NW, LPAD = (NW + 3) & ~3, BW = MO_TW + 2 * LPAD;
    return (size_t)4 * ((MO_FB * ER * BW * 4 + 127) & ~127) + (size_t)2 * ER * MO_TW * sizeof(float);
}

// ------------------------------------------------------------------ table-driven walk

struct WalkParams {
    const float *tabX;              // the tables: entry (row, shift, col) of the cross table at
                                    // tabX[row * row_stride + shift * tpitch + col], of the mean table (DF) m_off floats
                                    // further (shift_table.cuh: TableParams)
    size_t row_stride, m_off;
    unsigned tpitch;                // floats between consecutive shifts of one pixel
    const AuxS *auxS;               // [H][pitch], raw coordinates
    const AuxR *auxR;
    int pitch;
    int oy, ox;                     // raw coords of output pixel (0,0) of the dense region
    int dxX;                        // column of that pixel inside the cross table (TMA alignment shift)
    int Na, max_shift, subpx;
    double sw;                      // sum of window
    const double *consts;           // device: sum_k c_k d_k, c_k^2, d_k^2
    double inv_sw, inv_Na;
    const double *quad;
    const float *ktab;              // DFKernel: pixel-major rows [t5c(S^2) | t3c(S^2) | sigma-1] (kernel_path.cu)
    int kstride;                    // floats per row
    double swk;                     // exact sum of the FP32 2-D window kernel_path.cu applies
};

// One cost evaluation from the tables (the walk's functor).
// RS = reference_shift (assign_coordinates = 'ref', Model.cpp:408-421 / 688-701): the SAMPLE window
// moves by -s and the reference window stays at the pixel.  The tables are the same sums with the
// roles of the stacks swapped (table_match feeds the sample stack as the moving operand) and the shift
// negated; in the assembly the reference's aux record is then read at the pixel and the sample's at p - s.
// KIND is a template parameter so that no evaluation tests the model kind.
template <bool RS, int KIND>
struct TableEval {
    const WalkParams &w;
    AuxS ps;                        // sample record: at the pixel (!RS) -- or the last one fetched at p - s (RS)
    AuxR pr;                        // reference record: at the pixel (RS) -- or the last one fetched at p + s (!RS)
    const AuxS *pS;                 // RS: the sample's aux image at this pixel (shift 0)
    const AuxR *pR;                 // !RS: the reference's aux image at this pixel
    const float *pX;                // this pixel at shift 0 of the cross table (DFKernel: its table row)
    double sig, k5, k3;             // DFKernel: sigma, sigma swk sum c_k d_k, sigma^2 swk sum c_k^2

    __device__ __noinline__ static int out_of_bounds(int si, int sj, int ms)      // error_status bits of Model.cpp:654-681 (cold path)
    {
        if (si <= -ms || si >= ms) return UMPA_ST_BOUND;
        if (sj <= -ms) return UMPA_ST_BOUND | UMPA_ST_DIM;
        return UMPA_ST_BOUND | UMPA_ST_DIM | UMPA_ST_POS;
    }

    __device__ __forceinline__ int operator()(int si, int sj, double &cst, FitArgs &args)
    {
        const int ms = w.max_shift, S = 2 * ms - 1;
        const int ti = RS ? -si : si, tj = RS ? -sj : sj;
        const unsigned a = (unsigned)(ti + ms - 1), b = (unsigned)(tj + ms - 1);
        if (a >= (unsigned)S || b >= (unsigned)S) return out_of_bounds(si, sj, ms);
        const unsigned sidx = a * (unsigned)S + b;
        const int q = ti * w.pitch + tj;           // the moving window's pixel relative to this one
        if (KIND == UMPA_DFKERNEL) {
            // t3 = sum w B^2, t5 = sum w B S with B = k_p (*) R (Model.cpp:1076-1099), rebuilt from the
            // centred FP32 sums: B = B' + sigma c_k.  RS: t1 and the sample's V belong to p - s.
            const float x = __ldg(pX + sidx), m = __ldg(pX + S * S + sidx);
            if (RS) {
                const double2 v = __ldg(reinterpret_cast<const double2 *>(pS + q));
                ps.t1 = v.x; ps.V = v.y;
            }
            const double t5 = (double)x + sig * ps.V + k5;
            const double t3 = (double)m + k3;
            args.t = t5 / t3;
            cst = (ps.t1 - t5 * args.t) * w.inv_Na;
            return UMPA_ST_OK;
        }
        // the gathers of one evaluation: one aux record + one entry per table, a fixed distance apart
        const float *px = pX + (size_t)sidx * w.tpitch;
        const float x = __ldg(px);
        const float m = KIND == UMPA_DF ? __ldg(px + w.m_off) : 0.f;
        if (RS) {
            const double2 v = __ldg(reinterpret_cast<const double2 *>(pS + q));
            ps.t1 = v.x; ps.V = v.y;
        } else {
            const double2 v0 = __ldg(reinterpret_cast<const double2 *>(pR + q));
            const double2 v1 = __ldg(reinterpret_cast<const double2 *>(pR + q) + 1);
            pr.t3 = v0.x; pr.t2 = v0.y; pr.rden = v1.x; pr.linq = v1.y;
        }
        const double lin = pr.linq + ps.V;         // U + V + sw sum c_k d_k
        const double t5 = (double)x + lin;
        if (KIND == UMPA_DF) {
            const double t6 = w.sw * pr.t2;
            const double t4 = (double)m * w.inv_sw + lin;
            const double Kc = (pr.t2 * t5 - t4 * t6) * pr.rden;
            const double beta = (pr.t3 * t4 - t5 * t6) * pr.rden;
            args.t = beta + Kc;
            args.v = Kc;                           // dark field = Kc / t, divided once at the end
            // the reference's residual t1 + b^2 t2 + K^2 t3 - 2 b t4 - 2 K t5 + 2 b K t6 (Model.cpp:855-858) at the
            // solution of the normal equations (b t2 + K t6 = t4, b t6 + K t3 = t5) is t1 - b t4 - K t5
            cst = (ps.t1 - beta * t4 - Kc * t5) * w.inv_Na;
            return UMPA_ST_OK;
        }
        args.t = t5 * pr.rden;                     // NoDF: rden = 1 / t3
        cst = (ps.t1 - t5 * args.t) * w.inv_Na;
        return UMPA_ST_OK;
    }
};

constexpr int WALK_NT = 128;
#ifndef WALK_MINB
#define WALK_MINB 7
#endif

// d (the 5x5 cost cache) lives in shared memory, one column per thread: dynamic indexing
// without local-memory traffic.
struct SharedGrid {
    double *base;                   // &d_sm[0][threadIdx.x]
    __device__ __forceinline__ double &operator[](int n) const { return base[n * WALK_NT]; }
};

template <bool RS, int KIND>
__global__ void __launch_bounds__(WALK_NT, WALK_MINB) table_walk_kernel(WalkParams w, RoiView roi, umpa_outputs out)
{
    __shared__ double d_sm[25][WALK_NT];
    const int xj = blockIdx.x * blockDim.x + threadIdx.x;
    const int xi = blockIdx.y;
    if (xj >= roi.N1 || xi >= roi.N0) return;
    const size_t n = (size_t)xi * roi.N1 + xj;
    if (roi.cover && roi.cover[n] < roi.cover_threshold) return;
    if (roi.dirty && (roi.dirty[n] != 0) != (roi.dirty_want != 0)) return;   // mixed path: the lazy kernel owns this pixel
    const int ty = roi.step0 * xi, tx = roi.step1 * xj;
    const size_t pix = (size_t)(w.oy + ty) * w.pitch + (w.ox + tx);
    TableEval<RS, KIND> eval{w};
    eval.pS = w.auxS + pix; eval.pR = w.auxR + pix;
    if (RS) {
        const double2 v0 = __ldg(reinterpret_cast<const double2 *>(eval.pR));
        const double2 v1 = __ldg(reinterpret_cast<const double2 *>(eval.pR) + 1);
        eval.pr = AuxR{v0.x, v0.y, v1.x, v1.y};
        eval.ps = AuxS{0., 0.};
    } else {
        const double2 v = __ldg(reinterpret_cast<const double2 *>(eval.pS));
        eval.ps = AuxS{v.x, v.y};
        eval.pr = AuxR{0., 0., 0., 0.};
    }
    eval.sig = eval.k5 = eval.k3 = 0.;
    if (KIND == UMPA_DFKERNEL) {
        const int S = 2 * w.max_shift - 1;
        eval.pX = w.ktab + n * (size_t)w.kstride;
        eval.sig = 1. + (double)__ldg(eval.pX + 2 * S * S);
        eval.k5 = eval.sig * w.swk * __ldg(w.consts);
        eval.k3 = eval.sig * eval.sig * w.swk * __ldg(w.consts + 1);
    } else {
        eval.pX = w.tabX + (size_t)ty * w.row_stride + tx + w.dxX;
    }
    FitArgs args{0., 0.};
    SharedGrid d{&d_sm[0][threadIdx.x]};
    double uv[2] = {roi.uv0[0], roi.uv0[1]}, f = 0.;
    int ncalls;
    WalkState ws;
    const int st = walk_search(eval, args, f, uv, d, ncalls, ws);
    store_debug(out, n, d, ws);                    // (before the fit: it reuses the cache's cells)
    if (ws.finished) walk_refine(w.subpx, w.quad, d, ws, f, uv);
    if (KIND == UMPA_DF && args.t != 0.) args.v = args.v / args.t;
    store_pixel(out, n, KIND, st, f, args, uv, ncalls);
}

template <bool RS>
void launch_walk(int kind, dim3 grid, const WalkParams &w, const RoiView &roi, const umpa_outputs &out, cudaStream_t st)
{
    if (kind == UMPA_DF) table_walk_kernel<RS, UMPA_DF><<<grid, WALK_NT, 0, st>>>(w, roi, out);
    else if (kind == UMPA_NODF) table_walk_kernel<RS, UMPA_NODF><<<grid, WALK_NT, 0, st>>>(w, roi, out);
    else table_walk_kernel<RS, UMPA_DFKERNEL><<<grid, WALK_NT, 0, st>>>(w, roi, out);
}

// ------------------------------------------------------------------ host side

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn()
{
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

// 3-D map over a stack [Na][H][pitch] of floats, box (bw, bh, 1), zero fill outside [0,W)x[0,H)
int make_stack_map(CUtensorMap *map, const float *base, int Na, int H, int W, int pitch, int bw, int bh, int bd = 1)
{
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) { umpa_set_error("cuTensorMapEncodeTiled is not available from the driver"); return UMPA_ERR_CUDA; }
    const cuuint64_t dims[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)Na};
    const cuuint64_t strides[2] = {(cuuint64_t)pitch * sizeof(float), (cuuint64_t)pitch * H * sizeof(float)};
    const cuuint32_t box[3] = {(cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)bd};
    const cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void *)base, dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        umpa_set_error("cuTensorMapEncodeTiled failed (%d) for W=%d H=%d Na=%d pitch=%d box=%dx%d", (int)r, W, H, Na, pitch, bw, bh);
        return UMPA_ERR_CUDA;
    }
    return UMPA_OK;
}

template <int NW>
int launch_moments_nw(const MomentsParams &mp, const float *ref32, const float *sam32, dim3 grid, cudaStream_t st)
{
    constexpr int ER = MO_TH + 2 * NW, LPAD = (NW + 3) & ~3, BW = MO_TW + 2 * LPAD;
    CUtensorMap mr, ms;
    int rc;
    if ((rc = make_stack_map(&mr, ref32, mp.Na, mp.H, mp.W, mp.pitch, BW, ER, MO_FB))) return rc;
    if ((rc = make_stack_map(&ms, sam32, mp.Na, mp.H, mp.W, mp.pitch, BW, ER, MO_FB))) return rc;
    const size_t smem = moments_smem<NW>();
    UMPA_CUDA(cudaFuncSetAttribute(moments_kernel<NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    moments_kernel<NW><<<grid, MO_NT, smem, st>>>(mr, ms, mp);
    UMPA_CUDA(cudaGetLastError());
    return UMPA_OK;
}

int launch_moments(int Nw, const MomentsParams &mp, const float *ref32, const float *sam32, dim3 grid, cudaStream_t st)
{
    switch (Nw) {
        case 0: return launch_moments_nw<0>(mp, ref32, sam32, grid, st);
        case 1: return launch_moments_nw<1>(mp, ref32, sam32, grid, st);
        case 2: return launch_moments_nw<2>(mp, ref32, sam32, grid, st);
        case 3: return launch_moments_nw<3>(mp, ref32, sam32, grid, st);
        case 4: return launch_moments_nw<4>(mp, ref32, sam32, grid, st);
        case 5: return launch_moments_nw<5>(mp, ref32, sam32, grid, st);
        case 6: return launch_moments_nw<6>(mp, ref32, sam32, grid, st);
    }
    umpa_set_error("table path: Nw %d not instantiated", Nw);
    return UMPA_ERR_UNSUPPORTED;
}

// filter = false: plain table; true: window filter of half-width p.Nw (0..6)
int dispatch_shift_table(bool filter, int S, const CUtensorMap &a, const CUtensorMap &b, const TableParams &p, dim3 grid,
                         int nt, size_t smem, cudaStream_t st)
{
    if (!filter) return shift_table_launch_plain(S, a, b, p, grid, nt, smem, st);
    switch (p.Nw) {
        case 0: return shift_table_launch_nw0(S, a, b, p, grid, nt, smem, st);
        case 1: return shift_table_launch_nw1(S, a, b, p, grid, nt, smem, st);
        case 2: return shift_table_launch_nw2(S, a, b, p, grid, nt, smem, st);
        case 3: return shift_table_launch_nw3(S, a, b, p, grid, nt, smem, st);
        case 4: return shift_table_launch_nw4(S, a, b, p, grid, nt, smem, st);
        case 5: return shift_table_launch_nw5(S, a, b, p, grid, nt, smem, st);
        case 6: return shift_table_launch_nw6(S, a, b, p, grid, nt, smem, st);
    }
    umpa_set_error("table path: Nw %d not instantiated", p.Nw);
    return UMPA_ERR_UNSUPPORTED;
}

int row_block_of(int S) { return S <= 9 ? 3 : (S <= 17 ? 2 : 1); }

int ctas_per_sm() { const char *e = getenv("UMPA_TAB_CTAS"); return e ? std::max(1, atoi(e)) : 1; }

// Geometry of one table kernel: chunk height, warp groups, frame ring, and how the table is cut into items (column
// strips x row segments, shift_table.cuh).  Returns dynamic smem bytes (0 = unsupported) and the block size.
size_t plan_tiles(TableParams &p, int S, bool filter, int *nt, int rows, int cols, int ctas, int ctas_sm)
{
    const int HS = (S - 1) / 2, halo = filter ? p.Nw : 0, H2 = 2 * halo;
    const int delta = (4 - HS % 4) % 4;
    const int NA4 = (delta + S + 3 + 3) / 4, SH = row_block_of(S);
    p.TW = (EXT_W - H2) & ~3;
    if (p.TW < 8) return 0;
    p.rows = rows;
    p.nstrips = (cols + p.TW - 1) / p.TW;
    p.cols_p = p.nstrips * p.TW;
    p.AP = EXT_W - 4 + 4 * NA4;
    auto up32 = [](int floats) { return (floats + 31) & ~31; };      // 128 B
    const size_t budget = SMEM_CAP / ctas_sm - 2048;           // (shared memory per SM: 228 KB, 1 KB reserved per CTA)
    const int max_nt = ctas_sm > 1 ? (MAX_NT / ctas_sm) & ~31 : MAX_NT;  // registers: 168 per thread for MAX_NT threads per SM
    // Candidates: chunk height EH (a tall chunk leaves room for fewer warp groups, i.e. more passes over the
    // frames) x streaming or not.  STREAMING keeps the last 2*halo row-filtered rows of the shift planes in shared
    // memory for the next chunk of the segment, so no chunk row is wasted on the window halo; without it every
    // segment is one chunk and EH - 2*halo of its EH rows are outputs.  Two streaming orders: chunk-major (1: all
    // passes of a chunk before the next chunk, carry = all S*S planes) and pass-major (2: all chunks of the segment
    // before the next pass, carry = the G*SH*S planes of one pass -- what fits when S = 15).  Cost model fitted to
    // measurements: rows computed per useful row; shift rows covered per shift row of the table (S = 15: 3 passes
    // of 3 groups cover 18, 4 passes of 2 groups 16 -- config 4 cross table 21.06 vs 20.49 ms); +5 % per extra pass
    // over the frames; the TMA box cost (a box takes the same TMA time whatever its depth FB; config 2, FB 1 / 2 /
    // 5 / 9 -> 1.51 / 1.22 / 1.08 / 1.04 ms ~ 1 + 0.5 / FB); pass-major +5 % (config 2, where both orders fit:
    // 0.957 vs 0.872 ms).
    double best = 1e30;
    TableParams bp = p;
    size_t best_smem = 0;
    const char *e_eh = getenv("UMPA_TAB_EH"), *e_st = getenv("UMPA_TAB_STREAM"), *e_fb = getenv("UMPA_TAB_FB"), *e_g = getenv("UMPA_TAB_G");
    for (int eh : {8, 16, 24, 32, 48})
        for (int stream = (filter && halo > 0) ? 2 : 0; stream >= 0; stream--) {     // 2: streaming, pass-major (see below)
            if (e_eh ? atoi(e_eh) != eh : (eh == 8) != (ctas_sm > 1)) continue;     // 8-row chunks: two CTAs per SM only
            if (e_st && filter && halo > 0 && atoi(e_st) != stream) continue;
            if (!stream && eh - H2 < 2) continue;
            // the carry of a chunk is its last 2*halo rows: a shorter chunk would leave carry rows unwritten that the
            // next chunk's column pass reads (8-row chunks of UMPA_TAB_CTAS=2 / UMPA_TAB_EH=8 with Nw 5, 6)
            if (stream && eh < H2) continue;
            TableParams q = p;
            q.EH = eh;
            q.G = std::min(max_nt / (eh * 8), (S + SH - 1) / SH);
            if (e_g) q.G = std::max(1, std::min(q.G, atoi(e_g)));
            if (q.G < 1) continue;
            q.npass = (S + q.G * SH - 1) / (q.G * SH);
            q.AH = eh + 2 * HS;
            const size_t cbuf = filter ? (size_t)q.G * S * eh * EXT_W * sizeof(float) : 0;
            // carry: all S*S planes, or (pass-major order, stream == 2) only the G*SH*S planes of one pass
            if (stream == 2 && (q.npass == 1 || S < 11)) continue;       // (the S <= 9 kernels are compiled without it)
            const size_t carry = stream == 1 ? (size_t)S * S * H2 * EXT_W * sizeof(float)
                               : stream == 2 ? (size_t)q.G * SH * S * H2 * EXT_W * sizeof(float) : 0;
            if (cbuf + carry >= budget) continue;
            // frames per TMA box = per ring stage: the fewest boxes of at most 9 frames, as long as 3 stages fit (2 at least)
            const int nboxes = (p.Na + 8) / 9;
            q.FB = (p.Na + nboxes - 1) / nboxes;
            if (e_fb) q.FB = std::max(1, std::min(32, atoi(e_fb)));
            q.FB = std::max(1, std::min(q.FB, p.Na));
            int ns = 0;
            for (;; q.FB--) {
                q.a_stage_floats = up32(q.FB * q.AH * q.AP);
                q.stage_floats = q.a_stage_floats + up32(q.FB * eh * EXT_W);
                ns = (int)((budget - cbuf - carry) / ((size_t)q.stage_floats * sizeof(float)));
                if (ns >= 3 || q.FB == 1 || (ns >= 2 && q.FB <= 4)) break;
            }
            if (ns < 2) continue;
            q.nstage = std::min(ns, q.FB >= 4 ? 4 : MAX_STAGES);
            // shift rows the passes cover per shift row of the table (a pass takes the time of G full warp groups)
            const double cover = (double)q.npass * q.G * SH / S;
            const double cost = (stream ? 1. : (double)eh / (eh - H2)) * cover * (1. + .05 * (q.npass - 1)) * (1. + .5 / q.FB)
                              * (stream == 2 ? 1.05 : 1.);
            if (cost < best - 1e-9) {
                best = cost; bp = q;
                bp.seg_rows = stream ? 0 : eh - H2;              // streaming: chosen below
                bp.pass_major = stream == 2;
                bp.stream = stream;
                best_smem = (size_t)q.nstage * q.stage_floats * sizeof(float) + cbuf + carry;
            }
        }
    if (!best_smem) return 0;
    p = bp;
    if (const char *e = getenv("UMPA_TAB_DBG")) p.dbg = atoi(e);
    if (const char *e = getenv("UMPA_TAB_NST")) p.nstage = std::max(2, std::min(p.nstage, atoi(e)));
    if (p.seg_rows == 0) {
        // streaming: segments per strip such that the slowest CTA has the fewest chunks (every segment pays the
        // window halo once; every CTA works through ceil(items / ctas) items)
        long best_span = -1;
        int best_n = 1;
        for (int n = 1; n <= std::max(1, rows / p.EH); n++) {
            const int sr = (rows + n - 1) / n, nseg = (rows + sr - 1) / sr;
            const long waves = ((long)p.nstrips * nseg + ctas - 1) / ctas, chunks = (sr + H2 + p.EH - 1) / p.EH;
            if (best_span < 0 || waves * chunks < best_span) { best_span = waves * chunks; best_n = n; }
        }
        if (const char *e = getenv("UMPA_TAB_NSEG")) best_n = std::max(1, atoi(e));
        p.seg_rows = (rows + best_n - 1) / best_n;
    }
    p.nseg = (rows + p.seg_rows - 1) / p.seg_rows;
    p.nchunk_full = (p.seg_rows + H2 + p.EH - 1) / p.EH;
    p.nchunk_last = (rows - (p.nseg - 1) * p.seg_rows + H2 + p.EH - 1) / p.EH;
    *nt = p.G * p.EH * 8;
    return best_smem;
}

}  // namespace

// The geometry plan_tiles chooses for the cross table of a match (host arithmetic only; bench.py and the tests
// read the plan from here instead of restating it).  out: EH, streaming order (0 halo tiles, 1 chunk-major,
// 2 pass-major), G, npass, FB, nstage, TW, nseg, nstrips, block size.
extern "C" UMPA_API int umpa_table_plan(int Na, int Nw, int max_shift, int rows, int cols, int sm_count, int out[10])
{
    if (Na < 1 || Nw < 0 || Nw > 6 || max_shift < 1 || rows < 1 || cols < 1 || sm_count < 1 || !out) {
        umpa_set_error("umpa_table_plan: bad arguments");
        return UMPA_ERR_ARG;
    }
    TableParams p{};
    p.Na = Na; p.Nw = Nw;
    int nt = 0;
    const size_t smem = plan_tiles(p, 2 * max_shift - 1, true, &nt, rows, cols, sm_count * ctas_per_sm(), ctas_per_sm());
    if (!smem) { umpa_set_error("table path: no tile plan (shared memory, or chunks forced by UMPA_TAB_EH / UMPA_TAB_CTAS too short for the window)"); return UMPA_ERR_UNSUPPORTED; }
    const int v[10] = {p.EH, p.stream, p.G, p.npass, p.FB, p.nstage, p.TW, p.nseg, p.nstrips, nt};
    for (int i = 0; i < 10; i++) out[i] = v[i];
    return UMPA_OK;
}

// FP64 device stacks -> centring constants + centred FP32 stacks (pitch multiple of 4 floats)
int table_row_step(int H) { return std::max(1, H / 32); }

// equal frames, or (unmasked) ragged frames / positions on the common canvas
static bool table_applicable(const umpa_model *m) { return m->uniform || !m->masked; }

int table_alloc32(umpa_model *m)
{
    if (!table_applicable(m) || m->d_sam32) return UMPA_OK;
    const int Na = m->Na;
    m->pitch = 4 * ((m->W + 3) / 4);
    const size_t n32 = (size_t)Na * m->H * m->pitch;
    UMPA_CUDA(pool_malloc((void **)&m->d_sam32, n32 * sizeof(float)));
    UMPA_CUDA(pool_malloc((void **)&m->d_ref32, n32 * sizeof(float)));
    // (the constants and the partial sums live in the model's arena, capi.cu: arena_carve)
    m->dev_bytes += 2 * n32 * sizeof(float);
    return UMPA_OK;
}

int table_means(umpa_model *m, cudaStream_t st)
{
    if (!table_applicable(m)) return UMPA_OK;
    const int Na = m->Na;
    frame_partial_sums<<<dim3(SUM_BLOCKS, 2 * Na), 256, 0, st>>>(m->d_sam_ptrs, m->d_ref_ptrs, m->d_dim, Na, m->d_partials);
    finish_means<<<1, 256, 0, st>>>(m->d_partials, m->d_dim, Na, m->d_means64, m->d_mean_s, m->d_mean_r, m->d_consts);
    UMPA_CUDA(cudaGetLastError());
    return UMPA_OK;
}

int table_set_means(umpa_model *m, const double *mu, cudaStream_t st)
{
    if (!table_applicable(m)) return UMPA_OK;
    const int Na = m->Na;
    const size_t nd = 2 * (size_t)Na + 3;
    if (!m->h_small) {
        m->h_small = pinned_small_take(nd * sizeof(double) + 2 * Na * sizeof(float), &m->h_small_own);
        if (!m->h_small) { umpa_set_error("cudaHostAlloc failed for the model constants"); return UMPA_ERR_CUDA; }
    }
    double *hd = (double *)m->h_small;
    float *hf = (float *)(hd + nd);
    double cd = 0., cc = 0., dd = 0.;
    for (int k = 0; k < Na; k++) {
        const double d = mu[k], c = mu[Na + k];
        hd[k] = d; hd[Na + k] = c;
        hf[k] = (float)d; hf[Na + k] = (float)c;
        cd += c * d; cc += c * c; dd += d * d;
    }
    hd[2 * Na] = cd; hd[2 * Na + 1] = cc; hd[2 * Na + 2] = dd;
    UMPA_CUDA(cudaMemcpyAsync(m->d_means64, hd, 2 * Na * sizeof(double), cudaMemcpyHostToDevice, st));
    UMPA_CUDA(cudaMemcpyAsync(m->d_consts, hd + 2 * Na, 3 * sizeof(double), cudaMemcpyHostToDevice, st));
    UMPA_CUDA(cudaMemcpyAsync(m->d_mean_s, hf, Na * sizeof(float), cudaMemcpyHostToDevice, st));
    UMPA_CUDA(cudaMemcpyAsync(m->d_mean_r, hf + Na, Na * sizeof(float), cudaMemcpyHostToDevice, st));
    return UMPA_OK;
}

int table_center_rows(umpa_model *m, int y0, int y1, cudaStream_t st)
{
    if (!table_applicable(m) || y1 <= y0) return UMPA_OK;
    center_frames<<<dim3((m->pitch + 255) / 256, y1 - y0, 2 * m->Na), 256, 0, st>>>(
        m->d_sam_ptrs, m->d_ref_ptrs, m->d_dim, m->d_pos, m->d_means64, m->Na, m->H, m->pitch, y0, m->d_sam32, m->d_ref32);
    UMPA_CUDA(cudaGetLastError());
    return UMPA_OK;
}

int table_center_rows_inplace(umpa_model *m, int y0, int y1, cudaStream_t st)
{
    if (!m->uniform || y1 <= y0) return UMPA_OK;
    center_inplace<<<dim3((m->pitch + 255) / 256, y1 - y0, 2 * m->Na), 256, 0, st>>>(
        m->d_means64, m->Na, m->H, m->W, m->pitch, y0, m->d_sam32, m->d_ref32);
    UMPA_CUDA(cudaGetLastError());
    return UMPA_OK;
}

int table_prepare_frames(umpa_model *m, cudaStream_t st)
{
    int rc;
    if ((rc = table_alloc32(m))) return rc;
    if ((rc = table_means(m, st))) return rc;
    return table_center_rows(m, 0, m->H, st);
}

bool table_eligible(const umpa_model *m, const RoiView &roi, std::string *why, bool mixed)
{
    auto no = [&](const char *s) { if (why) *why = s; return false; };
    if (!m->uniform && !mixed) return no("ragged frames or non-zero positions");
    if (!m->uniform && m->masked) return no("masks together with ragged frames / positions");
    if (m->masked && !mixed) return no("masks");
    if (!m->separable) return no("window is not separable");
    // a handful of samples per cost (e.g. a 1x1 window on 3 frames): the fit is nearly exact, cost << signal
    // energy, and FP32 sums lose it to cancellation (367 of 2509 pixels off by > 1e-4 in that example)
    if (m->K * m->K * m->Na < 25) return no("fewer than 25 samples per cost: FP32 sums too coarse");
    if (m->kind == UMPA_DFKERNEL) {
        if (!ktable_supported(m->Nw, m->max_shift, roi.step0, m->refshift != 0)) return no("DFKernel: (Nw, max_shift, step) outside the instantiated blur-table kernels");
        if (!m->d_sam32) return no("FP32 stacks not prepared");
        return true;
    }
    if (m->max_shift < 2 || m->max_shift > 10) return no("max_shift outside 2..10");
    if (m->Nw > 6) return no("window too large for the tiled kernel (Nw > 6)");
    if (roi.step0 * roi.step1 > 16) return no("sparse ROI (step product > 16)");
    if (!m->d_sam32) return no("FP32 stacks not prepared");
    if (!encode_tiled_fn()) return no("driver has no cuTensorMapEncodeTiled");
    return true;
}

// UMPA_DEBUG_SYNC=1: synchronise after every stage and name the one that faulted
static int stage_check(const char *name, cudaStream_t st)
{
    static const bool on = getenv("UMPA_DEBUG_SYNC") != nullptr;
    if (!on) return UMPA_OK;
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { umpa_set_error("stage '%s' failed: %s", name, cudaGetErrorString(e)); return UMPA_ERR_CUDA; }
    return UMPA_OK;
}

static int table_match_impl(umpa_model *m, const RoiView &roi, const umpa_outputs &out, cudaStream_t st, WalkParams *keep);

int table_match(umpa_model *m, const RoiView &roi, const umpa_outputs &out, cudaStream_t st)
{
    return table_match_impl(m, roi, out, st, nullptr);
}

// keep: where to leave the walk's view of the tables (mixed_match: the corrected walk of binary masks reads them too)
static int table_match_impl(umpa_model *m, const RoiView &roi, const umpa_outputs &out, cudaStream_t st, WalkParams *keep)
{
    const int S = 2 * m->max_shift - 1, HS = m->max_shift - 1;
    const bool df = m->kind == UMPA_DF;
    const int Na = m->Na, H = m->H, pitch = m->pitch;
    // dense table region in raw coordinates
    const int oy = roi.off0, ox = roi.off1;
    const int rows = (roi.N0 - 1) * roi.step0 + 1, cols = (roi.N1 - 1) * roi.step1 + 1;

    const bool dfk = m->kind == UMPA_DFKERNEL;
    TableParams px{};
    px.Na = Na; px.Nw = m->Nw; px.oy = oy; px.g = m->d_g;
    TableParams pm = px;
    // shift each table's origin left so that its B-tile columns (origin - halo) are 16 B aligned
    const int dxX = (ox - m->Nw) & 3, dxM = ox & 3;
    px.ox = ox - dxX; pm.ox = ox - dxM;
    int ntx = 0, ntm = 0;
    size_t smx = 0, smm = 0;
    int rc;
    if (dfk) {
        if (!roi.abc) { umpa_set_error("abc array has to be provided"); return UMPA_ERR_ARG; }
        if ((rc = scratch_reserve(m, m->tabX, (size_t)roi.N0 * roi.N1 * ktable_row_floats(m->max_shift) * sizeof(float)))) return rc;
    } else {
        const int ctas = m->sm_count * ctas_per_sm();
        smx = plan_tiles(px, S, true, &ntx, rows, cols + dxX, ctas, ctas_per_sm());
        smm = df ? plan_tiles(pm, S, false, &ntm, rows, cols + dxM, ctas, ctas_per_sm()) : 1;
        if (!smx || !smm) { umpa_set_error("table path: no tile plan (shared memory, or chunks forced by UMPA_TAB_EH / UMPA_TAB_CTAS too short for the window)"); return UMPA_ERR_UNSUPPORTED; }
        const int rows_alloc = rows;
        int tpitch = px.cols_p;
        if (df) tpitch = std::max(tpitch, pm.cols_p);
        // one buffer, [row][table][shift][col]: everything a pixel's walk reads lies within one row's S*S
        // (2 S*S for DF) segments -- a few hundred KB -- instead of S*S planes of the image size
        px.plane_stride = pm.plane_stride = tpitch;
        px.row_stride = pm.row_stride = (size_t)(df ? 2 : 1) * S * S * tpitch;
        if ((rc = scratch_reserve(m, m->tabX, (size_t)(df ? 2 : 1) * S * S * rows_alloc * tpitch * sizeof(float)))) return rc;

    }
    const size_t img = (size_t)H * pitch;
    if ((rc = scratch_reserve(m, m->auxS, img * sizeof(AuxS)))) return rc;
    if ((rc = scratch_reserve(m, m->auxR, img * sizeof(AuxR)))) return rc;
    if (df) {
        if ((rc = scratch_reserve(m, m->filtA, (size_t)Na * img * sizeof(float)))) return rc;
        if ((rc = scratch_reserve(m, m->filtB, (size_t)Na * img * sizeof(float)))) return rc;
    }
    if (m->profiling) {
        if (!m->ev[0]) for (int i = 0; i < 5; i++) UMPA_CUDA(cudaEventCreate(&m->ev[i]));
        UMPA_CUDA(cudaEventRecord(m->ev[0], st));
    }

    // 1. moments over the bounding box of everything the walk can touch
    {
        MomentsParams mp{};
        mp.sam = m->d_sam32; mp.ref = m->d_ref32;
        mp.fa = df ? (float *)m->filtA.p : nullptr; mp.fb = df ? (float *)m->filtB.p : nullptr;
        mp.auxS = (AuxS *)m->auxS.p; mp.auxR = (AuxR *)m->auxR.p;
        mp.g = m->d_g; mp.mean_s = m->d_mean_s; mp.mean_r = m->d_mean_r;
        mp.consts = m->d_consts; mp.kind = m->kind;
        mp.sw = m->win_sum; mp.inv_sw = 1. / mp.sw; mp.inv_sw2 = 1. / (mp.sw * mp.sw);
        mp.Na = Na; mp.Nw = m->Nw; mp.H = H; mp.W = m->W; mp.pitch = pitch;
        const int ylo = std::max(0, oy - HS), yhi = std::min(H, oy + rows + HS);
        const int xlo = std::max(0, ox - HS), xhi = std::min(m->W, ox + cols + HS);
        mp.ty0 = ylo / MO_TH; mp.tx0 = xlo / MO_TW;
        dim3 grid((xhi + MO_TW - 1) / MO_TW - mp.tx0, (yhi + MO_TH - 1) / MO_TH - mp.ty0);
        if ((rc = launch_moments(m->Nw, mp, m->d_ref32, m->d_sam32, grid, st))) return rc;
        m->last_launches++;
        if ((rc = stage_check("moments", st))) return rc;
    }
    if (m->profiling) UMPA_CUDA(cudaEventRecord(m->ev[1], st));

    // 2. DFKernel: per-pixel blur tables (kernel_path.cu)
    if (dfk) {
        if ((rc = ktable_build(m, roi, (float *)m->tabX.p, st))) return rc;
        if ((rc = stage_check("blur table", st))) return rc;
    }
    // 2. cross table: A = centred reference (read at p+s), B = centred sample, window-filtered
    else {
        CUtensorMap ma, mb;
        // the moving operand (read at p + s): the reference, or (reference_shift) the sample
        const float *mov = m->refshift ? m->d_sam32 : m->d_ref32, *fix = m->refshift ? m->d_ref32 : m->d_sam32;
        if ((rc = make_stack_map(&ma, mov, Na, H, m->W, pitch, px.AP, px.AH, px.FB))) return rc;
        if ((rc = make_stack_map(&mb, fix, Na, H, m->W, pitch, EXT_W, px.EH, px.FB))) return rc;
        px.table = (float *)m->tabX.p;
        dim3 grid(std::min(px.nstrips * px.nseg, m->sm_count * ctas_per_sm()));
        if ((rc = dispatch_shift_table(true, S, ma, mb, px, grid, ntx, smx, st))) return rc;
        m->last_launches++;
        if ((rc = stage_check("cross table", st))) return rc;
    }
    if (m->profiling) UMPA_CUDA(cudaEventRecord(m->ev[2], st));

    // 3. mean table (DF): A = a_k, B = b_k, no filter
    if (df) {
        CUtensorMap ma, mb;
        const float *mov = (const float *)(m->refshift ? m->filtB.p : m->filtA.p);
        const float *fix = (const float *)(m->refshift ? m->filtA.p : m->filtB.p);
        if ((rc = make_stack_map(&ma, mov, Na, H, m->W, pitch, pm.AP, pm.AH, pm.FB))) return rc;
        if ((rc = make_stack_map(&mb, fix, Na, H, m->W, pitch, EXT_W, pm.EH, pm.FB))) return rc;
        pm.table = (float *)m->tabX.p + (size_t)S * S * pm.plane_stride;     // (either layout: the mean table follows the S*S cross shifts)
        dim3 grid(std::min(pm.nstrips * pm.nseg, m->sm_count * ctas_per_sm()));
        if ((rc = dispatch_shift_table(false, S, ma, mb, pm, grid, ntm, smm, st))) return rc;
        m->last_launches++;
        if ((rc = stage_check("mean table", st))) return rc;
    }
    if (m->profiling) UMPA_CUDA(cudaEventRecord(m->ev[3], st));

    // 4. walk
    {
        WalkParams w{};
        w.tabX = (const float *)m->tabX.p;
        w.row_stride = px.row_stride; w.tpitch = (unsigned)px.plane_stride;
        w.m_off = (size_t)S * S * px.plane_stride + dxM - dxX;
        if (dfk) {
            w.ktab = w.tabX; w.kstride = ktable_row_floats(m->max_shift);
            double swk = 0.;                           // exact sum of float(g_a) * float(g_b) as FP32 products
            for (int a = 0; a < m->K; a++)
                for (int b = 0; b < m->K; b++) swk += (double)((float)m->g[a] * (float)m->g[b]);
            w.swk = swk;
        }
        w.auxS = (const AuxS *)m->auxS.p; w.auxR = (const AuxR *)m->auxR.p;
        w.pitch = pitch;
        w.oy = oy; w.ox = ox; w.dxX = dxX;
        w.Na = Na; w.max_shift = m->max_shift; w.subpx = m->subpx;
        w.sw = m->win_sum; w.quad = m->d_quad;
        w.inv_sw = 1. / w.sw; w.inv_Na = 1. / (double)Na;
        w.consts = m->d_consts;
        if (keep) *keep = w;
        dim3 grid((roi.N1 + WALK_NT - 1) / WALK_NT, roi.N0);
        if (m->refshift) launch_walk<true>(m->kind, grid, w, roi, out, st);
        else launch_walk<false>(m->kind, grid, w, roi, out, st);
        UMPA_CUDA(cudaGetLastError());
        m->last_launches++;
        if ((rc = stage_check("walk", st))) return rc;
    }
    if (m->profiling) { UMPA_CUDA(cudaEventRecord(m->ev[4], st)); m->ev_valid = true; }
    return UMPA_OK;
}

// ------------------------------------------------------------------ masked models: the mixed path
//
// With masks the weights g = m_r m_s / (m_r + m_s + 1e-8) (Utils.cpp:125-130) couple the two window
// positions and do not factor, so the masked cost (Model.cpp:461-499, 775-847) is not a sum of
// tables.  But where every mask value within reach of a pixel is exactly 1, g is the constant
// 1/(2+1e-8) and every sum of the masked branch is that constant times the unmasked one: cost, T
// and df are the unmasked ones (to 1e-16: sum w = 1 - 1e-16), and the coverage gate passes.  Real
// masks are mostly ones (dead pixels, a beam stop), so: table kernels on the clean pixels, the FP64
// lazy evaluation on the pixels with a mask value != 1 within +-padding.
namespace {

// any_k mask_k(y, x') != 1 for x' within +-pad of x  ->  bad[y][x]  (row-dilated; one pass over the mask stack)
__global__ void mask_rows_kernel(const double *mask, int Na, int H, int W, int pad, unsigned char *bad)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= W) return;
    const int x0 = max(0, x - pad), x1 = min(W - 1, x + pad);
    unsigned char b = 0;
    for (int k = 0; k < Na && !b; k++) {
        const double *row = mask + ((size_t)k * H + y) * W;
        for (int xx = x0; xx <= x1; xx++) b |= row[xx] != 1.;
    }
    bad[(size_t)y * W + x] = b;
}

// dirty[n] = any bad[y'][j] for y' within +-pad of the pixel's raw row
__global__ void dirty_kernel(const unsigned char *bad, int H, int W, int pad, RoiView roi, unsigned char *dirty)
{
    const int xj = blockIdx.x * blockDim.x + threadIdx.x, xi = blockIdx.y;
    if (xj >= roi.N1) return;
    const int i = roi.off0 + roi.step0 * xi, j = roi.off1 + roi.step1 * xj;
    unsigned char b = 0;
    for (int y = max(0, i - pad); y <= min(H - 1, i + pad); y++) b |= bad[(size_t)y * W + j];
    dirty[(size_t)xi * roi.N1 + xj] = b;
}

// Ragged frames / per-frame positions (sample stepping, model.pyx:265-283): frame k takes part in a pixel's
// cost only if the pixel +-padding lies inside it (Model.cpp:428-433, 716-719; wt stays Na).  On the canvas a
// frame that does not overlap the pixel's reach contributes nothing, a frame that contains it contributes what
// the reference reads: the table kernels are exact there.  A frame that overlaps the reach only PARTLY is
// skipped by the reference but would leak into the tables: those pixels are dirty.
__global__ void dirty_rect_kernel(const int *dim, const int *pos, int Na, int pad, RoiView roi, unsigned char *dirty)
{
    const int xj = blockIdx.x * blockDim.x + threadIdx.x, xi = blockIdx.y;
    if (xj >= roi.N1) return;
    const int i = roi.off0 + roi.step0 * xi, j = roi.off1 + roi.step1 * xj;
    unsigned char b = 0;
    for (int k = 0; k < Na; k++) {
        const int py = pos[2 * k], px = pos[2 * k + 1], fh = dim[2 * k], fw = dim[2 * k + 1];
        const int ri = i - py, rj = j - px;
        const bool reach = !(ri - pad < 0 || ri + pad > fh || rj - pad < 0 || rj + pad > fw);
        const bool overlap = i + pad >= py && i - pad < py + fh && j + pad >= px && j - pad < px + fw;
        b |= !reach && overlap;
    }
    dirty[(size_t)xi * roi.N1 + xj] = b;
}

// ---- binary masks shared by all frames: the table walk with corrected sums
//
// For mask values in {0, 1} the weight m_r m_s / (m_r + m_s + 1e-8) is gamma = 1/(2+1e-8) where both are 1, else 0;
// gamma cancels in T, df and the cost (every sum of Model.cpp:461-499 / 775-847 carries it, wt too).  With ONE mask
// M = 1 - D for all frames a masked sum is the unmasked one minus the window positions u where D(p+s+u) or D(p+u):
//     t1 = t1u - sum_E w(u) sum_k S_k(p+u)^2          t3 = t3u - sum_E w(u) sum_k R_k(p+s+u)^2
//     t5 = t5u - sum_E w(u) sum_k R_k(p+s+u) S_k(p+u)
//     t4 = t4u - sum_E w(u) sum_k m_k S_k(p+u)        t6 = t6u - sum_E w(u) sum_k m_k R_k(p+s+u)
//     t2 = (sum_k m_k^2) (sw - sum_E w(u))            wt = Na (sw - sum_E w(u))
// (m_k, the frame's window mean of the reference, is NOT masked in the reference: Model.cpp:789-806).  The unmasked
// sums are what the tables and aux images hold; E is read off the window's dead-pixel bits (one 64-bit word per
// pixel for Nw <= 3, else K row words of the bit image of D); a dead
// position costs the Na frame values of either stack at that position (+ m_k from the filtered reference stack, DF),
// read from frame-minor copies of the stacks and summed in FP32 like the tables.  Exact algebra
// (tests/test_table_algebra.py); the FP32 rounding is that of the unmasked path.

struct MaskedParams {
    const unsigned *bits;           // D: bit (x & 31) of bits[y * wb + (x >> 5)]
    int wb;
    const unsigned long long *dwin; // Nw <= 3: per raw pixel [H][W], bit (a K + b) = D(y - Nw + a, x - Nw + b); else nullptr
    int W;
    // frame-minor copies [H][pitch][Nap] of the centred stacks and (DF) of the filtered reference stack w (*) R'_k:
    // the Na values of one pixel are Nap = 8 ceil(Na / 8) consecutive floats (zero padded; 25 frames: exactly one
    // 128 B line) -- a dead window position costs four 256-bit loads per stack instead of 25 sectors in 25 frames
    const float *tS, *tR, *tA;
    int Nap;
    // what a dead position needs of ONE pixel, [H][pitch]: imgS = (sum S'^2, sum d_k S', sum c_k S', -),
    // imgR = (sum R'^2, sum c_k R', sum d_k R', sum c_k a'_k) with the FP32 centring constants d_k (sample), c_k (reference)
    const float4 *imgS, *imgR;
    const double *win;              // K x K window (FP64, the reference's)
    int Nw;
};

// [Na][H][pitch] -> [H][pitch][Nap], rows [y0, y1), and the frame sums that need ONE pixel only, as an image of
// float4 [H][pitch]: mode 0 -> (sum v^2, sum k1 v, sum k2 v) into x, y, z; mode 1 -> sum k1 v into w.
// grid (ceil(pitch / 32), y1 - y0), 256 threads
__global__ void frame_minor_kernel(const float *src, int Na, int Nap, int H, int pitch, int y0, float *dst,
                                   const float *k1, const float *k2, float *img, int mode)
{
    extern __shared__ float tile[];             // [Nap][33]
    const int y = y0 + blockIdx.y, x0 = blockIdx.x * 32, lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    for (int k = wrp; k < Nap; k += 8)
        tile[k * 33 + lane] = (k < Na && x0 + lane < pitch) ? src[((size_t)k * H + y) * pitch + x0 + lane] : 0.f;
    __syncthreads();
    const int n = min(32, pitch - x0) * Nap;
    float *out = dst + ((size_t)y * pitch + x0) * Nap;
    for (int i = threadIdx.x; i < n; i += 256) out[i] = tile[(i % Nap) * 33 + i / Nap];
    if (wrp == 0 && x0 + lane < pitch) {
        float a0 = 0.f, a1 = 0.f, a2 = 0.f;
        for (int k = 0; k < Na; k++) {
            const float v = tile[k * 33 + lane];
            a0 = fmaf(v, v, a0); a1 = fmaf(__ldg(k1 + k), v, a1);
            if (mode == 0) a2 = fmaf(__ldg(k2 + k), v, a2);
        }
        float *o = img + 4 * ((size_t)y * pitch + x0 + lane);
        if (mode == 0) { o[0] = a0; o[1] = a1; o[2] = a2; }
        else o[3] = a1;
    }
}

// flags[0] |= 1 where a mask value is neither 0 nor 1 or differs from frame 0; flags[1] / flags[2]: largest |centred
// value| of either stack over the dead / the live pixels (bits of a non-negative float: they order like the values;
// a NaN counts as larger than everything).  One warp per 32 columns: its ballot is the row's bit word.
__global__ void mask_classify_kernel(const double *mask, const float *sam32, const float *ref32, int Na, int H, int W,
                                     int pitch, unsigned *bits, int wb, unsigned *flags)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    const bool in = x < W;
    bool dead = false, odd = false;
    unsigned mx = 0;
    if (in) {
        const size_t px = (size_t)y * W + x, img64 = (size_t)H * W, img32 = (size_t)H * pitch, p32 = (size_t)y * pitch + x;
        const double v0 = mask[px];
        dead = v0 == 0.;
        odd = !(v0 == 0. || v0 == 1.);
        for (int k = 0; k < Na; k++) {
            if (k) odd |= mask[k * img64 + px] != v0;
            mx = max(mx, __float_as_uint(fabsf(sam32[k * img32 + p32])));
            mx = max(mx, __float_as_uint(fabsf(ref32[k * img32 + p32])));
        }
    }
    const unsigned word = __ballot_sync(0xffffffffu, dead);
    if ((threadIdx.x & 31) == 0 && (x >> 5) < wb) bits[(size_t)y * wb + (x >> 5)] = word;
    if (__any_sync(0xffffffffu, odd) && (threadIdx.x & 31) == 0) atomicOr(flags, 1u);
    unsigned md = dead ? mx : 0u, ml = (in && !dead) ? mx : 0u;
    for (int o = 16; o > 0; o >>= 1) {
        md = max(md, __shfl_xor_sync(0xffffffffu, md, o));
        ml = max(ml, __shfl_xor_sync(0xffffffffu, ml, o));
    }
    if ((threadIdx.x & 31) == 0) {
        if (md) atomicMax(flags + 1, md);
        if (ml) atomicMax(flags + 2, ml);
    }
}

// the dead pixels of every pixel's window as one word (K*K <= 49 bits): one gather per cost evaluation
__global__ void window_bits_kernel(const unsigned *bits, int wb, int H, int W, int Nw, unsigned long long *dwin)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= W) return;
    const int K = 2 * Nw + 1;
    unsigned long long e = 0;
    for (int a = 0; a < K; a++) {
        const int yy = y - Nw + a;
        if (yy < 0 || yy >= H) continue;
        // columns x - Nw ... x + Nw of row yy (bits beyond the row are 0; left of column 0: shift in zeros)
        const int x0 = x - Nw;
        unsigned r;
        if (x0 >= 0) {
            const unsigned *p = bits + (size_t)yy * wb + (x0 >> 5);
            r = __funnelshift_r(p[0], p[1], x0 & 31);
        } else {
            r = bits[(size_t)yy * wb] << (-x0);
        }
        e |= (unsigned long long)(r & ((1u << K) - 1u)) << (a * K);
    }
    dwin[(size_t)y * W + x] = e;
}

// eight consecutive floats, 32 B aligned, as ONE 256-bit load (sm_100: LDG.E.256): the walk below is bound by the
// number of load wavefronts its scattered lanes generate, not by bytes
struct Float8 { float v[8]; };
__device__ __forceinline__ Float8 ldg256(const float *p)
{
    Float8 r;
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]), "=f"(r.v[4]), "=f"(r.v[5]), "=f"(r.v[6]), "=f"(r.v[7])
                 : "l"(p));
    return r;
}

// RS = reference_shift (assign_coordinates = 'ref', Model.cpp:686-692): the reference window stays at the pixel and
// the SAMPLE window moves by -s; the tables hold the same sums with the roles of the stacks swapped (TableEval<RS>).
template <bool RS, int KIND>
struct MaskedEval {
    const WalkParams &w;
    const MaskedParams &mp;
    double cd, cc, dd;              // sum c_k d_k, sum c_k^2, sum d_k^2
    AuxS ps;                        // the sample's record at the pixel (!RS)
    AuxR pr;                        // the reference's record at the pixel (RS)
    const AuxS *pS;
    const AuxR *pR;
    const float *pX;
    int y0, x0;                     // raw coordinates of the pixel
    unsigned long long epw;         // the dead pixels of the pixel's own window (dwin)

    __device__ __forceinline__ unsigned row_bits(int y, int x, int K) const
    {
        const unsigned *r = mp.bits + (size_t)y * mp.wb + (x >> 5);
        return __funnelshift_r(__ldg(r), __ldg(r + 1), x & 31) & ((1u << K) - 1u);
    }

    __device__ __forceinline__ int operator()(int si, int sj, double &cst, FitArgs &args)
    {
        const int ms = w.max_shift, S = 2 * ms - 1;
        const int ti = RS ? -si : si, tj = RS ? -sj : sj;
        const unsigned a = (unsigned)(ti + ms - 1), b = (unsigned)(tj + ms - 1);
        if (a >= (unsigned)S || b >= (unsigned)S) return TableEval<RS, KIND>::out_of_bounds(si, sj, ms);
        const unsigned sidx = a * (unsigned)S + b;
        const int q = ti * w.pitch + tj;           // the moving window's pixel relative to this one
        const float *px = pX + (size_t)sidx * w.tpitch;
        const float x = __ldg(px);
        const float m = KIND == UMPA_DF ? __ldg(px + w.m_off) : 0.f;
        double2 v0, v1;                            // the reference's record {t3, t2}, {rden, linq}
        double st1, sV;                            // the sample's record
        if (RS) {
            const double2 v = __ldg(reinterpret_cast<const double2 *>(pS + q));
            st1 = v.x; sV = v.y;
            v0 = make_double2(pr.t3, pr.t2); v1 = make_double2(pr.rden, pr.linq);
        } else {
            v0 = __ldg(reinterpret_cast<const double2 *>(pR + q));
            v1 = __ldg(reinterpret_cast<const double2 *>(pR + q) + 1);
            st1 = ps.t1; sV = ps.V;
        }
        const double lin = v1.y + sV;
        double t1 = st1, t3 = v0.x, t5 = (double)x + lin;
        double t4 = (double)m * w.inv_sw + lin, t6 = w.sw * v0.y;
        // the window positions with a dead pixel in either window: the reference window at (qy, qx), the sample
        // window at (py, px_); (my, mx) is the one that moves
        const int Nw = mp.Nw, K = 2 * Nw + 1, n8 = mp.Nap >> 3;
        const int qy = RS ? y0 : y0 + si, qx = RS ? x0 : x0 + sj;
        const int py = RS ? y0 - si : y0, px_ = RS ? x0 - sj : x0;
        const int my = RS ? py : qy, mx = RS ? px_ : qx;
        const double U = v1.y - w.sw * cd;           // sum_k d_k a'_k(q)  (AuxR::linq = U + sw sum c_k d_k)
        double cw = 0.;
        const int rows = mp.dwin ? 1 : K;            // one word for the whole window, or a word per window row (Nw > 3)
        const unsigned rk = 65536u / (unsigned)K + 1u;      // (bit * rk) >> 16 == bit / K for bit < K*K <= 49
        // 32-bit pixel / element indices (classify_mask keeps models whose frame-minor copies exceed 2^32 floats off
        // this path): the address arithmetic is a third of the kernel's instructions
        const unsigned upitch = (unsigned)w.pitch, unap = (unsigned)mp.Nap;
        const unsigned qpix = (unsigned)qy * upitch + (unsigned)qx;
        const unsigned sbase = (unsigned)(py - Nw) * upitch + (unsigned)(px_ - Nw);
        const unsigned rbase = (unsigned)(qy - Nw) * upitch + (unsigned)(qx - Nw);
        const float *A8 = mp.tA + (size_t)(qpix * unap);
        for (int row = 0; row < rows; row++) {
            unsigned long long e = mp.dwin ? (epw | __ldg(mp.dwin + (size_t)my * mp.W + mx))
                                           : (unsigned long long)(row_bits(y0 - Nw + row, x0 - Nw, K) | row_bits(my - Nw + row, mx - Nw, K));
            while (e) {
                const int bit = __ffsll((long long)e) - 1;
                e &= e - 1;
                const int wa = mp.dwin ? (int)(((unsigned)bit * rk) >> 16) : row;
                const int wb = mp.dwin ? bit - wa * K : bit;
                const double wgt = __ldg(mp.win + wa * K + wb);
                const unsigned off = (unsigned)wa * upitch + (unsigned)wb, spix = sbase + off, rpix = rbase + off;
                const float4 iS = __ldg(mp.imgS + spix), iR = __ldg(mp.imgR + rpix);
                const float *S8 = mp.tS + (size_t)(spix * unap), *R8 = mp.tR + (size_t)(rpix * unap);
                // the sums over the frames that need both pixels, in FP32 on the centred values (the precision class
                // of the tables themselves).  (Two positions per trip, sharing the m_k loads, measured slower: 12.5 vs
                // 11.9 ms -- the second set of operands spills.)
                float rs = 0.f, as = 0.f, ar = 0.f;
#pragma unroll 2
                for (int k = 0; k < n8; k++) {
                    const Float8 s = ldg256(S8 + 8 * k), r = ldg256(R8 + 8 * k);
#pragma unroll
                    for (int u = 0; u < 8; u++) rs = fmaf(r.v[u], s.v[u], rs);
                    if (KIND == UMPA_DF) {
                        const Float8 av = ldg256(A8 + 8 * k);
#pragma unroll
                        for (int u = 0; u < 8; u++) { as = fmaf(av.v[u], s.v[u], as); ar = fmaf(av.v[u], r.v[u], ar); }
                    }
                }
                // uncentred: S = S' + d_k, R = R' + c_k, m_k = a'_k / sw + c_k
                cw += wgt;
                t1 -= wgt * ((double)iS.x + 2. * (double)iS.y + dd);
                t3 -= wgt * ((double)iR.x + 2. * (double)iR.y + cc);
                t5 -= wgt * ((double)rs + (double)iS.z + (double)iR.z + cd);
                if (KIND == UMPA_DF) {
                    const double ca = (double)__ldg(reinterpret_cast<const float *>(mp.imgR + qpix) + 3);
                    t4 -= wgt * (((double)as + U) * w.inv_sw + (double)iS.z + cd);
                    t6 -= wgt * (((double)ar + ca) * w.inv_sw + (double)iR.y + cc);
                }
            }
        }
        const double swm = w.sw - cw, wt = (double)w.Na * swm;
        if (KIND == UMPA_DF) {
            const double t2 = v0.y * swm;
            const double rden = 1. / (t2 * t3 - t6 * t6);
            const double Kc = (t2 * t5 - t4 * t6) * rden;
            const double beta = (t3 * t4 - t5 * t6) * rden;
            args.t = beta + Kc;
            args.v = Kc;
            cst = (t1 - beta * t4 - Kc * t5) / wt;
            return UMPA_ST_OK;
        }
        args.t = t5 / t3;
        cst = (t1 - t5 * args.t) / wt;
        return UMPA_ST_OK;
    }
};

#ifndef MASKED_MINB
#define MASKED_MINB 5
#endif

template <bool RS, int KIND>
__global__ void __launch_bounds__(WALK_NT, MASKED_MINB) masked_walk_kernel(WalkParams w, MaskedParams mp, RoiView roi, umpa_outputs out)
{
    __shared__ double d_sm[25][WALK_NT];
    const int xj = blockIdx.x * blockDim.x + threadIdx.x;
    const int xi = blockIdx.y;
    if (xj >= roi.N1 || xi >= roi.N0) return;
    const size_t n = (size_t)xi * roi.N1 + xj;
    if (roi.cover && roi.cover[n] < roi.cover_threshold) return;
    if (roi.dirty && (roi.dirty[n] != 0) != (roi.dirty_want != 0)) return;
    const int ty = roi.step0 * xi, tx = roi.step1 * xj;
    const size_t pix = (size_t)(w.oy + ty) * w.pitch + (w.ox + tx);
    MaskedEval<RS, KIND> eval{w, mp};
    eval.cd = __ldg(w.consts); eval.cc = __ldg(w.consts + 1); eval.dd = __ldg(w.consts + 2);
    eval.pS = w.auxS + pix; eval.pR = w.auxR + pix;
    if (RS) {
        const double2 v0 = __ldg(reinterpret_cast<const double2 *>(eval.pR));
        const double2 v1 = __ldg(reinterpret_cast<const double2 *>(eval.pR) + 1);
        eval.pr = AuxR{v0.x, v0.y, v1.x, v1.y};
        eval.ps = AuxS{0., 0.};
    } else {
        const double2 v = __ldg(reinterpret_cast<const double2 *>(eval.pS));
        eval.ps = AuxS{v.x, v.y};
        eval.pr = AuxR{0., 0., 0., 0.};
    }
    eval.pX = w.tabX + (size_t)ty * w.row_stride + tx + w.dxX;
    eval.y0 = w.oy + ty; eval.x0 = w.ox + tx;
    eval.epw = mp.dwin ? __ldg(mp.dwin + (size_t)eval.y0 * mp.W + eval.x0) : 0ull;
    FitArgs args{0., 0.};
    SharedGrid d{&d_sm[0][threadIdx.x]};
    double uv[2] = {roi.uv0[0], roi.uv0[1]}, f = 0.;
    int ncalls;
    WalkState ws;
    const int st = walk_search(eval, args, f, uv, d, ncalls, ws);
    store_debug(out, n, d, ws);
    if (ws.finished) walk_refine(w.subpx, w.quad, d, ws, f, uv);
    if (KIND == UMPA_DF && args.t != 0.) args.v = args.v / args.t;
    store_pixel(out, n, KIND, st, f, args, uv, ncalls);
}

}  // namespace

// Classifies the mask stack once per set of frames: 2 = values 0 / 1, the same in every frame, and no dead pixel
// holds a value far outside the live range (the corrections subtract what the unmasked tables summed: a hot pixel
// of 1e4 times the signal would cost the FP32 tables their precision) -> corrected table walk; else 1 (lazy).
static int classify_mask(umpa_model *m, cudaStream_t st)
{
    if (m->mask_mode) return UMPA_OK;
    m->mask_mode = 1;
    const char *e = getenv("UMPA_MASK_TABLES");
    if ((e && atoi(e) == 0) || !m->uniform || !m->d_sam32) return UMPA_OK;
    if (m->kind != UMPA_DF && m->kind != UMPA_NODF) return UMPA_OK;      // (DFKernel: the blur couples the windows once more)
    if ((size_t)m->H * m->pitch * ((m->Na + 7) & ~7) >= ((size_t)1 << 32)) return UMPA_OK;    // (32-bit element indices in the walk)
    const int H = m->H, W = m->W, wb = W / 32 + 2;
    int rc;
    if ((rc = scratch_reserve(m, m->maskbits, (size_t)H * wb * sizeof(unsigned)))) return rc;
    if ((rc = scratch_reserve(m, m->maskflags, 4 * sizeof(unsigned)))) return rc;
    UMPA_CUDA(cudaMemsetAsync(m->maskbits.p, 0, (size_t)H * wb * sizeof(unsigned), st));
    UMPA_CUDA(cudaMemsetAsync(m->maskflags.p, 0, 4 * sizeof(unsigned), st));
    mask_classify_kernel<<<dim3((W + 127) / 128, H), 128, 0, st>>>(m->d_mask64, m->d_sam32, m->d_ref32, m->Na, H, W, m->pitch,
                                                                  (unsigned *)m->maskbits.p, wb, (unsigned *)m->maskflags.p);
    UMPA_CUDA(cudaGetLastError());
    unsigned fl[4];
    UMPA_CUDA(cudaMemcpyAsync(fl, m->maskflags.p, sizeof(fl), cudaMemcpyDeviceToHost, st));
    UMPA_CUDA(cudaStreamSynchronize(st));
    float dead_max, live_max;
    memcpy(&dead_max, fl + 1, 4); memcpy(&live_max, fl + 2, 4);
    if (!(fl[0] & 1u) && dead_max <= 4.f * live_max) m->mask_mode = 2;      // (a NaN fails the comparison)
    m->maskwin_Nw = -1;
    return UMPA_OK;
}

// the per-pixel window words of the current window size (rebuilt when the window changes)
static int ensure_window_bits(umpa_model *m, cudaStream_t st)
{
    if (m->Nw > 3 || m->maskwin_Nw == m->Nw) return UMPA_OK;
    const int H = m->H, W = m->W, wb = W / 32 + 2;
    int rc;
    if ((rc = scratch_reserve(m, m->maskwin, (size_t)H * W * sizeof(unsigned long long)))) return rc;
    window_bits_kernel<<<dim3((W + 127) / 128, H), 128, 0, st>>>((const unsigned *)m->maskbits.p, wb, H, W, m->Nw,
                                                                 (unsigned long long *)m->maskwin.p);
    UMPA_CUDA(cudaGetLastError());
    m->maskwin_Nw = m->Nw;
    return UMPA_OK;
}

int mixed_match(umpa_model *m, const RoiView &roi, const umpa_outputs &out, cudaStream_t st)
{
    int rc;
    const int H = m->H, W = m->W, pad = m->padding;
    if (!m->masked) {
        if ((rc = scratch_reserve(m, m->dirty, (size_t)roi.N0 * roi.N1))) return rc;
        dirty_rect_kernel<<<dim3((roi.N1 + 127) / 128, roi.N0), 128, 0, st>>>(m->d_dim, m->d_pos, m->Na, pad, roi,
                                                                            (unsigned char *)m->dirty.p);
        UMPA_CUDA(cudaGetLastError());
        RoiView v = roi;
        v.dirty = (const unsigned char *)m->dirty.p;
        v.dirty_want = 0;
        if ((rc = table_match(m, v, out, st))) return rc;
        v.dirty_want = 1;
        if ((rc = lazy_match(m, v, out, st))) return rc;
        m->last_launches += 1;
        return UMPA_OK;
    }
    if (!m->maskbad_valid) {
        if ((rc = scratch_reserve(m, m->maskbad, (size_t)H * W))) return rc;
        mask_rows_kernel<<<dim3((W + 127) / 128, H), 128, 0, st>>>(m->d_mask64, m->Na, H, W, pad, (unsigned char *)m->maskbad.p);
        UMPA_CUDA(cudaGetLastError());
        m->maskbad_valid = true;
    }
    if ((rc = scratch_reserve(m, m->dirty, (size_t)roi.N0 * roi.N1))) return rc;
    dirty_kernel<<<dim3((roi.N1 + 127) / 128, roi.N0), 128, 0, st>>>((const unsigned char *)m->maskbad.p, H, W, pad, roi,
                                                                       (unsigned char *)m->dirty.p);
    UMPA_CUDA(cudaGetLastError());
    RoiView v = roi;
    v.dirty = (const unsigned char *)m->dirty.p;
    v.dirty_want = 0;
    if ((rc = classify_mask(m, st))) return rc;
    if (m->mask_mode == 2 && m->Nw <= 6) {      // (the window may change between matches)
        WalkParams w{};
        if ((rc = table_match_impl(m, v, out, st, &w))) return rc;
        v.dirty_want = 1;
        // frame-minor copies of what a dead window position reads, over the rows the walk can reach
        const bool df = m->kind == UMPA_DF;
        const int Na = m->Na, Nap = (Na + 7) & ~7, pitch = m->pitch, reach = m->max_shift - 1 + m->Nw;
        const int y0 = std::max(0, v.off0 - reach), y1 = std::min(H, v.off0 + (v.N0 - 1) * v.step0 + reach + 1);
        const size_t fm = (size_t)H * pitch * Nap * sizeof(float);
        if ((rc = scratch_reserve(m, m->fmS, fm)) || (rc = scratch_reserve(m, m->fmR, fm))) return rc;
        if (df && (rc = scratch_reserve(m, m->fmA, fm))) return rc;
        const size_t im = (size_t)H * pitch * sizeof(float4);
        if ((rc = scratch_reserve(m, m->fmImgS, im)) || (rc = scratch_reserve(m, m->fmImgR, im))) return rc;
        const dim3 tg((pitch + 31) / 32, y1 - y0);
        const size_t tsm = (size_t)Nap * 33 * sizeof(float);
        frame_minor_kernel<<<tg, 256, tsm, st>>>(m->d_sam32, Na, Nap, H, pitch, y0, (float *)m->fmS.p, m->d_mean_s, m->d_mean_r,
                                                 (float *)m->fmImgS.p, 0);
        frame_minor_kernel<<<tg, 256, tsm, st>>>(m->d_ref32, Na, Nap, H, pitch, y0, (float *)m->fmR.p, m->d_mean_r, m->d_mean_s,
                                                 (float *)m->fmImgR.p, 0);
        if (df) frame_minor_kernel<<<tg, 256, tsm, st>>>((const float *)m->filtA.p, Na, Nap, H, pitch, y0, (float *)m->fmA.p,
                                                         m->d_mean_r, nullptr, (float *)m->fmImgR.p, 1);
        UMPA_CUDA(cudaGetLastError());
        MaskedParams mp{};
        mp.bits = (const unsigned *)m->maskbits.p; mp.wb = W / 32 + 2;
        if ((rc = ensure_window_bits(m, st))) return rc;
        mp.dwin = m->Nw <= 3 ? (const unsigned long long *)m->maskwin.p : nullptr;
        mp.W = W;
        mp.tS = (const float *)m->fmS.p; mp.tR = (const float *)m->fmR.p; mp.tA = df ? (const float *)m->fmA.p : mp.tR;
        mp.Nap = Nap; mp.imgS = (const float4 *)m->fmImgS.p; mp.imgR = (const float4 *)m->fmImgR.p;
        mp.win = m->d_win; mp.Nw = m->Nw;
        dim3 grid((v.N1 + WALK_NT - 1) / WALK_NT, v.N0);
        if (m->refshift) {
            if (df) masked_walk_kernel<true, UMPA_DF><<<grid, WALK_NT, 0, st>>>(w, mp, v, out);
            else masked_walk_kernel<true, UMPA_NODF><<<grid, WALK_NT, 0, st>>>(w, mp, v, out);
        } else {
            if (df) masked_walk_kernel<false, UMPA_DF><<<grid, WALK_NT, 0, st>>>(w, mp, v, out);
            else masked_walk_kernel<false, UMPA_NODF><<<grid, WALK_NT, 0, st>>>(w, mp, v, out);
        }
        UMPA_CUDA(cudaGetLastError());
        m->last_launches += 6 + (df ? 1 : 0);
        m->last_path = UMPA_PATH_MASKED;
        return UMPA_OK;
    }
    if ((rc = table_match(m, v, out, st))) return rc;
    v.dirty_want = 1;
    if ((rc = lazy_match(m, v, out, st))) return rc;
    m->last_launches += 2;
    return UMPA_OK;
}
