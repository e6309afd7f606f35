// liblapf: kernels and C ABI of the B200-native LAPF step-2 hot path (see include/lapf.h).
//
// Kernels
//   K1  model_chi2_stamp_kernel / model_chi2_generic_kernel   stateless model + chi-square
//   K2  gibbs_batch_kernel  persistent sampler: a CTA owns a staged stamp (shared memory + TMEM),
//                           each warp up to 32 walkers (scalar work one walker per lane, pixel
//                           passes by the whole warp)
//       gibbs_kernel        4 or 16 warps per walker, for small batches
//   K4  totals_kernel / moments_kernel                         batch statistics
//   --  frame_prep_kernel, pack_state_kernel, peak_*_kernel
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo (olpefit_b200/build.py).
#include <algorithm>
#include <charconv>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <limits>
#include <new>
#include <string>
#include <vector>

#include <cuda.h>   // CUtensorMap (types only: the encoder is fetched from the driver at run time)

#include "../../include/lapf.h"
#include "lapf_device.cuh"

using namespace lapf;

// =============================================================================================
// error plumbing
// =============================================================================================
static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess)                                                                    \
            return fail(LAPF_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__),    \
                        __FILE__, __LINE__);                                                       \
    } while (0)

static int require_device() {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return fail(LAPF_ERR_NO_DEVICE, "no CUDA device: %s", cudaGetErrorString(e));
    int major = 0;
    e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    if (e != cudaSuccess) return fail(LAPF_ERR_NO_DEVICE, "no CUDA device: %s", cudaGetErrorString(e));
    if (major != 10)
        return fail(LAPF_ERR_NO_DEVICE, "device has compute capability %d.x; liblapf is built for sm_100a only", major);
    return LAPF_OK;
}

// liblapf takes its few temporaries (initial chi-squares, tile partials) from the device's default
// stream-ordered pool.  By default that pool hands everything back to the driver at every
// synchronisation and re-allocates on the next call -- milliseconds, now and then hundreds of them,
// in the middle of a stream of batches.  Keep the memory in the pool instead.
static void keep_pool_memory() {
    static bool done[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64 || done[dev]) return;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        uint64_t keep = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    cudaGetLastError();
    done[dev] = true;
}

// reference tables: apf_step2.py:215-217,234 and 3body/apf_step2_3body.py:220-238,292-295
static const double kWidths2[16] = {0.01, 0.01, 0.3, 0.3, 0.08, 0.09, 0.0025, 0.02,
                                    0.001, 0.0008, 0.002, 0.002, 0.001, 0.001, 0.008, 0.01};
static const double kWidths3[19] = {0.01, 0.01, 0.3, 0.3, 0.3, 0.3, 0.08, 0.09, 0.0025, 0.02,
                                    0.02, 0.001, 0.0008, 0.002, 0.002, 0.001, 0.001, 0.008, 0.01};
static const int kLog2[] = {6, 7, 9, 10, 11, 12, 13};
static const int kLog3[] = {8, 9, 10, 12, 13, 14, 15, 16};

static uint32_t log_mask_for(int nbody) {
    uint32_t m = 0;
    if (nbody == 2)
        for (int i : kLog2) m |= 1u << i;
    else
        for (int i : kLog3) m |= 1u << i;
    return m;
}

// =============================================================================================
// K1: stateless model + chi-square
// =============================================================================================
struct ProbPtrs {
    const float* data;
    const float* weight;
    const int32_t* origin;
    const double* outside;   // [F][3] or nullptr (see lapf_problem.outside)
    int n_frames, floor_index;
    int cull;                // far-field culling on/off
    int plain;               // always the plain pixel loop
};

// chi-square of the image pixels outside the cut-out, where the model is the constant floor f
__device__ __forceinline__ double outside_chi2(const double* __restrict__ outside, int frame, double f) {
    const double s0 = outside[3 * frame], s1 = outside[3 * frame + 1], s2 = outside[3 * frame + 2];
    return fma(f, fma(f, s0, -2.0 * s1), s2);
}

template <int NB, int NX, int NY, bool STORE>
__global__ void __launch_bounds__(128)
model_chi2_stamp_kernel(ProbPtrs pr, const double* __restrict__ params, int64_t B,
                        const int32_t* __restrict__ frame_of, float* __restrict__ model_out,
                        double* __restrict__ chi2_out) {
    constexpr int P = Layout<NB>::P;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t b = (int64_t)blockIdx.x * 4 + warp;
    if (b >= B) return;
    const int f = frame_of ? frame_of[b] : 0;
    if (f < 0 || f >= pr.n_frames) {
        if (lane == 0 && chi2_out) chi2_out[b] = nan("");
        return;
    }
    __shared__ float tf[4][32];
    const double mine = (lane < P) ? params[b * P + lane] : 0.0;
    stage_trial<NB>(tf[warp], lane, mine, (double)pr.origin[2 * f], (double)pr.origin[2 * f + 1]);
    Coef<NB> cf;
    load_centres_amps<NB>(cf, tf[warp]);
    cf.floor = tf[warp][pr.floor_index];
    load_shape<NB>(cf, 0, tf[warp]);
    load_shape<NB>(cf, 1, tf[warp]);
    __shared__ __align__(16) float rt[4][Scratch<NB, NX, NY>::FLOATS];
    set_fast<NB, NX, NY>(cf, lane);
    if (pr.plain) cf.fast = false;
    if (NX >= 64 && pr.cull) set_cull<NB, NX, NY>(cf, lane); else no_cull<NB, NX, NY>(cf);
    const size_t off = (size_t)f * NX * NY;
    double chi = warp_chi2<NB, NX, NY, STORE, false>(cf, rt[warp], pr.data + off, pr.weight + off,
                                                           STORE ? model_out + (size_t)b * NX * NY : nullptr, lane);
    if (lane == 0 && chi2_out)
        chi2_out[b] = pr.outside ? chi + outside_chi2(pr.outside, f, params[b * P + pr.floor_index]) : chi;
}

// 32-pixel stamps: two vectors per warp (warp_chi2_pair), the form the batched sampler uses for
// them, so the stateless operator and the sampler stay bit-identical.  The coefficients of a vector
// are worked out by the first lane of its half warp (coef_from_vector: the conversions of the
// cooperative path, one thread) and handed to the other 15 through a shared-memory image.
template <int NB, int NX, int NY, bool STORE>
__global__ void __launch_bounds__(128)
model_chi2_pair_kernel(ProbPtrs pr, const double* __restrict__ params, int64_t B,
                       const int32_t* __restrict__ frame_of, float* __restrict__ model_out,
                       double* __restrict__ chi2_out) {
    using L = Layout<NB>;
    using I = CoefImg<NB, 1>;
    constexpr int P = L::P;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, h = lane >> 4;
    const int64_t first = ((int64_t)blockIdx.x * 4 + warp) * 2;
    if (first >= B) return;
    const bool valid = first + h < B;                  // an odd batch: the last half warp repeats its neighbour's vector
    const int64_t b = valid ? first + h : first;
    const int fr = frame_of ? frame_of[b] : 0;
    const bool frame_ok = fr >= 0 && fr < pr.n_frames;
    const int f = frame_ok ? fr : 0;
    __shared__ __align__(16) float img[4][2][I::STRIDE];
    __shared__ __align__(16) float rt[4][Scratch<NB, NX, NY, 1, 2>::FLOATS];
    if ((lane & 15) == 0) {
        double v[P];
#pragma unroll
        for (int j = 0; j < P; ++j) v[j] = params[b * P + j];
        double fl = v[2 * NB];
#pragma unroll
        for (int j = 2 * NB + 1; j < P; ++j) fl = (j == pr.floor_index) ? v[j] : fl;
        Coef<NB> c0;
        coef_from_vector<NB>(c0, v, fl, (double)pr.origin[2 * f], (double)pr.origin[2 * f + 1]);
        set_fast_serial<NB, NX, NY>(c0);
        if (pr.plain) c0.fast = false;
        no_cull<NB, NX, NY>(c0);
        store_coef<NB, 1>(img[warp][h], c0);
    }
    __syncwarp();
    Coef<NB> cf;
    load_coef<NB, 1>(cf, img[warp][h]);
    const size_t off = (size_t)f * NX * NY;
    const double chi = warp_chi2_pair<NB, NX, NY, STORE, false>(cf, rt[warp], pr.data + off, pr.weight + off,
                                                                STORE ? model_out + (size_t)b * NX * NY : nullptr, lane);
    if ((lane & 15) == 0 && valid && chi2_out)
        chi2_out[b] = !frame_ok ? nan("") : (pr.outside ? chi + outside_chi2(pr.outside, f, params[b * P + pr.floor_index]) : chi);
}

// Any (ny, nx), e.g. the reference's whole 1024 x 1024 frame (apf_step2.py:94,237): grid =
// (row tiles, B); per-tile FP64 partials are summed in a fixed order by reduce_tiles_kernel.
// Centres are split into integer + fraction so pixel offsets stay accurate in FP32 at any
// distance from the frame corner.
template <int NB>
__global__ void __launch_bounds__(256)
model_chi2_generic_kernel(ProbPtrs pr, int ny, int nx, int rows_per_tile, const double* __restrict__ params,
                          const int32_t* __restrict__ frame_of, float* __restrict__ model_out,
                          double* __restrict__ partial) {
    using L = Layout<NB>;
    constexpr int K = 2 * NB;
    const int64_t b = blockIdx.y;
    const int tile = blockIdx.x, ntile = gridDim.x;
    const int f = frame_of ? frame_of[b] : 0;
    __shared__ double red[8];
    if (f < 0 || f >= pr.n_frames) {
        if (threadIdx.x == 0 && partial) partial[b * ntile + tile] = nan("");
        return;
    }
    const double* pv = params + b * L::P;
    Coef<NB> cf;
    set_shape<NB>(cf, 0, (float)pv[L::I_SX], (float)pv[L::I_SY], (float)pv[L::I_TH]);
    set_shape<NB>(cf, 1, (float)pv[L::I_SX2], (float)pv[L::I_SY2], (float)pv[L::I_TH2]);
    {
        const float ratio = (float)pv[L::I_RATIO], bkgd = (float)pv[L::I_BKGD];
#pragma unroll
        for (int o = 0; o < NB; ++o) {
            const float amp = (float)pv[L::I_AMP + o] - bkgd;   // apf_step2.py:95-97
            const float aw = amp * ratio;
            cf.amp[2 * o] = amp - aw;
            cf.amp[2 * o + 1] = aw;
        }
        cf.floor = (float)pv[pr.floor_index];
    }
    int xi[K], yi[K];
    float xf[K], yf[K];
    {
        const double dx = pv[L::I_DX], dy = pv[L::I_DY];
        const int ox = pr.origin[2 * f], oy = pr.origin[2 * f + 1];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int o = k >> 1;
            const double xc = pv[2 * o] - (double)ox + ((k & 1) ? dx : 0.0);
            const double yc = pv[2 * o + 1] - (double)oy + ((k & 1) ? dy : 0.0);
            // clamp so the int conversion is defined for wild proposals; exactness only matters nearby
            const double fx = floor(fmin(fmax(xc, -1e9), 1e9)), fy = floor(fmin(fmax(yc, -1e9), 1e9));
            xi[k] = (int)fx;
            yi[k] = (int)fy;
            xf[k] = (float)(xc - fx);
            yf[k] = (float)(yc - fy);
        }
    }
    const float* d = pr.data + (size_t)f * ny * nx;
    const float* w = pr.weight + (size_t)f * ny * nx;
    float* mo = model_out ? model_out + (size_t)b * ny * nx : nullptr;
    const int r0 = tile * rows_per_tile, r1 = min(ny, r0 + rows_per_tile);
    double acc = 0.0;
    for (int r = r0; r < r1; ++r) {
        float yd[K];
#pragma unroll
        for (int k = 0; k < K; ++k) yd[k] = (float)(r - yi[k]) - yf[k];
        for (int c = threadIdx.x; c < nx; c += blockDim.x) {
            float m = cf.floor;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const float xd = (float)(c - xi[k]) - xf[k];
                const float t = fmaf(cf.sa[k & 1], xd, cf.sb[k & 1] * yd[k]);
                const float q = fmaf(xd, t, (cf.sc[k & 1] * yd[k]) * yd[k]);
                m = fmaf(cf.amp[k], ex2_approx(q), m);
            }
            const size_t idx = (size_t)r * nx + c;
            if (mo) mo[idx] = m;
            const float sq = sqrtf(w[idx]);
            const float res = fmaf(-sq, m, d[idx] * sq);
            acc += (double)(res * res);
        }
    }
    acc = warp_sum_f64(acc);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0 && partial) {
        double s = 0.0;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s += red[i];
        if (tile == 0 && pr.outside) s += outside_chi2(pr.outside, f, pv[pr.floor_index]);
        partial[b * ntile + tile] = s;
    }
}

__global__ void reduce_tiles_kernel(const double* __restrict__ partial, int ntile, int64_t B,
                                    double* __restrict__ chi2_out) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    double s = 0.0;
    for (int t = 0; t < ntile; ++t) s += partial[b * ntile + t];
    chi2_out[b] = s;
}

// =============================================================================================
// K2: persistent Gibbs sampler
// =============================================================================================
struct RunArgs {
    const float* data;
    const float* weight;
    const int32_t* origin;
    const double* outside;       // [F][3] or nullptr
    const int32_t* item_frame;   // [n_items]
    const int32_t* item_first;   // [n_items] offset into walker_of
    const int32_t* item_count;   // [n_items] walkers in the item (<= warps per CTA)
    // batched kernel: an item may hold walkers of TWO frames, both resident in the pixel store (slots 0 and 1):
    // the first item_count_a walkers belong to the frame of slot item_slot_a, the others to the other slot
    const int32_t* item_frame2;  // [n_items] frame of slot 1 (-1: none); item_frame is the frame of slot 0
    const int32_t* item_count_a; // [n_items]
    const int32_t* item_slot_a;  // [n_items]
    const int32_t* walker_of;    // local walker indices grouped by frame
    const int32_t* cta_item;     // [grid + 1] first item of every CTA (batched kernel only)
    double* state;               // [W][P+1]  parameters, chi-square
    const double* shift;         // [W][P+1]  initial state (shift of the running moments)
    double* moments;             // [W][P+1][2] running sum / sum of squares of recorded rows
    uint32_t* tries;             // [W][P]
    uint32_t* accepts;           // [W][P]
    unsigned long long* exps;    // [W] exponentials actually evaluated (after far-field culling)
    void* chain;                 // [rows][W][P+1] double, or float (value - shift) when chain_f32; or nullptr
                                 // (chain_ev: row 0 only, the key of the event buffer)
    // event formats (chain_ev): per recorded row and walker one code byte (k | accepted << 7), the value of
    // column k and chi-square, as double or as float (value - shift) like the rows; parts of the chain buffer
    unsigned char* ev_code;      // [rows][W]
    void* ev_val;                // [rows][W]
    void* ev_chi;                // [rows][W]
    // separation / position-angle sketches of the recorded rows (apf_step3.py:255-256,283-291), or nullptr
    uint32_t* sk_hist;           // [F][NB-1][2][sk_bins + 2]: underflow, bins, overflow
    const double* sk_center;     // [F][NB-1][2]: separation (pixels), position angle (degrees) of bin sk_bins / 2
    double* sk_mom;              // [W][NB-1][2][2]: per walker sum / sum of squares of (value - centre)
    double sk_inv_sep, sk_inv_pa;   // 1 / bin width
    int sk_bins, chain_f32, chain_ev;
    // batch means (lapf_sampler_batchmeans_enable), or nullptr: per walker, quantity (the P+1 columns, then
    // the sketch slots) and level l the running sum at the last level-l boundary and the sum of squared batch sums
    double* bm;                  // [W][bm_c][bm_levels][2]
    int64_t bm_q0;               // complete bm_rows-row batches of every walker before this launch
    int bm_rows, bm_phase;       // batch length of level 0; rows recorded since the last level-0 boundary
    int bm_levels, bm_c;
    // posterior draws (lapf_sampler_draws_enable), or nullptr: a reservoir of dr_k recorded rows per walker
    double* dr_val;              // [W][dr_k][P+1]
    int64_t* dr_row;             // [W][dr_k] recorded-row index of the slot, -1: empty
    int64_t dr_row0;             // rows every walker recorded before this launch
    int dr_k;
    // per-frame jump widths (lapf_sampler_set_frame_widths), or nullptr: the proposal of a walker of frame f
    // reads fwidths[f * P + k] instead of widths[k]
    const double* fwidths;       // [F][P]
    // parameter priors (lapf_sampler_set_priors), or nullptr: per frame and parameter the box [lo, hi] and the
    // Gaussian term's mu and h = 0.5 / sigma^2 (0: none)
    const double* prior;         // [F][P][4] lo, hi, mu, h
    double* probe;               // self-test only: [rows][W][3] = parameter index (-1 - index: the proposal lay
                                 // outside its box, no pass), proposed value, TRIAL chi-square
    unsigned long long* cta_times;   // diagnosis only (LAPF_CTA_TIMES): [CTAs][3] = start, end (globaltimer ns), SM id
    int64_t n_walkers;
    int64_t t0, n_updates;       // first update index, updates in this launch
    int64_t next_record;         // first count >= t0+1 at which a row is recorded
    int64_t id_base, id_stride;
    uint64_t seed;
    double widths[LAPF_MAX_PARAMS];
    uint32_t log_mask;
    int thin, floor_index, n_items, cull, plain;
};

// Batch means: the number of levels that launch-relative row `row` closes.  With it the walker has
// recorded bm_q0 * bm_rows + bm_phase + row + 1 rows; level l closes when that count is a multiple
// of bm_rows * 2^l.  0 when batch means are off or the row closes no batch (all but one row in bm_rows).
__device__ __forceinline__ int bm_closing(const RunArgs& a, int row) {
    if (!a.bm) return 0;
    const int r = a.bm_phase + row + 1;
    if (r % a.bm_rows) return 0;
    return min(__ffsll((long long)(a.bm_q0 + r / a.bm_rows)), a.bm_levels);
}

// Close the first n_lev levels of quantity c (< bm_c) of walker wl once the row's running sums are
// stored: S = M1 - snap, s2 += S*S, snap = M1, never contracted (DESIGN.md 5: the tests restate it bit
// for bit).  M1 is read back from L2, where this thread -- its single writer -- performed its atomics:
// exactly the value the last atomicAdd stored.  So the moment updates stay fire-and-forget REDs, with
// batch means on or off, and no return value is held in registers through the row.
template <int NB>
__device__ __forceinline__ void bm_close(const RunArgs& a, int wl, int c, int n_lev) {
    constexpr int P = Layout<NB>::P;
    const double m1 = __ldcg(c <= P ? a.moments + 2 * ((size_t)wl * (P + 1) + c)
                                    : a.sk_mom + 2 * ((size_t)wl * (a.bm_c - P - 1) + (c - P - 1)));
    double* b = a.bm + ((size_t)wl * a.bm_c + c) * a.bm_levels * 2;
#pragma unroll 1
    for (int l = 0; l < n_lev; ++l) {
        const double S = __dsub_rn(m1, b[2 * l]);
        b[2 * l + 1] = __dadd_rn(b[2 * l + 1], __dmul_rn(S, S));
        b[2 * l] = m1;
    }
}

// Quantities a recorded row adds to: the P+1 columns, and the sketch slots when sketches are recorded
// (the self-test records none)
template <int NB>
__device__ __forceinline__ int bm_quantities(const RunArgs& a) { return a.sk_hist ? a.bm_c : Layout<NB>::P + 1; }

// One recorded row of one walker enters the sketches of its frame: for every companion the
// separation sqrt(dx^2 + dy^2) in pixels and the position angle degrees(atan2(-dx, dy))
// (apf_step3.py:255-256,283-291; 3-body: both pairs, 3body/apf_step3_3body.py:273-276,318-324)
// relative to the frame's centre values, into fixed-width bins (integer atomics: order-independent)
// and into the walker's own running sums (single writer: deterministic).
template <int NB>
__device__ __forceinline__ void record_sketch(const RunArgs& a, int wl, int frame, const double* __restrict__ xy) {
    const double xs = xy[0], ys = xy[1];
#pragma unroll
    for (int o = 1; o < NB; ++o) {
        const double dx = xy[2 * o] - xs, dy = xy[2 * o + 1] - ys;
        const double val[2] = {sqrt(dx * dx + dy * dy), atan2(-dx, dy) * 57.29577951308232};
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const size_t slot = ((size_t)frame * (NB - 1) + (o - 1)) * 2 + q;
            double d = val[q] - a.sk_center[slot];
            if (q == 1) d -= 360.0 * rint(d * (1.0 / 360.0));            // angles wrap
            const double pos = floor(d * (q ? a.sk_inv_pa : a.sk_inv_sep)) + (double)(a.sk_bins / 2);
            // nan goes to the overflow bin
            const int bin = (pos >= 0.0) ? ((pos < (double)a.sk_bins) ? 1 + (int)pos : a.sk_bins + 1) : ((pos < 0.0) ? 0 : a.sk_bins + 1);
            atomicAdd(&a.sk_hist[slot * (size_t)(a.sk_bins + 2) + bin], 1u);
            double* m = a.sk_mom + (((size_t)wl * (NB - 1) + (o - 1)) * 2 + q) * 2;
            atomicAdd(m, d);
            atomicAdd(m + 1, d * d);
        }
    }
}

// Priors (lapf_sampler_set_priors): `pr` is the table entry {lo, hi, mu, h} of the walker's frame and the
// updated parameter.  A value outside the box (or nan) is outside.
__device__ __forceinline__ bool prior_outside(const double* pr, double v) { return !(v >= pr[0] && v <= pr[1]); }
// The Gaussian term of the Metropolis ratio for a move pk -> nv, g = h ((nv - mu)^2 - (pk - mu)^2); 0 without one
// (h = 0: never multiplied, 0 * inf would be nan).  Rounded to nearest and never contracted (DESIGN.md 5): the
// tests restate it in numpy.
__device__ __forceinline__ double prior_g(const double* pr, double nv, double pk) {
    const double h = pr[3];
    if (h == 0.0) return 0.0;
    const double dn = __dsub_rn(nv, pr[2]), dp = __dsub_rn(pk, pr[2]);
    return __dmul_rn(h, __dsub_rn(__dmul_rn(dn, dn), __dmul_rn(dp, dp)));
}

// One walker for n_updates updates.  TEAM = 1: one warp does everything.  TEAM > 1 (few walkers,
// latency matters): TEAM warps run this function for the SAME walker in lock-step; each repeats the
// cheap scalar part (identical inputs, identical results), evaluates its share of the rows, and the
// partial chi-squares meet in shared memory behind one named barrier per update.  Only warp 0 of
// the team writes counters, chain rows and the final state.
template <int NB, int NX, int NY, int TEAM>
__device__ __forceinline__ void run_walker(const RunArgs& a, const float* sd, const float* sw,
                                           WarpScratch& ws, float* rt, float* team_ct, double* team_part, int team,
                                           int tw, int wl, int frame, int lane) {
    using L = Layout<NB>;
    constexpr int P = L::P;
    const uint64_t gid = (uint64_t)(a.id_base + (int64_t)wl * a.id_stride);
    const double oxd = (double)a.origin[2 * frame], oyd = (double)a.origin[2 * frame + 1];
    double* st = a.state + (size_t)wl * (P + 1);

    // lane j < P owns parameter j; lane P holds chi-square
    double p = (lane <= P) ? st[lane] : 0.0;
    double chi_c = shfl_f64(p, P);

    Coef<NB> cf;
    stage_trial<NB>(ws.tf, lane, p, oxd, oyd);
    {
        float s0, c0, s1, c1;
        sincosf(ws.tf[L::I_TH], &s0, &c0);
        sincosf(ws.tf[L::I_TH2], &s1, &c1);
        set_shape_sc<NB>(cf, 0, ws.tf[L::I_SX], ws.tf[L::I_SY], s0, c0);
        set_shape_sc<NB>(cf, 1, ws.tf[L::I_SX2], ws.tf[L::I_SY2], s1, c1);
        if (lane == 0) {
            ws.shape[0] = cf.sa[0]; ws.shape[1] = cf.sb[0]; ws.shape[2] = cf.sc[0];
            ws.shape[4] = cf.sa[1]; ws.shape[5] = cf.sb[1]; ws.shape[6] = cf.sc[1];
            ws.trig[0] = s0; ws.trig[1] = c0; ws.trig[2] = s1; ws.trig[3] = c1;
        }
    }

    // launch-relative 32-bit counters (lapf_sampler_run caps a launch at 2^30 updates)
    const int n_upd = (int)a.n_updates;
    int next_rec = (int)min(a.next_record - a.t0 - 1, (int64_t)0x7fffffff);   // update index that records next
    int row = 0;
    unsigned long long n_exps = 0;

#pragma unroll 1
    for (int u = 0; u < n_upd; ++u) {
        const int slot = u & 31;
        if (slot == 0) {
            // lane l prepares the draws of update t0+u+l: 32 updates of random numbers at once
            const Draw dr = make_draw(a.seed, gid, (uint64_t)(a.t0 + u + lane), P);
            const double wk = a.fwidths ? a.fwidths[(size_t)frame * P + dr.k] : a.widths[dr.k];   // (uniform branch)
            const double wz = __dmul_rn(wk, dr.z);    // never contracted into the sum below (lapf_device.cuh, set_shape_sc)
            __syncwarp();
            ws.k[lane] = dr.k;
            ws.step[lane] = ((a.log_mask >> dr.k) & 1u) ? exp10(wz) : wz;
            ws.lnu[lane] = dr.lnu;
            // posterior draws: the next 32 updates record at most 32 rows, row .. row + 31; lane l decides row + l
            if (a.dr_val && tw == 0) ws.dslot[(row + lane) & 31] = draw_slot(a.seed, gid, (uint64_t)(a.dr_row0 + row + lane), a.dr_k);
            __syncwarp();
        }
        const int k = ws.k[slot];                                     // apf_step2.py:302
        const double step = ws.step[slot];
        const double pk = shfl_f64(p, k);
        // proposal (apf_step2.py:63-70): additive, or multiplicative 10^(w z) for the log10
        // parameters; log10 of a negative value is nan there, and 0 stays 0.
        const double nv = ((a.log_mask >> k) & 1u) ? (pk < 0.0 ? nan("") : __dmul_rn(pk, step)) : __dadd_rn(pk, step);

        stage_trial<NB>(ws.tf, lane, (lane == k) ? nv : p, oxd, oyd);  // :312-313
        load_centres_amps<NB>(cf, ws.tf);
        cf.floor = ws.tf[a.floor_index];
        {
            const float4 s0 = *reinterpret_cast<const float4*>(&ws.shape[0]);
            const float4 s1 = *reinterpret_cast<const float4*>(&ws.shape[4]);
            cf.sa[0] = s0.x; cf.sb[0] = s0.y; cf.sc[0] = s0.z;
            cf.sa[1] = s1.x; cf.sb[1] = s1.y; cf.sc[1] = s1.z;
        }
        // a shape parameter moved: redo that shape's a, b, c; sin/cos only if its angle moved
        const bool shape_moved = k >= L::I_SX;
        const int which = (k == L::I_SX2 || k == L::I_SY2 || k == L::I_TH2) ? 1 : 0;
        float tsin = 0.f, tcos = 1.f;
        if (shape_moved) {
            const float4 tg = *reinterpret_cast<const float4*>(&ws.trig[0]);
            if (which) {
                tsin = tg.z; tcos = tg.w;
                if (k == L::I_TH2) sincosf(ws.tf[L::I_TH2], &tsin, &tcos);
                set_shape_sc<NB>(cf, 1, ws.tf[L::I_SX2], ws.tf[L::I_SY2], tsin, tcos);
            } else {
                tsin = tg.x; tcos = tg.y;
                if (k == L::I_TH) sincosf(ws.tf[L::I_TH], &tsin, &tcos);
                set_shape_sc<NB>(cf, 0, ws.tf[L::I_SX], ws.tf[L::I_SY], tsin, tcos);
            }
        }
        set_fast<NB, NX, NY>(cf, lane);
        if (a.plain) cf.fast = false;
        // in a team the update time is set by the warp with the busiest rows: culling cannot help there
        if (NX >= 64 && TEAM == 1 && a.cull) set_cull<NB, NX, NY, TEAM>(cf, lane); else no_cull<NB, NX, NY, TEAM>(cf);
        if (TEAM > 1 && cf.fast) {
            // the column tables of this proposal, by the whole team; the barrier at the end of the previous
            // update (partials) lies between the last reader of the old table and these writes
            team_consts<NB, NX, TEAM>(team_ct, cf, tw * 32 + lane);
            asm volatile("bar.sync %0, %1;" ::"r"(1 + team), "r"(TEAM * 32) : "memory");
        }
        unsigned e_upd = 0;
        double chi_t;                                                                                 // :314-316
        if constexpr (TEAM > 1) chi_t = team_chi2<NB, NX, NY, TEAM>(cf, rt, sd, sw, lane, tw, &e_upd, team_ct);
        else chi_t = warp_chi2<NB, NX, NY, false, true, 1>(cf, rt, sd, sw, nullptr, lane, 0, &e_upd, 0u);
        n_exps += e_upd;
        if (TEAM > 1) {
            double* slot_p = team_part + (u & 1) * TEAM;       // double-buffered: one barrier per update
            if (lane == 0) slot_p[tw] = chi_t;
            asm volatile("bar.sync %0, %1;" ::"r"(1 + team), "r"(TEAM * 32) : "memory");
            // the same fixed pairwise tree in every warp of the team (depth log2 TEAM, not a chain of TEAM additions)
            double v[TEAM];
#pragma unroll
            for (int t = 0; t < TEAM; ++t) v[t] = slot_p[t];
#pragma unroll
            for (int h = TEAM / 2; h >= 1; h >>= 1)
#pragma unroll
                for (int t = 0; t < h; ++t) v[t] += v[t + h];
            chi_t = v[0];
        }
        if (a.outside) chi_t += outside_chi2(a.outside, frame, (k == a.floor_index) ? nv : shfl_f64(p, a.floor_index));

        // priors: a proposal outside its box was evaluated like any other (every warp of the team keeps the
        // barrier count) and is rejected here; the Gaussian term joins the ratio
        bool in_box = true;
        double g = 0.0;
        if (a.prior) {                                                // (uniform branch)
            const double* pr = a.prior + ((size_t)frame * P + k) * 4;
            in_box = !prior_outside(pr, nv);
            g = prior_g(pr, nv, shfl_f64(p, k));                      // p is still the state before the update
        }
        // accept iff u < exp(-(chi_t - chi_c)/2 - g) (apf_step2.py:139-148); false on nan
        const bool acc = in_box && ws.lnu[slot] < __dsub_rn(__dmul_rn(-0.5, __dsub_rn(chi_t, chi_c)), g);
        if (lane == 0 && tw == 0) {
            atomicAdd(&a.tries[(size_t)wl * P + k], 1u);              // :304
            if (acc) atomicAdd(&a.accepts[(size_t)wl * P + k], 1u);   // :323
        }
        if (acc) {
            if (lane == k) p = nv;                                    // :325
            chi_c = chi_t;                                            // :327
            if (shape_moved && lane == 0) {   // constant indices only: keeps cf in registers
                if (which) { ws.shape[4] = cf.sa[1]; ws.shape[5] = cf.sb[1]; ws.shape[6] = cf.sc[1];
                             ws.trig[2] = tsin; ws.trig[3] = tcos; }
                else       { ws.shape[0] = cf.sa[0]; ws.shape[1] = cf.sb[0]; ws.shape[2] = cf.sc[0];
                             ws.trig[0] = tsin; ws.trig[1] = tcos; }
            }
        }
        if (u == next_rec) {                                          // :342-351
            if (lane <= P && tw == 0) {
                const size_t mi = (size_t)wl * (P + 1) + lane;
                const double v = (lane == P) ? chi_c : p;
                const double dl = v - a.shift[mi];
                if (a.chain && (row == 0 || !a.chain_ev)) {           // events: row 0 is the key
                    const size_t ci = ((size_t)row * a.n_walkers + wl) * (P + 1) + lane;
                    if (a.chain_f32) static_cast<float*>(a.chain)[ci] = (float)dl; else static_cast<double*>(a.chain)[ci] = v;
                }
                if (a.chain_ev && (lane == k || lane == P)) {            // the lanes that hold column k and chi-square
                    const size_t ei = (size_t)row * a.n_walkers + wl;
                    if (lane == k) a.ev_code[ei] = (unsigned char)(k | (acc ? 0x80 : 0));
                    void* dst = (lane == k) ? a.ev_val : a.ev_chi;
                    if (a.chain_f32) static_cast<float*>(dst)[ei] = (float)dl; else static_cast<double*>(dst)[ei] = v;
                }
                atomicAdd(&a.moments[2 * mi], dl);                    // single writer: plain RED, in order
                atomicAdd(&a.moments[2 * mi + 1], dl * dl);
                if (const int n_lev = bm_closing(a, row)) bm_close<NB>(a, wl, lane, n_lev);   // lane c closes column c
                if (a.dr_val) {                                          // lane c writes column c of the slot
                    const int j = ws.dslot[row & 31];
                    if (j >= 0) {
                        const size_t di = (size_t)wl * a.dr_k + j;
                        a.dr_val[di * (P + 1) + lane] = v;
                        if (lane == 0) a.dr_row[di] = a.dr_row0 + row;
                    }
                }
            }
            if (a.sk_hist) {
                double xy[2 * NB];
#pragma unroll
                for (int j = 0; j < 2 * NB; ++j) xy[j] = shfl_f64(p, j);
                if (lane == 0 && tw == 0) {
                    record_sketch<NB>(a, wl, frame, xy);
                    if (const int n_lev = bm_closing(a, row))
#pragma unroll 1
                        for (int c = Layout<NB>::P + 1; c < a.bm_c; ++c) bm_close<NB>(a, wl, c, n_lev);
                }
            }
            ++row;
            next_rec += a.thin;   // (saturates harmlessly: a launch is shorter than 2^30)
        }
    }

    if (tw == 0) {
        if (lane < P) st[lane] = p;
        if (lane == P) st[P] = chi_c;
        if (lane == 0) a.exps[wl] += n_exps;
    }
}

template <int NB, int NX, int NY, int NW, int MINB, int TEAM>
__global__ void __launch_bounds__(NW * 32, MINB) gibbs_kernel(const __grid_constant__ RunArgs a) {
    static_assert(NW % TEAM == 0 && (TEAM == 1 || NW / TEAM <= 15), "teams must tile the CTA (named barriers 1..15)");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ WarpScratch scratch[NW];
    __shared__ double team_part[NW / TEAM][2 * TEAM];
    __shared__ uint64_t bar;
    float* sd = reinterpret_cast<float*>(smem_raw);
    float* sw = sd + NX * NY;
    float* rt = sw + NX * NY;                       // [NW] row + column tables (Scratch)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) mbar_init(&bar, 1);
    __syncthreads();

    // contiguous share of the item list: consecutive items mostly share a frame
    const int i0 = (int)(((int64_t)a.n_items * blockIdx.x) / gridDim.x);
    const int i1 = (int)(((int64_t)a.n_items * (blockIdx.x + 1)) / gridDim.x);
    int cur_frame = -1;
    uint32_t phase = 0;
    for (int it = i0; it < i1; ++it) {
        const int f = a.item_frame[it];
        if (f != cur_frame) {
            __syncthreads();   // every warp has finished reading the previous stamp
            if (threadIdx.x == 0) {
                constexpr uint32_t kBytes = NX * NY * sizeof(float);
                fence_proxy_async();
                mbar_expect_tx(&bar, 2 * kBytes);
                tma_bulk_g2s(sd, a.data + (size_t)f * NX * NY, kBytes, &bar);
                tma_bulk_g2s(sw, a.weight + (size_t)f * NX * NY, kBytes, &bar);
            }
            mbar_wait(&bar, phase);
            phase ^= 1u;
            cur_frame = f;
            prep_stamp(sd, sw, NX * NY);            // (d, w) -> (d*sqrt(w), -sqrt(w)), once per staged frame
            __syncthreads();
        }
        const int team = warp / TEAM, tw = warp % TEAM;
        if (team < a.item_count[it]) {
            using S = Scratch<NB, NX, NY, TEAM>;
            float* base = rt + team * (TEAM > 1 ? S::TEAM_FLOATS : S::FLOATS);
            run_walker<NB, NX, NY, TEAM>(a, sd, sw, scratch[warp], base + (TEAM > 1 ? tw * S::TAB : 0), base + TEAM * S::TAB,
                                         team_part[team], team, tw, a.walker_of[a.item_first[it] + team], f, lane);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Batched form (team_warps = 1, the throughput configuration).  A warp owns up to LW walkers of
// the staged frame.  Everything that is scalar work per walker -- random numbers, proposal,
// coefficients of the trial vector, culling bounds, accept/reject, counters, chain row -- is done
// with ONE WALKER PER LANE, once per round, and costs 1/LW of a warp instruction per update.  In
// between, the warp evaluates the trial vectors one after the other (a "pass": block table, lane
// constants, pixel loop, FP64 reduction of the lane partials), reading each walker's coefficients
// from its shared-memory image.  At 64 pixels the reduction of all passes waits for the end of the
// round: a pass leaves its lane partials in the image it has read, and each walker's lane adds its
// 32 partials in the butterfly's order (warp_sum_f64_of).  FP64 state lives in global memory
// (L1/L2 resident: one parameter read and at most one written per update).  The arithmetic per
// walker is the one of run_walker: chains are bit-identical between the two forms.
// ---------------------------------------------------------------------------------------------
// `frame0`, `frame1`: the frames in the two pixel-store slots (frame1 < 0: none; both uniform over the CTA);
// `slot`: the slot of the lane's walker; `la`: lanes [0, la) of this warp use one slot, [la, nl) the other
// (la = nl: one frame); `slot_cols`: TMEM columns per slot.  Everything per frame is kept uniform and picked
// by `slot` where it is used: a per-lane frame held the origins in vector registers through the passes and
// cost 2 % at 128 pixels.
template <int NB, int NX, int NY, int LW, int TM, int WPP>
__device__ __forceinline__ void run_batch(const RunArgs& a, const float* sd, const float* sw, float* rt, float* img,
                                          int wl, int nl, int la, int frame0, int frame1, int slot, int lane,
                                          uint32_t tmem, uint32_t slot_cols) {
    using L = Layout<NB>;
    using I = CoefImg<NB, Geo<NX>::PANELS>;
    constexpr int P = L::P;
    // one-panel, one-table stamps evaluated one walker per pass (64 pixels): see the passes below
    constexpr bool LANE_SUMS = WPP == 1 && Geo<NX>::PANELS == 1 && Rows<NY, 1>::HALVES == 1;
    static_assert(!LANE_SUMS || I::STRIDE >= 32, "a walker's image holds the 32 lane partials of its pass");
    const bool mine = wl >= 0;
    const uint64_t gid = (uint64_t)(a.id_base + (int64_t)wl * a.id_stride);
    const bool two = TM == 1 && frame1 >= 0;
    const int ox0 = a.origin[2 * frame0], oy0 = a.origin[2 * frame0 + 1];
    const int ox1 = two ? a.origin[2 * frame1] : ox0, oy1 = two ? a.origin[2 * frame1 + 1] : oy0;
    double* st = a.state + (size_t)(mine ? wl : 0) * (P + 1);
    double chi_c = mine ? st[P] : 0.0;

    const int n_upd = (int)a.n_updates;
    int next_rec = (int)min(a.next_record - a.t0 - 1, (int64_t)0x7fffffff);   // update index that records next
    int row = 0;
    unsigned long long n_exps = 0;

#pragma unroll 1
    for (int u = 0; u < n_upd; ++u) {
        // ---- one walker per lane: draws, proposal, coefficients of the trial vector -------------
        int k = 0;
        double nv = 0.0, lnu = 0.0;
        bool skip = false;
        if (mine) {
            const Draw dr = make_draw(a.seed, gid, (uint64_t)(a.t0 + u), P);   // apf_step2.py:302, :64/:68, :143
            const double oxd = (double)((two && slot) ? ox1 : ox0), oyd = (double)((two && slot) ? oy1 : oy0);
            k = dr.k;
            lnu = dr.lnu;
            // per-frame widths: the lane's frame, picked like its origin (uniform branch)
            const double wk = a.fwidths ? a.fwidths[(size_t)((two && slot) ? frame1 : frame0) * P + k] : a.widths[k];
            const double wz = __dmul_rn(wk, dr.z);
            const bool is_log = (a.log_mask >> k) & 1u;
            double v[P];
#pragma unroll
            for (int j = 0; j < P; ++j) v[j] = st[j];
            double pk = v[0];
#pragma unroll
            for (int j = 1; j < P; ++j) pk = (j == k) ? v[j] : pk;
            // proposal (apf_step2.py:63-70): additive, or multiplicative 10^(w z) for the log10
            // parameters; log10 of a negative value is nan there, and 0 stays 0.
            nv = is_log ? (pk < 0.0 ? nan("") : __dmul_rn(pk, exp10(wz))) : __dadd_rn(pk, wz);
#pragma unroll
            for (int j = 0; j < P; ++j) v[j] = (j == k) ? nv : v[j];            // :312-313
            double fl = v[2 * NB];
#pragma unroll
            for (int j = 2 * NB + 1; j < P; ++j) fl = (j == a.floor_index) ? v[j] : fl;
            Coef<NB> cf;
            coef_from_vector<NB>(cf, v, fl, oxd, oyd);
            set_fast_serial<NB, NX, NY>(cf);
            if (a.plain) cf.fast = false;
            if (NX >= 64 && a.cull) set_cull_serial<NB, NX, NY>(cf); else no_cull<NB, NX, NY>(cf);
            // A proposal that is nan by construction (log10 of a negative value, apf_step2.py:66-70: a start
            // with a negative background never moves it) has chi-square nan and is rejected (:139-148): its
            // pass is skipped instead of sending a nan vector through the plain loop at twice the cost of a
            // pass.  (With two vectors per pass it keeps its partner company in the factorised loop instead.)
            // With priors, so is a proposal outside its frame's box (nan is outside every box).
            skip = a.prior ? prior_outside(a.prior + ((size_t)((two && slot) ? frame1 : frame0) * P + k) * 4, nv) : nv != nv;
            if (skip && WPP > 1) cf.fast = true;
            if (LANE_SUMS && !skip) n_exps += cf.nexp;
            store_coef<NB, Geo<NX>::PANELS>(img + lane * I::STRIDE, cf, slot | (skip ? 2 : 0));
        }
        __syncwarp();

        // ---- passes: the warp evaluates chi-square of its walkers' trial vectors in turn --------
        double chi_t = 0.0;
        if constexpr (LANE_SUMS) {
            // each pass leaves its 32 lane partials in its walker's image (read, hence dead, by then); the
            // walker's lane reduces them after the last pass: one reduction per round instead of a butterfly per pass
#pragma unroll 1
            for (int i = 0; i < nl; ++i) {
                Coef<NB> cf;
                int sl = 0;
                float* slot_img = img + i * I::STRIDE;
                load_coef<NB, 1>(cf, slot_img, &sl);
                if (sl & 2) continue;                   // a nan proposal: no pass (uniform: the image is the warp's)
                __syncwarp();                           // every lane has read the image before any lane overwrites it
                const float part = lane_chi2<NB, NX, NY, TM>(cf, rt, sd, sw, lane,
                                                             TM == 1 ? tmem + (uint32_t)(sl & 1) * slot_cols : tmem);   // :314-316
                slot_img[lane] = part;
            }
            __syncwarp();
            if (mine) chi_t = warp_sum_f64_of(img + lane * I::STRIDE);
        } else if constexpr (WPP == 1) {
#pragma unroll 1
            for (int i = 0; i < nl; ++i) {
                Coef<NB> cf;
                int sl = 0;
                load_coef<NB, Geo<NX>::PANELS>(cf, img + i * I::STRIDE, &sl);
                if (sl & 2) continue;                   // a nan proposal: no pass (uniform: the image is the warp's)
                unsigned e_upd = 0;
                const double c = warp_chi2<NB, NX, NY, false, true, 1, TM>(cf, rt, sd, sw, nullptr, lane, 0, &e_upd,
                                                                           TM == 1 ? tmem + (uint32_t)(sl & 1) * slot_cols : tmem);   // :314-316
                if (lane == i) { chi_t = c; n_exps += e_upd; }
            }
        } else {
            // two walkers per pass: lanes 0-15 evaluate walker i, lanes 16-31 walker i + 1 (or i again, discarded);
            // both of the same pixel-store slot (the TMEM address of a load is the warp's): walkers [0, la), then [la, nl)
#pragma unroll 1
            for (int seg = 0; seg < 2; ++seg) {
                const int i0 = seg ? la : 0, i1 = seg ? nl : la;
#pragma unroll 1
                for (int i = i0; i < i1; i += 2) {
                    const int mine_i = min(i + (lane >> 4), i1 - 1);
                    Coef<NB> cf;
                    int sl = 0;
                    load_coef<NB, 1>(cf, img + mine_i * I::STRIDE, &sl);
                    if (__all_sync(kFull, (sl & 2) != 0)) continue;      // both are nan proposals: no pass
                    sl = __shfl_sync(kFull, sl, 0) & 1;
                    unsigned e_upd = 0;
                    const double c = warp_chi2_pair<NB, NX, NY, false, true, TM>(cf, rt, sd, sw, nullptr, lane, &e_upd,
                                                                                 tmem + (uint32_t)sl * slot_cols);   // :314-316
                    const double c0 = shfl_f64(c, 0), c1 = shfl_f64(c, 16);
                    const unsigned e0 = __shfl_sync(kFull, e_upd, 0), e1 = __shfl_sync(kFull, e_upd, 16);
                    if (lane == i) { chi_t = c0; n_exps += e0; }
                    if (lane == i + 1 && i + 1 < i1) { chi_t = c1; n_exps += e1; }
                }
            }
        }
        __syncwarp();   // every pass has read its image before the next round overwrites it

        // ---- one walker per lane: accept / reject, counters, chain row --------------------------
        if (mine) {
            if (skip) chi_t = nan("");
            if (a.outside) {
                double fl = st[a.floor_index];
                if (k == a.floor_index) fl = nv;
                chi_t += outside_chi2(a.outside, (two && slot) ? frame1 : frame0, fl);
            }
            // priors: the Gaussian term from the table and st[k], which still holds pk (a skipped proposal has
            // chi_t = nan and is rejected whatever g is)
            const double g = a.prior ? prior_g(a.prior + ((size_t)((two && slot) ? frame1 : frame0) * P + k) * 4, nv, st[k]) : 0.0;
            // accept iff u < exp(-(chi_t - chi_c)/2 - g) (apf_step2.py:139-148); false on nan
            const bool acc = lnu < __dsub_rn(__dmul_rn(-0.5, __dsub_rn(chi_t, chi_c)), g);
            atomicAdd(&a.tries[(size_t)wl * P + k], 1u);                  // :304
            if (acc) {
                atomicAdd(&a.accepts[(size_t)wl * P + k], 1u);            // :323
                st[k] = nv;                                               // :325
                chi_c = chi_t;                                            // :327
            }
            if (a.chain_ev && u == next_rec) {                            // the event of this row
                const size_t ei = (size_t)row * a.n_walkers + wl, si = (size_t)wl * (P + 1);
                a.ev_code[ei] = (unsigned char)(k | (acc ? 0x80 : 0));
                const double kv = st[k];
                if (a.chain_f32) {
                    static_cast<float*>(a.ev_val)[ei] = (float)(kv - a.shift[si + k]);
                    static_cast<float*>(a.ev_chi)[ei] = (float)(chi_c - a.shift[si + P]);
                } else {
                    static_cast<double*>(a.ev_val)[ei] = kv;
                    static_cast<double*>(a.ev_chi)[ei] = chi_c;
                }
            }
        }
        if (u == next_rec) {                                              // :342-351
            if (mine) {
                const bool dense = a.chain && (row == 0 || !a.chain_ev);   // events: row 0 is the key
                double* dv = nullptr;                                     // posterior draws: the slot this row takes
                if (a.dr_val) {
                    const int64_t n = a.dr_row0 + row;
                    const int jd = draw_slot(a.seed, gid, (uint64_t)n, a.dr_k);
                    if (jd >= 0) {
                        const size_t di = (size_t)wl * a.dr_k + jd;
                        a.dr_row[di] = n;
                        dv = a.dr_val + di * (P + 1);
                    }
                }
#pragma unroll 1
                for (int j = 0; j <= P; ++j) {
                    const size_t mi = (size_t)wl * (P + 1) + j;
                    const double v = (j == P) ? chi_c : st[j];
                    const double dl = v - a.shift[mi];
                    if (dense) {
                        const size_t ci = ((size_t)row * a.n_walkers + wl) * (P + 1) + j;
                        if (a.chain_f32) static_cast<float*>(a.chain)[ci] = (float)dl; else static_cast<double*>(a.chain)[ci] = v;
                    }
                    if (dv) dv[j] = v;
                    atomicAdd(&a.moments[2 * mi], dl);                    // single writer: plain RED, in order
                    atomicAdd(&a.moments[2 * mi + 1], dl * dl);
                }
                if (a.sk_hist) {
                    double xy[2 * NB];
#pragma unroll
                    for (int j = 0; j < 2 * NB; ++j) xy[j] = st[j];
                    record_sketch<NB>(a, wl, (two && slot) ? frame1 : frame0, xy);
                }
                if (a.bm) {
                    const int n_lev = bm_closing(a, row);
                    if (n_lev) {
                        const int nq = bm_quantities<NB>(a);
#pragma unroll 1
                        for (int c = 0; c < nq; ++c) bm_close<NB>(a, wl, c, n_lev);
                    }
                }
                if (a.probe) {                                            // lapf_sampler_selftest
                    double* pb = a.probe + ((size_t)row * a.n_walkers + wl) * 3;
                    pb[0] = (a.prior && skip) ? (double)(-1 - k) : (double)k; pb[1] = nv; pb[2] = chi_t;
                }
            }
            ++row;
            next_rec += a.thin;   // (saturates harmlessly: a launch is shorter than 2^30)
        }
    }
    if (mine) {
        st[P] = chi_c;
        a.exps[wl] += n_exps;
    }
}

template <int NB, int NX, int NY, int NW, int LW>
__global__ void __launch_bounds__(NW * 32, 1) gibbs_batch_kernel(const __grid_constant__ RunArgs a) {
    using I = CoefImg<NB, Geo<NX>::PANELS>;
    constexpr int WPP = NX == 32 ? 2 : 1;           // walkers per pass: a half warp each on 32-pixel stamps
    constexpr int TAB = Scratch<NB, NX, NY, 1, WPP>::FLOATS;
    // stamps of up to 64 x 64 pixels also live in the TMEM pixel store (see tmem_fill_stamp)
    // (128 x 128: the weight plane only, the data plane is read from shared memory)
    constexpr int TM = (Geo<NX>::PANELS == 1 && Rows<NY, 1>::HALVES == 1) ? 1 : 2;
    // TM == 1: the pixel store has TWO slots, so that an item can hold walkers of two frames (the shared-memory
    // planes are then only where a stamp is staged and converted; both loops read the pixel store)
    constexpr uint32_t SLOT_COLS = TM == 1 ? 16 * (NY / Geo<NX, WPP>::RG) : 512;
    constexpr int SLOTS = TM == 1 ? 2 : 1;
    constexpr uint32_t TM_COLS = SLOTS * SLOT_COLS;
    static_assert(TM_COLS >= 32 && TM_COLS <= 512 && (TM_COLS & (TM_COLS - 1)) == 0, "TMEM allocations are powers of two");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_slot;
    float* sd = reinterpret_cast<float*>(smem_raw);
    float* sw = sd + NX * NY;
    float* rt = sw + NX * NY;                       // [NW] row + column tables (Scratch)
    float* img = rt + NW * TAB;                     // [NW][LW][CoefImg::STRIDE] trial coefficients
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) mbar_init(&bar, 1);
    if (TM && warp == 0) tmem_alloc(&tmem_slot, TM_COLS);
    if (TM) tmem_fence_before_sync();
    __syncthreads();
    if (TM) tmem_fence_after_sync();
    const uint32_t tmem_base = TM ? tmem_slot : 0u;

    if (a.cta_times && threadIdx.x == 0) {
        unsigned long long t;
        unsigned sm;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        asm volatile("mov.u32 %0, %%smid;" : "=r"(sm));
        a.cta_times[3 * blockIdx.x] = t;
        a.cta_times[3 * blockIdx.x + 2] = sm;
    }
    const int i0 = a.cta_item[blockIdx.x], i1 = a.cta_item[blockIdx.x + 1];
    int cur_frame[2] = {-1, -1};
    uint32_t phase = 0;
    for (int it = i0; it < i1; ++it) {
        const int fr[2] = {a.item_frame[it], a.item_frame2[it]};
#pragma unroll
        for (int sl = 0; sl < SLOTS; ++sl) {
            const int f = fr[sl];
            if (f < 0 || f == cur_frame[sl]) continue;          // (uniform over the CTA)
            __syncthreads();   // every warp has finished with the previous stamp (and with the staging planes)
            if (threadIdx.x == 0) {
                constexpr uint32_t kBytes = NX * NY * sizeof(float);
                fence_proxy_async();
                mbar_expect_tx(&bar, 2 * kBytes);
                tma_bulk_g2s(sd, a.data + (size_t)f * NX * NY, kBytes, &bar);
                tma_bulk_g2s(sw, a.weight + (size_t)f * NX * NY, kBytes, &bar);
            }
            mbar_wait(&bar, phase);
            phase ^= 1u;
            cur_frame[sl] = f;
            prep_stamp(sd, sw, NX * NY);            // (d, w) -> (d*sqrt(w), -sqrt(w)), once per staged frame
            __syncthreads();
            {
                if constexpr (TM == 1) { if (warp < 4) tmem_fill_stamp<NX, NY, WPP>(tmem_base + (uint32_t)sl * SLOT_COLS, sd, sw, warp, lane); }
                else { if (warp < 4) tmem_fill_weights<NX, NY>(tmem_base, sw, warp, lane); }
                tmem_fence_before_sync();
                __syncthreads();
                tmem_fence_after_sync();
            }
        }
        // walker j of the item goes to warp j % NW, lane j / NW: the warps' loads differ by at most one.  The first
        // na walkers are of the frame in slot sa, the others of the frame in the other slot.
        const int n = a.item_count[it], na = a.item_count_a[it], sa = a.item_slot_a[it];
        const int nl = n > warp ? (n - warp + NW - 1) / NW : 0;
        const int la = na > warp ? min((na - warp + NW - 1) / NW, nl) : 0;
        const int j = warp + NW * lane;
        const int slot = (lane < la) ? sa : 1 - sa;
        if (nl > 0)
            run_batch<NB, NX, NY, LW, TM, WPP>(a, sd, sw, rt + warp * TAB, img + warp * (LW * I::STRIDE),
                                          (lane < nl) ? a.walker_of[a.item_first[it] + j] : -1, nl, la,
                                          fr[0], SLOTS > 1 ? fr[1] : -1, slot, lane,
                                          tmem_base + ((uint32_t)(32 * (warp & 3)) << 16), SLOT_COLS);
    }
    if (TM) {
        tmem_fence_before_sync();
        __syncthreads();
        if (warp == 0) tmem_dealloc(tmem_base, TM_COLS);
    }
    if (a.cta_times && threadIdx.x == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        a.cta_times[3 * blockIdx.x + 1] = t;
    }
}

// lapf_sampler_selftest: trial vector of update u = state before it (start, or the row recorded by
// update u-1) with the proposed value in place; and the comparison of the sampler's trial
// chi-squares with the stateless operator's, bit for bit.
__global__ void selftest_trials_kernel(const double* __restrict__ start, const double* __restrict__ chain,
                                       const double* __restrict__ probe, int U, int64_t W, int P,
                                       double* __restrict__ trials /*[U][W][P]*/) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)U * W) return;
    const int64_t u = i / W, w = i % W;
    const double* before = u ? chain + ((u - 1) * W + w) * (P + 1) : start + w * (P + 1);
    int k = (int)probe[i * 3];
    if (k < 0) k = -1 - k;                                         // a proposal outside its prior box
    for (int j = 0; j < P; ++j) trials[i * P + j] = (j == k) ? probe[i * 3 + 1] : before[j];
}

// With priors a probe row marked as outside its box (no pass, no trial chi-square) must hold a proposal that lies
// outside the box of its frame (`frame_of` [U][W]) and every other row one inside it, so a wrong skip fails too.
__global__ void selftest_compare_kernel(const double* __restrict__ probe, const double* __restrict__ chi_k1, int64_t n,
                                        const double* __restrict__ prior, const int32_t* __restrict__ frame_of, int P,
                                        unsigned long long* __restrict__ out /*[2]: mismatches, first index + 1*/) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double a = probe[i * 3 + 2], b = chi_k1[i], kd = probe[i * 3];
    const int k = kd < 0.0 ? (int)(-1.0 - kd) : (int)kd;
    const bool outside = prior && prior_outside(prior + ((size_t)frame_of[i] * P + k) * 4, probe[i * 3 + 1]);
    const bool same = kd < 0.0 ? outside : ((a == b) || (isnan(a) && isnan(b))) && !outside;
    if (!same) {
        atomicAdd(out, 1ull);
        atomicMin(out + 1, (unsigned long long)i + 1ull);
    }
}

// state[w] = (init params, chi2); shift = state; counters and moments zeroed
__global__ void pack_state_kernel(const double* __restrict__ init, const double* __restrict__ chi, int P,
                                  int64_t W, double* __restrict__ state, double* __restrict__ shift) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W * (P + 1)) return;
    const int64_t w = i / (P + 1);
    const int j = (int)(i % (P + 1));
    const double v = (j < P) ? init[w * P + j] : chi[w];
    state[i] = v;
    shift[i] = v;
}

// Priors: per walker w (of frame frame_of[w]), the parameters params[w * stride + j] outside the frame's box;
// out[0] += that count, out[1] = min(out[1], w * P + j + 1) over them
__global__ void prior_outside_kernel(const double* __restrict__ params, int stride, const int32_t* __restrict__ frame_of,
                                     const double* __restrict__ prior, int P, int64_t W, unsigned long long* __restrict__ out) {
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= W) return;
    const double* pr = prior + (size_t)frame_of[w] * P * 4;
    unsigned n = 0;
    int first = -1;
    for (int j = 0; j < P; ++j)
        if (prior_outside(pr + 4 * j, params[w * stride + j])) {
            if (!n) first = j;
            ++n;
        }
    if (n) {
        atomicAdd(out, (unsigned long long)n);
        atomicMin(out + 1, (unsigned long long)(w * P + first) + 1ull);
    }
}

// =============================================================================================
// K4: batch statistics
// =============================================================================================
__global__ void totals_kernel(const uint32_t* __restrict__ tries, const uint32_t* __restrict__ accepts,
                              const unsigned long long* __restrict__ exps, int P, int64_t W,
                              unsigned long long* __restrict__ out /*[2P+2]*/) {
    // integer sums and a min: order-independent, so atomics are deterministic here
    const int j = blockIdx.y;
    unsigned long long st = 0, sa = 0, mn = ~0ull, se = 0;
    for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < W; w += (int64_t)gridDim.x * blockDim.x) {
        const unsigned long long t = tries[w * P + j];
        st += t;
        sa += accepts[w * P + j];
        mn = min(mn, t);
        if (j == 0) se += exps[w];
    }
    for (int off = 16; off >= 1; off >>= 1) {
        st += __shfl_xor_sync(kFull, st, off);
        sa += __shfl_xor_sync(kFull, sa, off);
        mn = min(mn, __shfl_xor_sync(kFull, mn, off));
        se += __shfl_xor_sync(kFull, se, off);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(out + j, st);
        atomicAdd(out + P + j, sa);
        atomicMin(out + 2 * P, mn);
        if (j == 0) atomicAdd(out + 2 * P + 1, se);
    }
}

__global__ void totals_init_kernel(unsigned long long* out, int P) {
    const int i = threadIdx.x;
    if (i < 2 * P || i == 2 * P + 1) out[i] = 0ull;
    if (i == 2 * P) out[i] = ~0ull;
}

// One CTA per frame, one warp per column: fixed-order FP64 reduction over that frame's walkers.
// Chain means are taken relative to a per-frame reference value (the first walker's starting
// point) so that the between-chain sum of squares does not cancel for parameters with a large
// mean and a tiny spread (positions: ~512 +- 0.003).
__global__ void moments_kernel(const double* __restrict__ moments, const double* __restrict__ shift,
                               const int32_t* __restrict__ walker_of, const int32_t* __restrict__ frame_start,
                               int P, int64_t n_rows, double* __restrict__ out /*[F][P+1][4]*/) {
    const int f = blockIdx.x, col = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (col > P) return;
    const int b = frame_start[f], e = frame_start[f + 1];
    const double ref = (e > b) ? shift[(size_t)walker_of[b] * (P + 1) + col] : 0.0;
    double s_mean = 0.0, s_mean2 = 0.0, s_var = 0.0;
    if (n_rows > 0) {
        const double inv = 1.0 / (double)n_rows;
        for (int i = b + lane; i < e; i += 32) {
            const size_t w = (size_t)walker_of[i];
            const double m1 = moments[(w * (P + 1) + col) * 2] * inv;
            const double m2 = moments[(w * (P + 1) + col) * 2 + 1] * inv;
            const double mean = (shift[w * (P + 1) + col] - ref) + m1;
            s_mean += mean;
            s_mean2 += mean * mean;
            s_var += m2 - m1 * m1;     // population variance, np.std()**2 of apf_step3.py:270
        }
    }
    s_mean = warp_sum_f64(s_mean);
    s_mean2 = warp_sum_f64(s_mean2);
    s_var = warp_sum_f64(s_var);
    if (lane == 0) {
        double* o = out + ((size_t)f * (P + 1) + col) * 4;
        o[0] = ref;
        o[1] = s_mean;
        o[2] = s_mean2;
        o[3] = s_var;
    }
}

__global__ void counts_kernel(const int32_t* __restrict__ frame_start, int F, int64_t n_rows,
                              long long* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < F) out[i] = frame_start[i + 1] - frame_start[i];
    if (i == F) out[F] = n_rows;
}

// The sampler's random stream, exposed so tests can pin it against the oracle's restatement.
__global__ void philox_draws_kernel(uint64_t seed, uint64_t walker, uint64_t t0, int n, int nparam,
                                    int32_t* __restrict__ k_out, double* __restrict__ z_out,
                                    double* __restrict__ lnu_out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Draw d = make_draw(seed, walker, t0 + (uint64_t)i, nparam);
    k_out[i] = d.k;
    z_out[i] = d.z;
    lnu_out[i] = d.lnu;
}

// =============================================================================================
// frame preparation (apf_step2.py:176-210) + cut-out
// =============================================================================================
__global__ void frame_prep_kernel(const float* __restrict__ frames, int F, int fy, int fx,
                                  const int32_t* __restrict__ origin, int ny, int nx, double satcut,
                                  double rn2, float* __restrict__ data_out, float* __restrict__ weight_out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t n = (int64_t)F * ny * nx;
    if (i >= n) return;
    const int f = (int)(i / ((int64_t)ny * nx));
    const int r = (int)((i / nx) % ny), c = (int)(i % nx);
    const int y = origin[2 * f + 1] + r, x = origin[2 * f] + c;
    float d = 0.f, w = 0.f;
    if (y >= 0 && y < fy && x >= 0 && x < fx) {
        const float v = frames[((size_t)f * fy + y) * fx + x];
        // masked (apf_step2.py:188: image > 0.8*satlevel) or non-finite pixels get zero weight
        if (isfinite(v) && !((double)v > satcut)) {
            d = v;
            w = (float)(1.0 / (rn2 + fabs((double)v)));   // 1/err^2, err^2 = readnoise^2 + |image| (:207-210)
        }
    }
    data_out[i] = d;
    weight_out[i] = w;
}

// Centre values of the sketches when the caller gives none: separation / position angle of the
// starting point of the frame's first walker.
__global__ void sketch_center_kernel(const double* __restrict__ shift, const int32_t* __restrict__ walker_of,
                                     const int32_t* __restrict__ frame_start, int F, int P, int nbody,
                                     double* __restrict__ center /*[F][nbody-1][2]*/) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= F * (nbody - 1)) return;
    const int f = i / (nbody - 1), o = 1 + i % (nbody - 1);
    double sep = 0.0, pa = 0.0;
    if (frame_start[f + 1] > frame_start[f]) {
        const double* x = shift + (size_t)walker_of[frame_start[f]] * (P + 1);
        const double dx = x[2 * o] - x[0], dy = x[2 * o + 1] - x[1];
        sep = sqrt(dx * dx + dy * dy);
        pa = atan2(-dx, dy) * 57.29577951308232;
    }
    center[2 * i] = sep;
    center[2 * i + 1] = pa;
}

// Per frame and sketch slot: centre, sum and sum of squares of (value - centre) over the frame's
// walkers (fixed order) and the number of values -- mean and standard deviation without the chain.
__global__ void sketch_reduce_kernel(const double* __restrict__ sk_mom, const double* __restrict__ center,
                                     const int32_t* __restrict__ walker_of, const int32_t* __restrict__ frame_start,
                                     int slots /*(nbody-1)*2*/, int64_t n_rows, double* __restrict__ out /*[F][slots][4]*/) {
    const int f = blockIdx.x, q = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (q >= slots) return;
    const int b = frame_start[f], e = frame_start[f + 1];
    double s1 = 0.0, s2 = 0.0;
    for (int i = b + lane; i < e; i += 32) {
        const double* m = sk_mom + ((size_t)walker_of[i] * slots + q) * 2;
        s1 += m[0];
        s2 += m[1];
    }
    s1 = warp_sum_f64(s1);
    s2 = warp_sum_f64(s2);
    if (lane == 0) {
        double* o = out + ((size_t)f * slots + q) * 4;
        o[0] = center[(size_t)f * slots + q];
        o[1] = s1;
        o[2] = s2;
        o[3] = (double)(e - b) * (double)n_rows;
    }
}

// Batch means per frame, one CTA per frame; warp i takes the items i, i + warps, ... of [C][1 + L] and
// reduces over the frame's walkers in the fixed order of moments_kernel.  Item (c, 0): sum of the
// walkers' population variance of quantity c over their recorded rows (np.std()**2, apf_step3.py:270),
// from the running moments (columns) or the sketch sums (separation / position angle).  Item (c, 1 + l):
// sum of the sample variances of the walkers' level-l batch means, each from its (snap, s2) and J
// complete batches of b = b0 * 2^l rows: (s2 - snap^2 / J) / (b^2 (J - 1)); 0 where J < 2.
__global__ void batchmeans_reduce_kernel(const double* __restrict__ bm, const double* __restrict__ moments,
                                         const double* __restrict__ sk_mom, const int32_t* __restrict__ walker_of,
                                         const int32_t* __restrict__ frame_start, int P, int C, int L, int b0,
                                         int64_t n_rows, double* __restrict__ out /*[F][C][1 + L]*/) {
    const int f = blockIdx.x, lane = threadIdx.x & 31, warps = blockDim.x >> 5;
    const int b = frame_start[f], e = frame_start[f + 1], slots = C - (P + 1);
    for (int it = threadIdx.x >> 5; it < C * (1 + L); it += warps) {
        const int c = it / (1 + L), j = it % (1 + L);
        double s = 0.0;
        if (j == 0 && n_rows > 0) {
            const double inv = 1.0 / (double)n_rows;
            for (int i = b + lane; i < e; i += 32) {
                const size_t w = (size_t)walker_of[i];
                const double* m = (c <= P) ? moments + (w * (P + 1) + c) * 2 : sk_mom + (w * slots + (c - P - 1)) * 2;
                const double m1 = m[0] * inv, m2 = m[1] * inv;
                s += m2 - m1 * m1;
            }
        } else if (j > 0) {
            const int64_t bl = (int64_t)b0 << (j - 1), J = n_rows / bl;
            if (J >= 2) {
                const double inv_j = 1.0 / (double)J, scale = 1.0 / ((double)bl * (double)bl * (double)(J - 1));
                for (int i = b + lane; i < e; i += 32) {
                    const double* q = bm + (((size_t)walker_of[i] * C + c) * L + (j - 1)) * 2;
                    s += (q[1] - q[0] * q[0] * inv_j) * scale;
                }
            }
        }
        s = warp_sum_f64(s);
        if (lane == 0) out[((size_t)f * C + c) * (1 + L) + j] = s;
    }
}

// Per-frame acceptance: one CTA per frame, one warp per parameter, over the frame's walkers in the
// order of moments_kernel.  Integer sums: exact in any order, and ranks may add them.
__global__ void frame_counts_kernel(const uint32_t* __restrict__ tries, const uint32_t* __restrict__ accepts,
                                    const int32_t* __restrict__ walker_of, const int32_t* __restrict__ frame_start,
                                    int P, long long* __restrict__ out /*[F][P][2]*/) {
    const int f = blockIdx.x, j = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (j >= P) return;
    unsigned long long st = 0, sa = 0;
    for (int i = frame_start[f] + lane; i < frame_start[f + 1]; i += 32) {
        const size_t w = (size_t)walker_of[i];
        st += tries[w * P + j];
        sa += accepts[w * P + j];
    }
    for (int off = 16; off >= 1; off >>= 1) {
        st += __shfl_xor_sync(kFull, st, off);
        sa += __shfl_xor_sync(kFull, sa, off);
    }
    if (lane == 0) {
        out[((size_t)f * P + j) * 2] = (long long)st;
        out[((size_t)f * P + j) * 2 + 1] = (long long)sa;
    }
}

// Per-frame width update from the window since the last one (lapf_sampler_adapt_widths): dt = T - T_prev,
// da = A - A_prev; if dt > 0, w *= min(max(exp(da / dt - target), 0.5), 2); the snapshot becomes the counts.
// Every operation rounded to nearest and never contracted (DESIGN.md 5): the tests restate it in numpy.
__global__ void adapt_widths_kernel(const long long* __restrict__ counts, long long* __restrict__ snap,
                                    double* __restrict__ fw, int n /*F * P*/, double target) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long t = counts[2 * i], ac = counts[2 * i + 1];
    const long long dt = t - snap[2 * i], da = ac - snap[2 * i + 1];
    if (dt > 0) {
        const double e = exp(__dsub_rn(__ddiv_rn((double)da, (double)dt), target));
        fw[i] = __dmul_rn(fw[i], fmin(fmax(e, 0.5), 2.0));
    }
    snap[2 * i] = t;
    snap[2 * i + 1] = ac;
}

// The same cut-out + mask + noise map with the pixels fetched by the TMA unit: a 3-D tensor map over
// the frames [F][fy][fx] and one box of kPrepRows x (nx + 4) pixels per CTA (cp.async.bulk.tensor,
// SASS UTMALDG) -- rows of a cut-out are nx * 4 bytes long and fx * 4 bytes apart, which is exactly
// the strided pattern a tensor map describes.  The unit wants the first byte of a box 16-byte
// aligned (a box starting at column 10 of a float frame raises "illegal instruction", measured with
// tools/tma_probe.cu), so the box starts at the multiple of 4 columns at or below the cut-out and is 4
// columns wider.  Pixels outside the frame come back as zeros from the unit and are given zero
// weight here from their coordinates, as in frame_prep_kernel.
constexpr int kPrepRows = 32;

__global__ void __launch_bounds__(256)
frame_prep_tma_kernel(const __grid_constant__ CUtensorMap tmap, int fy, int fx, const int32_t* __restrict__ origin,
                      int ny, int nx, double satcut, double rn2, float* __restrict__ data_out,
                      float* __restrict__ weight_out) {
    extern __shared__ __align__(128) unsigned char prep_smem[];
    __shared__ uint64_t bar;
    float* tile = reinterpret_cast<float*>(prep_smem);
    const int f = blockIdx.y, r0 = blockIdx.x * kPrepRows;
    const int x0 = origin[2 * f], y0 = origin[2 * f + 1];
    const int xa = x0 & ~3;                       // floor to a multiple of 4, also for negative x0
    const int bw = nx + 4, shift = x0 - xa;
    if (threadIdx.x == 0) mbar_init(&bar, 1);
    __syncthreads();
    if (threadIdx.x == 0) {
        fence_proxy_async();
        mbar_expect_tx(&bar, (uint32_t)(kPrepRows * bw * sizeof(float)));
        asm volatile(
            "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
            ::"r"(smem_u32(tile)), "l"(reinterpret_cast<uint64_t>(&tmap)), "r"(xa), "r"(y0 + r0), "r"(f), "r"(smem_u32(&bar))
            : "memory");
    }
    mbar_wait(&bar, 0);
    const int rows = min(kPrepRows, ny - r0);
    for (int i = threadIdx.x; i < rows * nx; i += blockDim.x) {
        const int r = i / nx, c = i % nx;
        const int y = y0 + r0 + r, x = x0 + c;
        float d = 0.f, w = 0.f;
        if (y >= 0 && y < fy && x >= 0 && x < fx) {
            const float v = tile[r * bw + shift + c];
            if (isfinite(v) && !((double)v > satcut)) {
                d = v;
                w = (float)(1.0 / (rn2 + fabs((double)v)));
            }
        }
        const size_t o = ((size_t)f * ny + r0 + r) * nx + c;
        data_out[o] = d;
        weight_out[o] = w;
    }
}

// sum w, sum w d, sum w d^2 over the pixels of each frame OUTSIDE its cut-out, with the weight map
// of frame_prep_kernel (lapf_problem.outside): per (frame, row tile) partials in FP64, fixed order.
__global__ void __launch_bounds__(256)
outside_partial_kernel(const float* __restrict__ frames, int fy, int fx, const int32_t* __restrict__ cut, int ny, int nx,
                       double satcut, double rn2, int rows_per_tile, double* __restrict__ partial /*[F][tiles][3]*/) {
    const int f = blockIdx.y, tile = blockIdx.x;
    const int cx = cut[2 * f], cy = cut[2 * f + 1];
    const int r0 = tile * rows_per_tile, r1 = min(fy, r0 + rows_per_tile);
    double s0 = 0.0, s1 = 0.0, s2 = 0.0;
    for (int r = r0; r < r1; ++r) {
        const bool row_in = r >= cy && r < cy + ny;
        const float* src = frames + ((size_t)f * fy + r) * fx;
        for (int c = threadIdx.x; c < fx; c += blockDim.x) {
            if (row_in && c >= cx && c < cx + nx) continue;
            const float v = src[c];
            if (isfinite(v) && !((double)v > satcut)) {
                const double w = (double)(float)(1.0 / (rn2 + fabs((double)v)));
                const double d = (double)v;
                s0 += w;
                s1 += w * d;
                s2 += w * d * d;
            }
        }
    }
    __shared__ double red[8][3];
    s0 = warp_sum_f64(s0); s1 = warp_sum_f64(s1); s2 = warp_sum_f64(s2);
    if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5][0] = s0; red[threadIdx.x >> 5][1] = s1; red[threadIdx.x >> 5][2] = s2; }
    __syncthreads();
    if (threadIdx.x < 3) {
        double t = 0.0;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += red[i][threadIdx.x];
        partial[((size_t)f * gridDim.x + tile) * 3 + threadIdx.x] = t;
    }
}

__global__ void outside_reduce_kernel(const double* __restrict__ partial, int F, int tiles, double* __restrict__ out /*[F][3]*/) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 3 * F) return;
    const int f = i / 3, q = i % 3;
    double t = 0.0;
    for (int k = 0; k < tiles; ++k) t += partial[((size_t)f * tiles + k) * 3 + q];
    out[i] = t;
}

// =============================================================================================
// roofline micro-benchmarks
// =============================================================================================
__global__ void __launch_bounds__(256) peak_ex2_kernel(float* out, int iters) {
    float x[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) x[j] = 0.1f * (float)(threadIdx.x & 7) + 0.05f * j;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int rep = 0; rep < 8; ++rep) {
#pragma unroll
            for (int j = 0; j < 8; ++j) x[j] = ex2_approx(-x[j]);
        }
    }
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) s += x[j];
    if (s == 123.456f) out[0] = s;
}

__global__ void __launch_bounds__(256) peak_ffma_kernel(float* out, int iters, float a, float b) {
    float x[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) x[j] = 0.1f * (float)(threadIdx.x & 7) + 0.05f * j;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int rep = 0; rep < 8; ++rep) {
#pragma unroll
            for (int j = 0; j < 8; ++j) x[j] = fmaf(x[j], a, b);
        }
    }
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) s += x[j];
    if (s == 123.456f) out[0] = s;
}

// =============================================================================================
// host side
// =============================================================================================
struct lapf_sampler {
    lapf_config cfg;
    int P = 0;
    int device = 0;
    int nw = 0, minb = 0, grid = 0, team = 1;
    size_t smem = 0;
    int64_t count = 0;      // updates done so far
    int64_t launches = 0;
    int n_items = 0;
    double widths[LAPF_MAX_PARAMS];
    uint32_t log_mask = 0;
    // device buffers owned by the handle
    double* state = nullptr;
    double* shift = nullptr;
    double* moments = nullptr;
    uint32_t* tries = nullptr;
    uint32_t* accepts = nullptr;
    unsigned long long* exps = nullptr;
    int32_t* walker_of = nullptr;
    int32_t* frame_start = nullptr;
    int32_t* item_frame = nullptr;
    int32_t* item_first = nullptr;
    int32_t* item_count = nullptr;
    int32_t* item_frame2 = nullptr;   // batched kernel: second resident frame of an item (see RunArgs)
    int32_t* item_count_a = nullptr;
    int32_t* item_slot_a = nullptr;
    int32_t* cta_item = nullptr;   // batched kernel: first item of every CTA
    int32_t* frame_of = nullptr;   // [W] the caller's frame index per walker (a copy: reset and the self-test need it)
    // chain rows leave as double values or as float differences from the starting point
    int chain_format = LAPF_CHAIN_F64;
    // separation / position-angle sketches (lapf_sampler_sketch_enable)
    int sk_bins = 0;
    bool sk_auto_center = true;
    double sk_sep_bin = 0.0, sk_pa_bin = 0.0;
    uint32_t* sk_hist = nullptr;
    double* sk_center = nullptr;
    double* sk_mom = nullptr;
    // batch means (lapf_sampler_batchmeans_enable): [W][bm_c][bm_levels][2]
    double* bm = nullptr;
    int bm_rows = 0, bm_levels = 0, bm_c = 0;
    // posterior draws (lapf_sampler_draws_enable): [W][dr_k][P+1] values, [W][dr_k] row indices
    double* dr_val = nullptr;
    int64_t* dr_row = nullptr;
    int dr_k = 0;
    // per-frame jump widths (lapf_sampler_set_frame_widths): [F][P], and the counts of the last
    // adaptation [F][P][2] (tries, accepts summed over the frame's walkers and over ranks)
    double* fw = nullptr;
    long long* fw_snap = nullptr;
    // parameter priors (lapf_sampler_set_priors): [F][P][4] {lo, hi, mu, h} for the kernels, and the table as
    // given, {lo, hi, mu, sigma}
    double* pr = nullptr;
    double* pr_given = nullptr;
    int chunk = 0;                 // batched kernel: walkers per item at most (warps x walkers per warp)
    int launch_grid = 0;           // batched kernel: CTAs that have work
};

// Far-field culling (set_cull) is on unless the caller sets bit 0 of lapf_problem.flags or the
// environment variable LAPF_NO_CULL is set; 32-pixel stamps have no far field worth the test.
static int cull_enabled(const lapf_problem* p) {
    if (p->flags & LAPF_FLAG_NO_CULL) return 0;
    if (getenv("LAPF_NO_CULL")) return 0;
    return p->nx >= 64 ? 1 : 0;
}

static int plain_loop(const lapf_problem* p) {
    return ((p->flags & LAPF_FLAG_PLAIN_LOOP) || getenv("LAPF_PLAIN_LOOP")) ? 1 : 0;
}

static bool stamp_supported(int ny, int nx) { return ny == nx && (nx == 32 || nx == 64 || nx == 128); }

static int check_problem(const lapf_problem* p) {
    if (!p) return fail(LAPF_ERR_INVALID, "problem is NULL");
    if (p->nbody != 2 && p->nbody != 3) return fail(LAPF_ERR_INVALID, "nbody must be 2 or 3, got %d", p->nbody);
    if (p->ny <= 0 || p->nx <= 0 || p->n_frames <= 0)
        return fail(LAPF_ERR_INVALID, "bad shape ny=%d nx=%d n_frames=%d", p->ny, p->nx, p->n_frames);
    const int P = 3 * p->nbody + 10;
    if (p->floor_index < 2 * p->nbody || p->floor_index >= P)
        return fail(LAPF_ERR_INVALID, "floor_index %d outside [%d,%d) (positions cannot be the floor)",
                    p->floor_index, 2 * p->nbody, P);
    if (!p->data || !p->weight || !p->origin) return fail(LAPF_ERR_INVALID, "data/weight/origin must be device pointers");
    if (((uintptr_t)p->data & 15) || ((uintptr_t)p->weight & 15))
        return fail(LAPF_ERR_INVALID, "data and weight must be 16-byte aligned (TMA bulk copies)");
    return LAPF_OK;
}

static int64_t rows_upto(int64_t count, int64_t burn_in, int thin) {
    // rows recorded by updates with count' in [1, count]: count' >= burn_in and
    // (count' - burn_in) % thin == 0 (apf_step2.py:333,342-351; thin = 1 there)
    if (count < burn_in || count < 1) return 0;
    int64_t n = (count - burn_in) / thin + 1;
    if (burn_in <= 0) n -= 1;   // count' = burn_in = 0 is not an update
    return n;
}

static int64_t next_record_after(int64_t count, int64_t burn_in, int thin) {
    // smallest count' > count with count' >= burn_in, count' >= 1, (count' - burn_in) % thin == 0
    int64_t c = std::max<int64_t>(count + 1, std::max<int64_t>(burn_in, 1));
    const int64_t rem = (c - burn_in) % thin;
    if (rem) c += thin - rem;
    return c;
}

template <int NB, int NX, bool STORE>
static void launch_stamp_k1(const ProbPtrs& pr, const double* params, int64_t B, const int32_t* frame_of,
                            float* model_out, double* chi2_out, cudaStream_t st) {
    if constexpr (NX == 32) {
        const unsigned grid = (unsigned)((B + 7) / 8);          // two vectors per warp, four warps per CTA
        model_chi2_pair_kernel<NB, NX, NX, STORE><<<grid, 128, 0, st>>>(pr, params, B, frame_of, model_out, chi2_out);
    } else {
        const unsigned grid = (unsigned)((B + 3) / 4);
        model_chi2_stamp_kernel<NB, NX, NX, STORE><<<grid, 128, 0, st>>>(pr, params, B, frame_of, model_out, chi2_out);
    }
}

template <int NB, int NX>
static void launch_stamp_k1_store(bool store, const ProbPtrs& pr, const double* params, int64_t B,
                                  const int32_t* frame_of, float* model_out, double* chi2_out, cudaStream_t st) {
    if (store)
        launch_stamp_k1<NB, NX, true>(pr, params, B, frame_of, model_out, chi2_out, st);
    else
        launch_stamp_k1<NB, NX, false>(pr, params, B, frame_of, model_out, chi2_out, st);
}

template <int NB>
static void launch_stamp_k1_size(int nx, bool store, const ProbPtrs& pr, const double* params, int64_t B,
                                 const int32_t* frame_of, float* model_out, double* chi2_out, cudaStream_t st) {
    if (nx == 32) launch_stamp_k1_store<NB, 32>(store, pr, params, B, frame_of, model_out, chi2_out, st);
    else if (nx == 64) launch_stamp_k1_store<NB, 64>(store, pr, params, B, frame_of, model_out, chi2_out, st);
    else launch_stamp_k1_store<NB, 128>(store, pr, params, B, frame_of, model_out, chi2_out, st);
}

extern "C" {

int lapf_abi_version(void) { return LAPF_ABI_VERSION; }
const char* lapf_last_error(void) { return g_err; }

int lapf_num_params(int nbody) {
    if (nbody != 2 && nbody != 3) return fail(LAPF_ERR_INVALID, "nbody must be 2 or 3, got %d", nbody);
    return 3 * nbody + 10;
}

int lapf_default_widths(int nbody, double* widths_out, int32_t* is_log_out) {
    const int P = lapf_num_params(nbody);
    if (P < 0) return P;
    const double* w = nbody == 2 ? kWidths2 : kWidths3;
    const uint32_t m = log_mask_for(nbody);
    for (int i = 0; i < P; ++i) {
        if (widths_out) widths_out[i] = w[i];
        if (is_log_out) is_log_out[i] = (m >> i) & 1u;
    }
    return LAPF_OK;
}

int lapf_model_chi2(const lapf_problem* prob, const double* params, int64_t B, const int32_t* frame_of,
                    float* model_out, double* chi2_out, void* stream) {
    int rc = check_problem(prob);
    if (rc) return rc;
    if (B < 0 || (B > 0 && !params)) return fail(LAPF_ERR_INVALID, "params is NULL or B < 0");
    if (B == 0) return LAPF_OK;
    if ((rc = require_device())) return rc;
    keep_pool_memory();
    cudaStream_t st = (cudaStream_t)stream;
    ProbPtrs pr{prob->data, prob->weight, prob->origin, prob->outside, prob->n_frames, prob->floor_index,
                cull_enabled(prob), plain_loop(prob)};
    if (stamp_supported(prob->ny, prob->nx) && (!model_out || ((uintptr_t)model_out & 15) == 0)) {
        if (prob->nbody == 2)
            launch_stamp_k1_size<2>(prob->nx, model_out != nullptr, pr, params, B, frame_of, model_out, chi2_out, st);
        else
            launch_stamp_k1_size<3>(prob->nx, model_out != nullptr, pr, params, B, frame_of, model_out, chi2_out, st);
        CU(cudaGetLastError());
        return LAPF_OK;
    }
    // generic domain (e.g. the whole frame)
    if (B > 65535) return fail(LAPF_ERR_INVALID, "generic-domain evaluation supports B <= 65535 per call, got %lld", (long long)B);
    const int rows_per_tile = 16;
    const int ntile = (prob->ny + rows_per_tile - 1) / rows_per_tile;
    double* partial = nullptr;
    if (chi2_out) CU(cudaMallocAsync((void**)&partial, sizeof(double) * (size_t)B * ntile, st));
    dim3 grid((unsigned)ntile, (unsigned)B);
    if (prob->nbody == 2)
        model_chi2_generic_kernel<2><<<grid, 256, 0, st>>>(pr, prob->ny, prob->nx, rows_per_tile, params, frame_of, model_out, partial);
    else
        model_chi2_generic_kernel<3><<<grid, 256, 0, st>>>(pr, prob->ny, prob->nx, rows_per_tile, params, frame_of, model_out, partial);
    CU(cudaGetLastError());
    if (chi2_out) {
        reduce_tiles_kernel<<<(unsigned)((B + 127) / 128), 128, 0, st>>>(partial, ntile, B, chi2_out);
        CU(cudaGetLastError());
        CU(cudaFreeAsync(partial, st));
    }
    return LAPF_OK;
}

// ---------------------------------------------------------------------------------------------
// sampler
// ---------------------------------------------------------------------------------------------
extern "C++" {
template <int NB, int NX, int NW, int MINB, int TEAM>
static int configure_gibbs(lapf_sampler* s) {
    auto kern = gibbs_kernel<NB, NX, NX, NW, MINB, TEAM>;
    s->nw = NW / TEAM;   // walkers per CTA item
    s->minb = MINB;
    constexpr size_t kBytes = 2 * sizeof(float) * NX * NX +
                              sizeof(float) * (TEAM > 1 ? (NW / TEAM) * Scratch<NB, NX, NX, TEAM>::TEAM_FLOATS
                                                        : NW * Scratch<NB, NX, NX, TEAM>::FLOATS);
    static_assert(kBytes + 16 * 1024 <= 227 * 1024, "team kernel: shared memory per CTA (dynamic + static scratch)");
    s->smem = kBytes;
    CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->smem));
    int per_sm = 0, sms = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, NW * 32, s->smem));
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, s->device));
    if (per_sm < 1) return fail(LAPF_ERR_CUDA, "gibbs kernel does not fit on an SM");
    s->grid = per_sm * sms;
    return LAPF_OK;
}

template <int NB, int NX, int NW, int MINB, int TEAM>
static int launch_gibbs(lapf_sampler* s, const RunArgs& a, cudaStream_t st) {
    const int grid = std::min(s->grid, a.n_items);
    gibbs_kernel<NB, NX, NX, NW, MINB, TEAM><<<grid, NW * 32, s->smem, st>>>(a);
    CU(cudaGetLastError());
    return LAPF_OK;
}

template <int NB, int NX, int NW, int LW>
static int configure_batch(lapf_sampler* s) {
    auto kern = gibbs_batch_kernel<NB, NX, NX, NW, LW>;
    s->nw = NW;
    s->chunk = NW * LW;
    s->minb = 1;
    constexpr size_t kBytes = sizeof(float) * (2 * NX * NX + NW * Scratch<NB, NX, NX, 1, (NX == 32 ? 2 : 1)>::FLOATS +
                                               NW * LW * CoefImg<NB, Geo<NX>::PANELS>::STRIDE);
    static_assert(kBytes + 256 <= 227 * 1024, "batched kernel: shared memory per CTA");
    s->smem = kBytes;
    CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->smem));
    int per_sm = 0, sms = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, NW * 32, s->smem));
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, s->device));
    if (per_sm < 1) return fail(LAPF_ERR_CUDA, "batched gibbs kernel does not fit on an SM");
    s->grid = sms;   // persistent: one CTA per SM
    return LAPF_OK;
}

template <int NB, int NX, int NW, int LW>
static int launch_batch(lapf_sampler* s, const RunArgs& a, cudaStream_t st) {
    gibbs_batch_kernel<NB, NX, NX, NW, LW><<<s->launch_grid, NW * 32, s->smem, st>>>(a);
    CU(cudaGetLastError());
    return LAPF_OK;
}

// walkers per warp (lanes used by the one-walker-per-lane phases): 32, fewer where the stamp or
// the 3-body tables leave less shared memory for the coefficient images
#define LAPF_DISPATCH_BATCH(FN, ...)                                                        \
    do {                                                                                    \
        const int nb__ = s->cfg.problem.nbody, nx__ = s->cfg.problem.nx;                    \
        if (nb__ == 2 && nx__ == 32) return FN<2, 32, 16, 32>(__VA_ARGS__);                 \
        if (nb__ == 2 && nx__ == 64) return FN<2, 64, 16, 32>(__VA_ARGS__);                 \
        if (nb__ == 2 && nx__ == 128) return FN<2, 128, 12, 16>(__VA_ARGS__);               \
        if (nb__ == 3 && nx__ == 32) return FN<3, 32, 16, 32>(__VA_ARGS__);                 \
        if (nb__ == 3 && nx__ == 64) return FN<3, 64, 16, 32>(__VA_ARGS__);                 \
        if (nb__ == 3 && nx__ == 128) return FN<3, 128, 12, 12>(__VA_ARGS__);               \
        return fail(LAPF_ERR_INVALID, "unsupported sampler shape nbody=%d nx=%d", nb__, nx__); \
    } while (0)

static int configure_batch_dispatch(lapf_sampler* s) { LAPF_DISPATCH_BATCH(configure_batch, s); }
static int launch_batch_dispatch(lapf_sampler* s, const RunArgs& a, cudaStream_t st) {
    LAPF_DISPATCH_BATCH(launch_batch, s, a, st);
}

#define LAPF_DISPATCH_TEAM(FN, NB_, NX_, NW_, ...)                                          \
    do {                                                                                    \
        if (s->team == 4) return FN<NB_, NX_, NW_, 1, 4>(__VA_ARGS__);                      \
        if (s->team == 16 && NX_ >= 64) return FN<NB_, NX_, 16, 1, (NX_ >= 64 ? 16 : 4)>(__VA_ARGS__); \
    } while (0)

#define LAPF_DISPATCH_GIBBS(FN, ...)                                                        \
    do {                                                                                    \
        const int nb__ = s->cfg.problem.nbody, nx__ = s->cfg.problem.nx;                    \
        if (nb__ == 2 && nx__ == 32) LAPF_DISPATCH_TEAM(FN, 2, 32, 16, __VA_ARGS__);        \
        if (nb__ == 2 && nx__ == 64) LAPF_DISPATCH_TEAM(FN, 2, 64, 16, __VA_ARGS__);        \
        if (nb__ == 2 && nx__ == 128) LAPF_DISPATCH_TEAM(FN, 2, 128, 16, __VA_ARGS__);      \
        if (nb__ == 3 && nx__ == 32) LAPF_DISPATCH_TEAM(FN, 3, 32, 16, __VA_ARGS__);        \
        if (nb__ == 3 && nx__ == 64) LAPF_DISPATCH_TEAM(FN, 3, 64, 16, __VA_ARGS__);        \
        if (nb__ == 3 && nx__ == 128) LAPF_DISPATCH_TEAM(FN, 3, 128, 12, __VA_ARGS__);      \
        return fail(LAPF_ERR_INVALID, "unsupported sampler shape nbody=%d nx=%d team_warps=%d", nb__, nx__, s->team); \
    } while (0)

static int configure_dispatch(lapf_sampler* s) {
    if (s->team == 1) return configure_batch_dispatch(s);
    LAPF_DISPATCH_GIBBS(configure_gibbs, s);
}
static int launch_dispatch(lapf_sampler* s, const RunArgs& a, cudaStream_t st) {
    if (s->team == 1) return launch_batch_dispatch(s, a, st);
    LAPF_DISPATCH_GIBBS(launch_gibbs, s, a, st);
}
}  // extern "C++"

static void free_sampler(lapf_sampler* s) {
    if (!s) return;
    cudaFree(s->state); cudaFree(s->shift); cudaFree(s->moments); cudaFree(s->tries); cudaFree(s->accepts); cudaFree(s->exps);
    cudaFree(s->walker_of); cudaFree(s->frame_start); cudaFree(s->item_frame); cudaFree(s->item_first);
    cudaFree(s->item_count); cudaFree(s->cta_item); cudaFree(s->frame_of);
    cudaFree(s->item_frame2); cudaFree(s->item_count_a); cudaFree(s->item_slot_a);
    cudaFree(s->sk_hist); cudaFree(s->sk_center); cudaFree(s->sk_mom);
    cudaFree(s->bm);
    cudaFree(s->dr_val); cudaFree(s->dr_row);
    cudaFree(s->fw); cudaFree(s->fw_snap);
    cudaFree(s->pr); cudaFree(s->pr_given);
    delete s;
}

int lapf_sampler_create(const lapf_config* cfg, lapf_sampler** out, void* stream) {
    if (!cfg || !out) return fail(LAPF_ERR_INVALID, "cfg/out is NULL");
    *out = nullptr;
    int rc = check_problem(&cfg->problem);
    if (rc) return rc;
    const lapf_problem& pb = cfg->problem;
    if (!stamp_supported(pb.ny, pb.nx))
        return fail(LAPF_ERR_INVALID, "sampler supports square stamps of 32, 64 or 128 pixels, got %dx%d", pb.ny, pb.nx);
    if (cfg->n_walkers <= 0 || cfg->n_walkers > (int64_t)1 << 30)
        return fail(LAPF_ERR_INVALID, "n_walkers %lld out of range", (long long)cfg->n_walkers);
    if (!cfg->init_params) return fail(LAPF_ERR_INVALID, "init_params is NULL");
    if (cfg->thin < 1 || cfg->thin > (1 << 30)) return fail(LAPF_ERR_INVALID, "thin must be in [1, 2^30]");
    if (cfg->burn_in < 0) return fail(LAPF_ERR_INVALID, "burn_in must be >= 0");
    if (cfg->team_warps != 0 && cfg->team_warps != 1 && cfg->team_warps != 4 && cfg->team_warps != 16)
        return fail(LAPF_ERR_INVALID, "team_warps %d not supported (0, 1, 4 or 16)", cfg->team_warps);
    if ((rc = require_device())) return rc;
    cudaStream_t st = (cudaStream_t)stream;

    lapf_sampler* s = new (std::nothrow) lapf_sampler();
    if (!s) return fail(LAPF_ERR_NOMEM, "out of host memory");
    s->cfg = *cfg;
    s->P = 3 * pb.nbody + 10;
    s->team = cfg->team_warps ? cfg->team_warps : 1;
    const int P = s->P;
    const int64_t W = cfg->n_walkers;
    cudaGetDevice(&s->device);
    const double* wsrc = cfg->widths ? cfg->widths : (pb.nbody == 2 ? kWidths2 : kWidths3);
    for (int i = 0; i < LAPF_MAX_PARAMS; ++i) s->widths[i] = i < P ? wsrc[i] : 0.0;
    s->cfg.widths = nullptr;
    s->log_mask = log_mask_for(pb.nbody);

#define CUS(call)                                                                                  \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) {                                                                  \
            free_sampler(s);                                                                       \
            return fail(LAPF_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__),    \
                        __FILE__, __LINE__);                                                       \
        }                                                                                          \
    } while (0)

    if ((rc = configure_dispatch(s))) { free_sampler(s); return rc; }

    // group walkers by frame (counting sort) and cut each frame's list into CTA-sized items
    std::vector<int32_t> fo((size_t)W, 0);
    if (cfg->frame_of) {
        CUS(cudaMemcpyAsync(fo.data(), cfg->frame_of, sizeof(int32_t) * W, cudaMemcpyDeviceToHost, st));
        CUS(cudaStreamSynchronize(st));
    }
    const int F = pb.n_frames;
    std::vector<int32_t> start((size_t)F + 1, 0);
    for (int64_t w = 0; w < W; ++w) {
        if (fo[w] < 0 || fo[w] >= F) {
            free_sampler(s);
            return fail(LAPF_ERR_INVALID, "frame_of[%lld] = %d outside [0,%d)", (long long)w, fo[w], F);
        }
        start[fo[w] + 1]++;
    }
    for (int f = 0; f < F; ++f) start[f + 1] += start[f];
    std::vector<int32_t> order((size_t)W), fill(start.begin(), start.end() - 1);
    for (int64_t w = 0; w < W; ++w) order[fill[fo[w]]++] = (int32_t)w;
    std::vector<int32_t> it_frame, it_first, it_count, cta_item, it_frame2, it_count_a, it_slot_a;
    if (s->team == 1) {
        // Batched kernel: CTA b owns the contiguous share [b W / G, (b+1) W / G) of the frame-sorted walkers, cut
        // into items of at most `chunk` walkers.  Up to 64 x 64 pixels the pixel store holds two stamps, and an
        // item may then run across ONE frame boundary: its first part is evaluated on one slot, the rest on the
        // other.  (Otherwise a share of 443 walkers over frames of 655 is two items of ~220, i.e. ~14 of a
        // warp's 32 lanes busy in the one-walker-per-lane section of every round.)  A frame stays in the slot
        // it was staged into while consecutive items of the CTA need it.
        const int64_t G = std::min<int64_t>(s->grid, W);
        const bool two = pb.nx <= 64;
        s->launch_grid = (int)G;
        int f = 0;
        for (int64_t b = 0; b < G; ++b) {
            cta_item.push_back((int32_t)it_frame.size());
            int64_t lo = (W * b) / G;
            const int64_t hi = (W * (b + 1)) / G;
            int slot_frame[2] = {-1, -1};
            while (lo < hi) {
                while (start[f + 1] <= lo) ++f;
                const int64_t n = std::min<int64_t>(hi - lo, s->chunk);                 // walkers of this item
                const int64_t na = std::min<int64_t>(n, start[f + 1] - lo);              // ... of frame f
                int f2 = -1;
                int64_t nb = 0;
                if (two && na < n) {                                                     // the rest: the next frame with walkers
                    f2 = f + 1;
                    while (start[f2 + 1] <= lo + na) ++f2;
                    nb = std::min<int64_t>(n - na, start[f2 + 1] - (lo + na));
                }
                // slot of frame f: where it already is, else the slot that does not hold f2
                int sa = (slot_frame[1] == f) ? 1 : (slot_frame[0] == f) ? 0 : (f2 >= 0 && slot_frame[0] == f2) ? 1 : 0;
                if (!two) sa = 0;
                slot_frame[sa] = f;
                if (f2 >= 0) slot_frame[1 - sa] = f2;
                it_frame.push_back(slot_frame[0]);
                it_frame2.push_back(two ? slot_frame[1] : -1);
                it_first.push_back((int32_t)lo);
                it_count.push_back((int32_t)(na + nb));
                it_count_a.push_back((int32_t)na);
                it_slot_a.push_back(sa);
                lo += na + nb;
            }
        }
        cta_item.push_back((int32_t)it_frame.size());
    } else {
        for (int f = 0; f < F; ++f)
            for (int32_t b = start[f]; b < start[f + 1]; b += s->nw) {
                it_frame.push_back(f);
                it_first.push_back(b);
                it_count.push_back(std::min<int32_t>(s->nw, start[f + 1] - b));
            }
        cta_item.push_back(0);
    }
    s->n_items = (int)it_frame.size();

    const size_t nst = (size_t)W * (P + 1);
    CUS(cudaMalloc((void**)&s->state, sizeof(double) * nst));
    CUS(cudaMalloc((void**)&s->shift, sizeof(double) * nst));
    CUS(cudaMalloc((void**)&s->moments, sizeof(double) * nst * 2));
    CUS(cudaMalloc((void**)&s->tries, sizeof(uint32_t) * W * P));
    CUS(cudaMalloc((void**)&s->accepts, sizeof(uint32_t) * W * P));
    CUS(cudaMalloc((void**)&s->exps, sizeof(unsigned long long) * W));
    CUS(cudaMalloc((void**)&s->walker_of, sizeof(int32_t) * W));
    CUS(cudaMalloc((void**)&s->frame_start, sizeof(int32_t) * (F + 1)));
    CUS(cudaMalloc((void**)&s->item_frame, sizeof(int32_t) * s->n_items));
    CUS(cudaMalloc((void**)&s->item_first, sizeof(int32_t) * s->n_items));
    CUS(cudaMalloc((void**)&s->item_count, sizeof(int32_t) * s->n_items));
    if (s->team == 1) {
        CUS(cudaMalloc((void**)&s->item_frame2, sizeof(int32_t) * s->n_items));
        CUS(cudaMalloc((void**)&s->item_count_a, sizeof(int32_t) * s->n_items));
        CUS(cudaMalloc((void**)&s->item_slot_a, sizeof(int32_t) * s->n_items));
        CUS(cudaMemcpyAsync(s->item_frame2, it_frame2.data(), sizeof(int32_t) * s->n_items, cudaMemcpyHostToDevice, st));
        CUS(cudaMemcpyAsync(s->item_count_a, it_count_a.data(), sizeof(int32_t) * s->n_items, cudaMemcpyHostToDevice, st));
        CUS(cudaMemcpyAsync(s->item_slot_a, it_slot_a.data(), sizeof(int32_t) * s->n_items, cudaMemcpyHostToDevice, st));
    }
    CUS(cudaMalloc((void**)&s->cta_item, sizeof(int32_t) * cta_item.size()));
    CUS(cudaMalloc((void**)&s->frame_of, sizeof(int32_t) * W));
    CUS(cudaMemcpyAsync(s->frame_of, fo.data(), sizeof(int32_t) * W, cudaMemcpyHostToDevice, st));
    s->cfg.frame_of = s->frame_of;
    CUS(cudaMemcpyAsync(s->walker_of, order.data(), sizeof(int32_t) * W, cudaMemcpyHostToDevice, st));
    CUS(cudaMemcpyAsync(s->frame_start, start.data(), sizeof(int32_t) * (F + 1), cudaMemcpyHostToDevice, st));
    CUS(cudaMemcpyAsync(s->item_frame, it_frame.data(), sizeof(int32_t) * s->n_items, cudaMemcpyHostToDevice, st));
    CUS(cudaMemcpyAsync(s->item_first, it_first.data(), sizeof(int32_t) * s->n_items, cudaMemcpyHostToDevice, st));
    CUS(cudaMemcpyAsync(s->item_count, it_count.data(), sizeof(int32_t) * s->n_items, cudaMemcpyHostToDevice, st));
    CUS(cudaMemcpyAsync(s->cta_item, cta_item.data(), sizeof(int32_t) * cta_item.size(), cudaMemcpyHostToDevice, st));

    CUS(cudaStreamSynchronize(st));   // the host vectors above are pageable
    rc = lapf_sampler_reset(s, cfg->init_params, cfg->seed, st);
    if (rc) { free_sampler(s); return rc; }
    // three probe updates against the stateless operator, then the state is put back (LAPF_NO_SELFTEST=1 skips it)
    if (!getenv("LAPF_NO_SELFTEST") && (rc = lapf_sampler_selftest(s, st))) { free_sampler(s); return rc; }
#undef CUS
    *out = s;
    return LAPF_OK;
}

static size_t sketch_hist_bytes(const lapf_sampler* s) {
    return sizeof(uint32_t) * (size_t)s->cfg.problem.n_frames * 2 * (s->cfg.problem.nbody - 1) * (s->sk_bins + 2);
}
static size_t sketch_mom_bytes(const lapf_sampler* s) {
    return sizeof(double) * (size_t)s->cfg.n_walkers * 2 * (s->cfg.problem.nbody - 1) * 2;
}
static size_t bm_state_bytes(const lapf_sampler* s) {
    return sizeof(double) * (size_t)s->cfg.n_walkers * s->bm_c * s->bm_levels * 2;
}
static size_t draws_val_bytes(const lapf_sampler* s) { return sizeof(double) * (size_t)s->cfg.n_walkers * s->dr_k * (s->P + 1); }
static size_t draws_row_bytes(const lapf_sampler* s) { return sizeof(int64_t) * (size_t)s->cfg.n_walkers * s->dr_k; }
static size_t fw_bytes(const lapf_sampler* s) { return sizeof(double) * (size_t)s->cfg.problem.n_frames * s->P; }
static size_t fw_snap_bytes(const lapf_sampler* s) { return 2 * sizeof(long long) * (size_t)s->cfg.problem.n_frames * s->P; }
static size_t prior_bytes(const lapf_sampler* s) { return 4 * sizeof(double) * (size_t)s->cfg.problem.n_frames * s->P; }

// Checkpoint layout: see lapf_sampler_save in lapf.h.  The head [count][seed][jump widths x LAPF_MAX_PARAMS] is
// built on the host; checkpoint_layout lists the sections that follow it, and every size, offset, copy, reset
// fill and load check is derived from that list.
constexpr size_t kCkptHead = 8 * (2 + LAPF_MAX_PARAMS);
constexpr size_t kCkptDesc = 32;   // int64 {magic, a, b, c}
constexpr int kKeep = -1;          // a part lapf_sampler_reset does not overwrite
// A device buffer of the sampler (the address of the field that owns it), its size and the byte that
// lapf_sampler_reset writes over it (or kKeep)
struct Part { void** dev; size_t bytes; int fill; };
// The sections that start with a descriptor; its magic identifies the section in any blob
struct Described { int64_t magic; const char* name; const char* fields; const char* enable; };
static const Described kBatchMeans = {0x31304d424650414cLL, "batch means", "batch_rows, levels, quantities",   // 'LAPFBM01'
                                      "lapf_sampler_batchmeans_enable"};
static const Described kDraws = {0x313053524650414cLL, "posterior draws", "per walker, columns, 0",            // 'LAPFRS01'
                                  "lapf_sampler_draws_enable"};
static const Described kFrameWidths = {0x313057464650414cLL, "per-frame jump widths", "frames, parameters, 0", // 'LAPFFW01'
                                       "lapf_sampler_set_frame_widths"};
static const Described kPriors = {0x313052504650414cLL, "parameter priors", "frames, parameters, 0",         // 'LAPFPR01'
                                  "lapf_sampler_set_priors"};
static const Described* const kDescribed[] = {&kBatchMeans, &kDraws, &kFrameWidths, &kPriors};
struct Section {
    const Described* desc;   // nullptr: no descriptor
    int64_t val[3];          // the descriptor's a, b, c
    int n_parts;
    Part part[6];
    size_t at;               // offset in the blob (of the descriptor, if any)
};
constexpr int kSections = 6;   // core, sketches, batch means, draws, per-frame widths, priors
struct CkptLayout { int n; Section sec[kSections]; size_t bytes; };

static CkptLayout checkpoint_layout(lapf_sampler* s) {
    const size_t W = (size_t)s->cfg.n_walkers, P = (size_t)s->P, nst = W * (P + 1);
    CkptLayout L = {};
    L.sec[L.n++] = {nullptr, {}, 6, {{(void**)&s->state, sizeof(double) * nst, kKeep},   // pack_state_kernel in reset
                                     {(void**)&s->shift, sizeof(double) * nst, kKeep},
                                     {(void**)&s->moments, sizeof(double) * nst * 2, 0},
                                     {(void**)&s->exps, sizeof(unsigned long long) * W, 0},
                                     {(void**)&s->tries, sizeof(uint32_t) * W * P, 0},
                                     {(void**)&s->accepts, sizeof(uint32_t) * W * P, 0}}};
    if (s->sk_hist)
        L.sec[L.n++] = {nullptr, {}, 2, {{(void**)&s->sk_mom, sketch_mom_bytes(s), 0},
                                         {(void**)&s->sk_hist, sketch_hist_bytes(s), 0}}};
    if (s->bm)
        L.sec[L.n++] = {&kBatchMeans, {s->bm_rows, s->bm_levels, s->bm_c}, 1, {{(void**)&s->bm, bm_state_bytes(s), 0}}};
    if (s->dr_val)   // an empty reservoir: every row index -1, every value the all-ones NaN
        L.sec[L.n++] = {&kDraws, {s->dr_k, s->P + 1, 0}, 2, {{(void**)&s->dr_val, draws_val_bytes(s), 0xFF},
                                                              {(void**)&s->dr_row, draws_row_bytes(s), 0xFF}}};
    if (s->fw)       // reset keeps the widths; the counters start again, so does the adaptation window
        L.sec[L.n++] = {&kFrameWidths, {s->cfg.problem.n_frames, s->P, 0}, 2,
                        {{(void**)&s->fw, fw_bytes(s), kKeep}, {(void**)&s->fw_snap, fw_snap_bytes(s), 0}}};
    if (s->pr)       // reset keeps the table (and refuses starts outside it)
        L.sec[L.n++] = {&kPriors, {s->cfg.problem.n_frames, s->P, 0}, 2,
                        {{(void**)&s->pr, prior_bytes(s), kKeep}, {(void**)&s->pr_given, prior_bytes(s), kKeep}}};
    L.bytes = kCkptHead;
    for (int i = 0; i < L.n; ++i) {
        Section& c = L.sec[i];
        c.at = L.bytes;
        L.bytes += c.desc ? kCkptDesc : 0;
        for (int j = 0; j < c.n_parts; ++j) L.bytes += c.part[j].bytes;
    }
    return L;
}

static size_t checkpoint_bytes(const lapf_sampler* s) {
    return checkpoint_layout(const_cast<lapf_sampler*>(s)).bytes;   // reads sizes only
}

// Priors: LAPF_ERR_INVALID, naming the first walker, frame and parameter, if any parameter of `params` (walker w
// at params[w * stride], frame s->frame_of[w]) lies outside the box of `table` (device [F][P][4] {lo, hi, ...}).
static int prior_check(lapf_sampler* s, const double* params, int stride, const double* table, const char* what,
                       cudaStream_t st) {
    const int64_t W = s->cfg.n_walkers;
    const int P = s->P;
    unsigned long long* out = nullptr;
    const unsigned long long init[2] = {0ull, ~0ull};
    unsigned long long res[2] = {0, 0};
    CU(cudaMallocAsync((void**)&out, sizeof(init), st));
    cudaError_t e = cudaMemcpyAsync(out, init, sizeof(init), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) {
        prior_outside_kernel<<<(unsigned)((W + 255) / 256), 256, 0, st>>>(params, stride, s->frame_of, table, P, W, out);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(res, out, sizeof(res), cudaMemcpyDeviceToHost, st);
    cudaFreeAsync(out, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);   // `init` and `res` live on this stack frame
    if (e != cudaSuccess) return fail(LAPF_ERR_CUDA, "prior check failed: %s", cudaGetErrorString(e));
    s->launches++;
    if (res[0] == 0) return LAPF_OK;
    const int64_t w = (int64_t)((res[1] - 1) / P);
    const int j = (int)((res[1] - 1) % P);
    int32_t f = 0;
    double v = 0.0, box[2] = {0.0, 0.0};
    CU(cudaMemcpyAsync(&f, s->frame_of + w, sizeof(f), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(&v, params + w * stride + j, sizeof(v), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaMemcpyAsync(box, table + ((size_t)f * P + j) * 4, sizeof(box), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return fail(LAPF_ERR_INVALID, "%s: %llu parameter value(s) lie outside their prior box; the first is frame %d, "
                "parameter %d of walker %lld: %.17g not in [%g, %g]", what, res[0], f, j, (long long)w, v, box[0], box[1]);
}

int lapf_sampler_reset(lapf_sampler* s, const double* init_params, uint64_t seed, void* stream) {
    if (!s || !init_params) return fail(LAPF_ERR_INVALID, "sampler/init_params is NULL");
    cudaStream_t st = (cudaStream_t)stream;
    const int P = s->P;
    const int64_t W = s->cfg.n_walkers;
    const size_t nst = (size_t)W * (P + 1);
    int rc = s->pr ? prior_check(s, init_params, P, s->pr, "reset refused", st) : LAPF_OK;
    if (rc) return rc;                                   // before anything changes
    const CkptLayout L = checkpoint_layout(s);
    for (int i = 0; i < L.n; ++i)
        for (int j = 0; j < L.sec[i].n_parts; ++j) {
            const Part& p = L.sec[i].part[j];
            if (p.fill != kKeep) CU(cudaMemsetAsync(*p.dev, p.fill, p.bytes, st));
        }
    // initial chi-square (apf_step2.py:283-289) through K1, then pack the state
    double* chi0 = nullptr;
    CU(cudaMallocAsync((void**)&chi0, sizeof(double) * W, st));
    rc = lapf_model_chi2(&s->cfg.problem, init_params, W, s->cfg.frame_of, nullptr, chi0, st);
    if (rc) { cudaFreeAsync(chi0, st); return rc; }
    pack_state_kernel<<<(unsigned)((nst + 255) / 256), 256, 0, st>>>(init_params, chi0, P, W, s->state, s->shift);
    CU(cudaGetLastError());
    CU(cudaFreeAsync(chi0, st));
    s->launches += 2;
    s->cfg.seed = seed;
    s->count = 0;
    if (s->sk_hist && s->sk_auto_center) {
        const int F = s->cfg.problem.n_frames, nbody = s->cfg.problem.nbody;
        sketch_center_kernel<<<(F * (nbody - 1) + 127) / 128, 128, 0, st>>>(s->shift, s->walker_of, s->frame_start, F, P,
                                                                          nbody, s->sk_center);
        CU(cudaGetLastError());
        s->launches++;
    }
    return LAPF_OK;
}

int64_t lapf_sampler_checkpoint_bytes(const lapf_sampler* s) {
    if (!s) return fail(LAPF_ERR_INVALID, "sampler is NULL");
    return (int64_t)checkpoint_bytes(s);
}

// Copies every part between the sampler and the blob; the descriptors are written (save) or checked (load) by
// the caller
static int checkpoint_copy(const CkptLayout& L, unsigned char* blob, bool save, cudaStream_t st) {
    for (int i = 0; i < L.n; ++i) {
        size_t off = L.sec[i].at + (L.sec[i].desc ? kCkptDesc : 0);
        for (int j = 0; j < L.sec[i].n_parts; ++j) {
            const Part& p = L.sec[i].part[j];
            CU(cudaMemcpyAsync(save ? (void*)(blob + off) : *p.dev, save ? *p.dev : (const void*)(blob + off), p.bytes,
                               cudaMemcpyDeviceToDevice, st));
            off += p.bytes;
        }
    }
    return LAPF_OK;
}

int lapf_sampler_save(lapf_sampler* s, void* blob, int64_t blob_bytes, void* stream) {
    if (!s || !blob) return fail(LAPF_ERR_INVALID, "sampler/blob is NULL");
    const CkptLayout L = checkpoint_layout(s);
    if ((size_t)blob_bytes < L.bytes) return fail(LAPF_ERR_INVALID, "checkpoint buffer too small");
    cudaStream_t st = (cudaStream_t)stream;
    int64_t head[2 + LAPF_MAX_PARAMS] = {s->count, (int64_t)s->cfg.seed};
    memcpy(head + 2, s->widths, sizeof(double) * LAPF_MAX_PARAMS);   // --adapt may have changed them
    CU(cudaMemcpyAsync(blob, head, kCkptHead, cudaMemcpyHostToDevice, st));
    int64_t desc[kSections][4];
    for (int i = 0; i < L.n; ++i) {
        const Section& c = L.sec[i];
        if (!c.desc) continue;
        desc[i][0] = c.desc->magic;
        memcpy(desc[i] + 1, c.val, sizeof(c.val));
        CU(cudaMemcpyAsync((unsigned char*)blob + c.at, desc[i], kCkptDesc, cudaMemcpyHostToDevice, st));
    }
    CU(cudaStreamSynchronize(st));   // `head` and the descriptors live on this stack frame
    return checkpoint_copy(L, (unsigned char*)blob, true, st);
}

static const Described* described_by(int64_t magic) {
    for (const Described* d : kDescribed)
        if (d->magic == magic) return d;
    return nullptr;
}

int lapf_sampler_load(lapf_sampler* s, const void* blob, int64_t blob_bytes, void* stream) {
    if (!s || !blob) return fail(LAPF_ERR_INVALID, "sampler/blob is NULL");
    const CkptLayout L = checkpoint_layout(s);
    if ((size_t)blob_bytes < L.bytes) return fail(LAPF_ERR_INVALID, "checkpoint buffer too small");
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned char* b = (const unsigned char*)blob;
    // the head, every descriptor this sampler expects, and the 32 bytes past its layout (where a section it
    // does not have would start), in one round trip
    int64_t head[2 + LAPF_MAX_PARAMS] = {0, 0};
    int64_t desc[kSections + 1][4] = {};
    CU(cudaMemcpyAsync(head, b, kCkptHead, cudaMemcpyDeviceToHost, st));
    for (int i = 0; i < L.n; ++i)
        if (L.sec[i].desc) CU(cudaMemcpyAsync(desc[i], b + L.sec[i].at, kCkptDesc, cudaMemcpyDeviceToHost, st));
    if ((size_t)blob_bytes >= L.bytes + kCkptDesc) CU(cudaMemcpyAsync(desc[L.n], b + L.bytes, kCkptDesc, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    double wd[LAPF_MAX_PARAMS];
    memcpy(wd, head + 2, sizeof(wd));
    bool ok = head[0] >= 0;
    for (int i = 0; i < s->P; ++i) ok = ok && wd[i] >= 0.0 && std::isfinite(wd[i]);
    if (!ok) return fail(LAPF_ERR_INVALID, "corrupt checkpoint (count %lld)", (long long)head[0]);
    for (int i = 0; i < L.n; ++i) {
        const Described* want = L.sec[i].desc;
        const int64_t* got = desc[i];
        const int64_t* val = L.sec[i].val;
        if (!want) continue;
        if (got[0] != want->magic) {
            if (const Described* found = described_by(got[0]))
                return fail(LAPF_ERR_INVALID, "checkpoint carries %s where this sampler expects %s", found->name, want->name);
            return fail(LAPF_ERR_INVALID, "checkpoint carries no %s where this sampler expects them", want->name);
        }
        if (got[1] != val[0] || got[2] != val[1] || got[3] != val[2])
            return fail(LAPF_ERR_INVALID, "checkpoint %s (%s) = (%lld, %lld, %lld) do not match this sampler's (%lld, %lld, "
                        "%lld)", want->name, want->fields, (long long)got[1], (long long)got[2], (long long)got[3],
                        (long long)val[0], (long long)val[1], (long long)val[2]);
    }
    if (const Described* extra = described_by(desc[L.n][0]))
        return fail(LAPF_ERR_INVALID, "checkpoint carries %s, this sampler has none (%s before lapf_sampler_load)",
                    extra->name, extra->enable);
    s->count = head[0];
    s->cfg.seed = (uint64_t)head[1];
    memcpy(s->widths, wd, sizeof(wd));
    return checkpoint_copy(L, (unsigned char*)const_cast<void*>(blob), false, st);
}

int lapf_sampler_set_widths(lapf_sampler* s, const double* widths) {
    if (!s || !widths) return fail(LAPF_ERR_INVALID, "sampler/widths is NULL");
    if (s->fw) return fail(LAPF_ERR_INVALID, "per-frame jump widths are on: set them with lapf_sampler_set_frame_widths");
    for (int i = 0; i < s->P; ++i)
        if (!(widths[i] >= 0.0)) return fail(LAPF_ERR_INVALID, "widths[%d] = %g is not a valid jump width", i, widths[i]);
    for (int i = 0; i < s->P; ++i) s->widths[i] = widths[i];
    return LAPF_OK;
}

int lapf_sampler_destroy(lapf_sampler* s) {
    free_sampler(s);
    return LAPF_OK;
}

int64_t lapf_sampler_rows_for(const lapf_sampler* s, int64_t n_updates) {
    if (!s || n_updates < 0) return fail(LAPF_ERR_INVALID, "bad arguments");
    return rows_upto(s->count + n_updates, s->cfg.burn_in, s->cfg.thin) -
           rows_upto(s->count, s->cfg.burn_in, s->cfg.thin);
}

static bool is_event_format(int format) { return format == LAPF_CHAIN_EVENTS_F64 || format == LAPF_CHAIN_EVENTS_F32_DELTA; }
static bool is_f32_format(int format) { return format == LAPF_CHAIN_F32_DELTA || format == LAPF_CHAIN_EVENTS_F32_DELTA; }
static int64_t event_codes_bytes(int64_t rows, int64_t W) { return (rows * W + 15) & ~(int64_t)15; }

// Bytes a run that records `rows` rows writes in the current format (include/lapf.h: the event layout).
static int64_t chain_bytes_for_rows(const lapf_sampler* s, int64_t rows) {
    const int64_t W = s->cfg.n_walkers, e = is_f32_format(s->chain_format) ? 4 : 8;
    if (!is_event_format(s->chain_format)) return rows * W * (s->P + 1) * e;
    if (rows == 0) return 0;
    return e * W * (s->P + 1) + event_codes_bytes(rows, W) + 2 * e * rows * W;
}

int64_t lapf_sampler_chain_bytes(const lapf_sampler* s, int64_t n_updates) {
    const int64_t rows = lapf_sampler_rows_for(s, n_updates);
    return rows < 0 ? rows : chain_bytes_for_rows(s, rows);
}

int64_t lapf_sampler_count(const lapf_sampler* s) { return s ? s->count : fail(LAPF_ERR_INVALID, "sampler is NULL"); }
int64_t lapf_sampler_launches(const lapf_sampler* s) { return s ? s->launches : fail(LAPF_ERR_INVALID, "sampler is NULL"); }

static void fill_run_args(const lapf_sampler* s, RunArgs& a, int64_t n_updates, void* chain_out) {
    const lapf_problem& pb = s->cfg.problem;
    a.data = pb.data; a.weight = pb.weight; a.origin = pb.origin; a.outside = pb.outside;
    a.item_frame = s->item_frame; a.item_first = s->item_first; a.item_count = s->item_count;
    a.item_frame2 = s->item_frame2; a.item_count_a = s->item_count_a; a.item_slot_a = s->item_slot_a;
    a.walker_of = s->walker_of; a.cta_item = s->cta_item;
    a.state = s->state; a.shift = s->shift; a.moments = s->moments;
    a.tries = s->tries; a.accepts = s->accepts; a.exps = s->exps;
    a.chain = chain_out;
    a.chain_f32 = is_f32_format(s->chain_format) ? 1 : 0;
    a.chain_ev = (chain_out && is_event_format(s->chain_format)) ? 1 : 0;
    a.ev_code = nullptr; a.ev_val = nullptr; a.ev_chi = nullptr;
    if (a.chain_ev) {
        const int64_t rows = lapf_sampler_rows_for(s, n_updates), W = s->cfg.n_walkers, e = a.chain_f32 ? 4 : 8;
        a.ev_code = static_cast<unsigned char*>(chain_out) + e * W * (s->P + 1);
        a.ev_val = a.ev_code + event_codes_bytes(rows, W);
        a.ev_chi = static_cast<unsigned char*>(a.ev_val) + e * rows * W;
    }
    a.sk_hist = s->sk_hist; a.sk_center = s->sk_center; a.sk_mom = s->sk_mom;
    a.sk_bins = s->sk_bins;
    a.sk_inv_sep = s->sk_bins ? 1.0 / s->sk_sep_bin : 0.0;
    a.sk_inv_pa = s->sk_bins ? 1.0 / s->sk_pa_bin : 0.0;
    a.n_walkers = s->cfg.n_walkers;
    a.t0 = s->count; a.n_updates = n_updates;
    a.next_record = next_record_after(s->count, s->cfg.burn_in, s->cfg.thin);
    a.id_base = s->cfg.id_base; a.id_stride = s->cfg.id_stride;
    a.seed = s->cfg.seed;
    memcpy(a.widths, s->widths, sizeof(a.widths));
    a.log_mask = s->log_mask;
    a.thin = s->cfg.thin; a.floor_index = pb.floor_index; a.n_items = s->n_items;
    a.cull = cull_enabled(&pb);
    a.plain = plain_loop(&pb);
    a.bm = s->bm; a.bm_rows = s->bm_rows; a.bm_levels = s->bm_levels; a.bm_c = s->bm_c;
    a.bm_q0 = 0; a.bm_phase = 0;
    if (s->bm) {
        const int64_t r0 = rows_upto(s->count, s->cfg.burn_in, s->cfg.thin);
        a.bm_q0 = r0 / s->bm_rows;
        a.bm_phase = (int)(r0 % s->bm_rows);
    }
    a.dr_val = s->dr_val; a.dr_row = s->dr_row; a.dr_k = s->dr_k;
    a.dr_row0 = s->dr_val ? rows_upto(s->count, s->cfg.burn_in, s->cfg.thin) : 0;
    a.fwidths = s->fw;
    a.prior = s->pr;
    a.probe = nullptr;
    a.cta_times = nullptr;
}

int lapf_sampler_run(lapf_sampler* s, int64_t n_updates, void* chain_out, int64_t rows_cap, void* stream) {
    if (!s) return fail(LAPF_ERR_INVALID, "sampler is NULL");
    if (n_updates < 0 || n_updates > ((int64_t)1 << 30))
        return fail(LAPF_ERR_INVALID, "n_updates must be in [0, 2^30] per launch");
    if (n_updates == 0) return LAPF_OK;
    if (is_event_format(s->chain_format) && s->cfg.thin != 1)
        return fail(LAPF_ERR_INVALID, "event chain formats need thin = 1 (thin is %d)", s->cfg.thin);
    const int64_t rows = lapf_sampler_rows_for(s, n_updates);
    if (chain_out && rows_cap < rows)
        return fail(LAPF_ERR_INVALID, "chain_out holds %lld rows but this run records %lld", (long long)rows_cap, (long long)rows);
    RunArgs a;
    fill_run_args(s, a, n_updates, chain_out);
    if (a.chain_ev && rows > 0) {
        // the padding of the codes: every byte of the buffer is written, so equal runs give equal buffers
        const int64_t n_codes = rows * s->cfg.n_walkers, pad = event_codes_bytes(rows, s->cfg.n_walkers) - n_codes;
        if (pad) CU(cudaMemsetAsync(a.ev_code + n_codes, 0, (size_t)pad, (cudaStream_t)stream));
    }
    // diagnosis (LAPF_CTA_TIMES=<file>): start, end and SM of every CTA of the batched kernel, one text line per launch
    const char* times_path = s->team == 1 ? getenv("LAPF_CTA_TIMES") : nullptr;
    if (times_path) CU(cudaMalloc((void**)&a.cta_times, sizeof(unsigned long long) * 3 * s->launch_grid));
    int rc = launch_dispatch(s, a, (cudaStream_t)stream);
    if (times_path) {
        std::vector<unsigned long long> h((size_t)3 * s->launch_grid);
        cudaStreamSynchronize((cudaStream_t)stream);
        cudaMemcpy(h.data(), a.cta_times, sizeof(unsigned long long) * h.size(), cudaMemcpyDeviceToHost);
        cudaFree(a.cta_times);
        if (FILE* f = fopen(times_path, "a")) {
            unsigned long long t0 = ~0ull;
            for (int b = 0; b < s->launch_grid; ++b) t0 = std::min(t0, h[3 * b]);
            for (int b = 0; b < s->launch_grid; ++b)
                fprintf(f, "%llu:%llu:%llu ", h[3 * b] - t0, h[3 * b + 1] - t0, h[3 * b + 2]);
            fprintf(f, "\n");
            fclose(f);
        }
    }
    if (rc) return rc;
    s->count += n_updates;
    s->launches++;
    return LAPF_OK;
}

int lapf_sampler_state(lapf_sampler* s, double* state_out, uint32_t* tries_out, uint32_t* accepts_out, void* stream) {
    if (!s) return fail(LAPF_ERR_INVALID, "sampler is NULL");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t W = s->cfg.n_walkers;
    if (state_out) CU(cudaMemcpyAsync(state_out, s->state, sizeof(double) * W * (s->P + 1), cudaMemcpyDeviceToDevice, st));
    if (tries_out) CU(cudaMemcpyAsync(tries_out, s->tries, sizeof(uint32_t) * W * s->P, cudaMemcpyDeviceToDevice, st));
    if (accepts_out) CU(cudaMemcpyAsync(accepts_out, s->accepts, sizeof(uint32_t) * W * s->P, cudaMemcpyDeviceToDevice, st));
    return LAPF_OK;
}

int lapf_sampler_stats(lapf_sampler* s, int64_t* totals_out, double* moments_out, int64_t* counts_out, void* stream) {
    if (!s) return fail(LAPF_ERR_INVALID, "sampler is NULL");
    cudaStream_t st = (cudaStream_t)stream;
    const int P = s->P;
    const int64_t W = s->cfg.n_walkers;
    const int64_t n_rows = rows_upto(s->count, s->cfg.burn_in, s->cfg.thin);
    if (totals_out) {
        totals_init_kernel<<<1, 64, 0, st>>>((unsigned long long*)totals_out, P);
        const unsigned gx = (unsigned)std::min<int64_t>(148, (W + 255) / 256);
        totals_kernel<<<dim3(gx, P), 256, 0, st>>>(s->tries, s->accepts, s->exps, P, W, (unsigned long long*)totals_out);
        CU(cudaGetLastError());
        s->launches += 2;
    }
    if (moments_out) {
        moments_kernel<<<s->cfg.problem.n_frames, 32 * (P + 1), 0, st>>>(s->moments, s->shift, s->walker_of,
                                                                        s->frame_start, P, n_rows, moments_out);
        CU(cudaGetLastError());
        s->launches++;
    }
    if (counts_out) {
        const int F = s->cfg.problem.n_frames;
        counts_kernel<<<(F + 1 + 127) / 128, 128, 0, st>>>(s->frame_start, F, n_rows, (long long*)counts_out);
        CU(cudaGetLastError());
        s->launches++;
    }
    return LAPF_OK;
}

int lapf_sampler_selftest(lapf_sampler* s, void* stream) {
    if (!s) return fail(LAPF_ERR_INVALID, "sampler is NULL");
    if (s->team != 1) return LAPF_OK;                       // the team kernels keep no TMEM pixel store
    cudaStream_t st = (cudaStream_t)stream;
    const int P = s->P, U = 3;
    const int64_t W = s->cfg.n_walkers;
    const size_t nst = (size_t)W * (P + 1), blob_bytes = checkpoint_bytes(s);
    unsigned char* blob = nullptr;
    double *chain = nullptr, *probe = nullptr, *trials = nullptr, *chi = nullptr, *start = nullptr;
    int32_t* fo = nullptr;
    unsigned long long* out = nullptr;
    auto cleanup = [&]() {
        for (void* q : {(void*)blob, (void*)chain, (void*)probe, (void*)trials, (void*)chi, (void*)start, (void*)fo, (void*)out})
            if (q) cudaFreeAsync(q, st);
    };
#define CUT(call)                                                                                  \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) {                                                                  \
            cleanup();                                                                             \
            return fail(LAPF_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
        }                                                                                          \
    } while (0)
    CUT(cudaMallocAsync((void**)&blob, blob_bytes, st));
    CUT(cudaMallocAsync((void**)&chain, sizeof(double) * nst * U, st));
    CUT(cudaMallocAsync((void**)&probe, sizeof(double) * (size_t)W * 3 * U, st));
    CUT(cudaMallocAsync((void**)&trials, sizeof(double) * (size_t)W * P * U, st));
    CUT(cudaMallocAsync((void**)&chi, sizeof(double) * (size_t)W * U, st));
    CUT(cudaMallocAsync((void**)&start, sizeof(double) * nst, st));
    CUT(cudaMallocAsync((void**)&fo, sizeof(int32_t) * (size_t)W * U, st));
    CUT(cudaMallocAsync((void**)&out, 16, st));
    int rc = lapf_sampler_save(s, blob, (int64_t)blob_bytes, st);
    if (rc) { cleanup(); return rc; }
    CUT(cudaMemcpyAsync(start, s->state, sizeof(double) * nst, cudaMemcpyDeviceToDevice, st));
    for (int u = 0; u < U; ++u)
        CUT(cudaMemcpyAsync(fo + (size_t)u * W, s->frame_of, sizeof(int32_t) * W, cudaMemcpyDeviceToDevice, st));
    // U updates, every one recorded (the build that failed mis-evaluated the update AFTER a recorded one), rows as
    // doubles, no sketches; the trial chi-squares leave through `probe`
    RunArgs a;
    fill_run_args(s, a, U, chain);
    a.thin = 1;
    a.next_record = a.t0 + 1;
    a.chain_f32 = 0;
    a.chain_ev = 0;
    a.ev_code = nullptr; a.ev_val = nullptr; a.ev_chi = nullptr;
    a.sk_hist = nullptr;
    // batch means (if on) with batch length 1: every recorded row closes a batch, so the update after each
    // closing row is checked too; the load below restores their state
    a.bm_rows = 1; a.bm_q0 = 0; a.bm_phase = 0;
    // posterior draws (if on) with one slot per walker: rows 1 and 2 take the replacement path (the slots
    // [W][1] lie inside the reservoir, which the load below restores)
    a.dr_k = 1; a.dr_row0 = 0;
    a.probe = probe;
    rc = launch_dispatch(s, a, st);
    if (rc) { cleanup(); return rc; }
    const int64_t n = (int64_t)U * W;
    selftest_trials_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(start, chain, probe, U, W, P, trials);
    CUT(cudaGetLastError());
    rc = lapf_model_chi2(&s->cfg.problem, trials, n, fo, nullptr, chi, st);
    if (rc) { cleanup(); return rc; }
    const unsigned long long init[2] = {0ull, ~0ull};
    CUT(cudaMemcpyAsync(out, init, 16, cudaMemcpyHostToDevice, st));
    selftest_compare_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(probe, chi, n, s->pr, fo, P, out);
    CUT(cudaGetLastError());
    unsigned long long res[2] = {0, 0};
    CUT(cudaMemcpyAsync(res, out, 16, cudaMemcpyDeviceToHost, st));
    rc = lapf_sampler_load(s, blob, (int64_t)blob_bytes, st);      // synchronises the stream: `init` and `res` are settled
    if (rc) { cleanup(); return rc; }
    CUT(cudaStreamSynchronize(st));
    if (const char* path = getenv("LAPF_SELFTEST_DUMP")) {
        // diagnosis of a failing build: [U, W, P] as int64, then probe [U W 3], chi [U W], trials [U W P] as doubles
        // (a probe row whose index is -1 - k: parameter k, the proposal lay outside its prior box and had no pass)
        std::vector<double> hp((size_t)n * 3), hc((size_t)n), ht((size_t)n * P);
        CUT(cudaMemcpy(hp.data(), probe, sizeof(double) * hp.size(), cudaMemcpyDeviceToHost));
        CUT(cudaMemcpy(hc.data(), chi, sizeof(double) * hc.size(), cudaMemcpyDeviceToHost));
        CUT(cudaMemcpy(ht.data(), trials, sizeof(double) * ht.size(), cudaMemcpyDeviceToHost));
        if (FILE* f = fopen(path, "wb")) {
            const int64_t head[3] = {U, W, P};
            fwrite(head, sizeof(int64_t), 3, f);
            fwrite(hp.data(), sizeof(double), hp.size(), f);
            fwrite(hc.data(), sizeof(double), hc.size(), f);
            fwrite(ht.data(), sizeof(double), ht.size(), f);
            fclose(f);
        }
    }
    cleanup();
#undef CUT
    s->launches += 3;
    if (res[0] != 0)
        return fail(LAPF_ERR_SELFTEST,
                    "self-test failed: %llu of %lld trial chi-squares of the batched sampler differ from the stateless "
                    "operator or mark a wrong prior-box skip (first: update %lld of walker %lld).  This build of liblapf.so mis-compiles the sampler "
                    "kernel; rebuild with the CUDA toolkit the tests were run with (see DESIGN.md 10).",
                    res[0], (long long)n, (long long)((res[1] - 1) / W), (long long)((res[1] - 1) % W));
    return LAPF_OK;
}

int lapf_sampler_set_chain_format(lapf_sampler* s, int32_t format) {
    if (!s) return fail(LAPF_ERR_INVALID, "sampler is NULL");
    if (format != LAPF_CHAIN_F64 && format != LAPF_CHAIN_F32_DELTA && !is_event_format(format))
        return fail(LAPF_ERR_INVALID, "unknown chain format %d", format);
    if (is_event_format(format) && s->cfg.thin != 1)
        return fail(LAPF_ERR_INVALID, "event chain formats need thin = 1 (thin is %d): rows further apart differ in more "
                    "than one parameter", s->cfg.thin);
    s->chain_format = format;
    return LAPF_OK;
}

int lapf_sampler_start(lapf_sampler* s, double* start_out, void* stream) {
    if (!s || !start_out) return fail(LAPF_ERR_INVALID, "sampler/start_out is NULL");
    CU(cudaMemcpyAsync(start_out, s->shift, sizeof(double) * (size_t)s->cfg.n_walkers * (s->P + 1), cudaMemcpyDeviceToDevice,
                       (cudaStream_t)stream));
    return LAPF_OK;
}

// Turns on optional device state, all or nothing: frees whatever the parts hold (re-enabling), allocates every
// part, writes its fill (kKeep: `init` fills it), then runs the self-test if asked (unless LAPF_NO_SELFTEST).  On
// any failure every part is freed and nulled again.
extern "C++" {
template <class Init>
static int enable_parts(lapf_sampler* s, std::initializer_list<Part> parts, bool selftest, cudaStream_t st, Init&& init) {
    auto drop = [&]() {
        cudaStreamSynchronize(st);
        for (const Part& p : parts) { cudaFree(*p.dev); *p.dev = nullptr; }
    };
    drop();
    int rc = LAPF_OK;
    for (const Part& p : parts) {
        cudaError_t e = cudaMalloc(p.dev, p.bytes);
        if (e == cudaSuccess && p.fill != kKeep) e = cudaMemsetAsync(*p.dev, p.fill, p.bytes, st);
        if (e != cudaSuccess) {
            rc = fail(LAPF_ERR_CUDA, "allocating %zu bytes of device state failed: %s", p.bytes, cudaGetErrorString(e));
            break;
        }
    }
    if (!rc) rc = init();
    if (!rc && selftest && !getenv("LAPF_NO_SELFTEST")) rc = lapf_sampler_selftest(s, st);
    if (rc) drop();
    return rc;
}
}  // extern "C++"

int lapf_sampler_sketch_enable(lapf_sampler* s, int32_t n_bins, double sep_bin, double pa_bin, const double* centers,
                               void* stream) {
    if (!s) return fail(LAPF_ERR_INVALID, "sampler is NULL");
    if (n_bins < 2 || n_bins > (1 << 20) || (n_bins & 1) || !(sep_bin > 0.0) || !(pa_bin > 0.0))
        return fail(LAPF_ERR_INVALID, "sketch needs an even n_bins in [2, 2^20] and positive bin widths");
    cudaStream_t st = (cudaStream_t)stream;
    const int F = s->cfg.problem.n_frames, nbody = s->cfg.problem.nbody, slots = 2 * (nbody - 1);
    if (s->bm)
        return fail(LAPF_ERR_INVALID, "sketches cannot be enabled after batch means (the batch means would change shape)");
    s->sk_bins = n_bins;
    s->sk_sep_bin = sep_bin;
    s->sk_pa_bin = pa_bin;
    s->sk_auto_center = centers == nullptr;
    const int rc = enable_parts(s, {{(void**)&s->sk_hist, sketch_hist_bytes(s), 0},
                                    {(void**)&s->sk_center, sizeof(double) * (size_t)F * slots, kKeep},
                                    {(void**)&s->sk_mom, sketch_mom_bytes(s), 0}}, false, st, [&]() -> int {
        if (centers) {
            CU(cudaMemcpyAsync(s->sk_center, centers, sizeof(double) * (size_t)F * slots, cudaMemcpyDeviceToDevice, st));
        } else {
            sketch_center_kernel<<<(F * (nbody - 1) + 127) / 128, 128, 0, st>>>(s->shift, s->walker_of, s->frame_start, F,
                                                                              s->P, nbody, s->sk_center);
            CU(cudaGetLastError());
            s->launches++;
        }
        return LAPF_OK;
    });
    if (rc) s->sk_bins = 0;
    return rc;
}

int lapf_sampler_sketch(lapf_sampler* s, uint32_t* hist_out, double* summary_out, void* stream) {
    if (!s) return fail(LAPF_ERR_INVALID, "sampler is NULL");
    if (!s->sk_hist) return fail(LAPF_ERR_INVALID, "sketches are not enabled (lapf_sampler_sketch_enable)");
    cudaStream_t st = (cudaStream_t)stream;
    const int F = s->cfg.problem.n_frames, slots = 2 * (s->cfg.problem.nbody - 1);
    if (hist_out) CU(cudaMemcpyAsync(hist_out, s->sk_hist, sketch_hist_bytes(s), cudaMemcpyDeviceToDevice, st));
    if (summary_out) {
        // rows recorded since the sketches were last zeroed = rows recorded so far (enable before the first run)
        const int64_t n_rows = rows_upto(s->count, s->cfg.burn_in, s->cfg.thin);
        sketch_reduce_kernel<<<F, 32 * slots, 0, st>>>(s->sk_mom, s->sk_center, s->walker_of, s->frame_start, slots, n_rows,
                                                      summary_out);
        CU(cudaGetLastError());
        s->launches++;
    }
    return LAPF_OK;
}

int lapf_sampler_batchmeans_enable(lapf_sampler* s, int32_t batch_rows, int32_t levels, void* stream) {
    if (!s) return fail(LAPF_ERR_INVALID, "sampler is NULL");
    if (batch_rows < 1 || batch_rows > (1 << 30) || levels < 1 || levels > 24)
        return fail(LAPF_ERR_INVALID, "batch means need batch_rows in [1, 2^30] and levels in [1, 24]");
    if (rows_upto(s->count, s->cfg.burn_in, s->cfg.thin) > 0)
        return fail(LAPF_ERR_INVALID, "batch means must be enabled before the first recorded row");
    s->bm_rows = batch_rows;
    s->bm_levels = levels;
    s->bm_c = s->P + 1 + (s->sk_hist ? 2 * (s->cfg.problem.nbody - 1) : 0);
    return enable_parts(s, {{(void**)&s->bm, bm_state_bytes(s), 0}}, true, (cudaStream_t)stream, [] { return LAPF_OK; });
}

int lapf_sampler_batchmeans(lapf_sampler* s, double* walker_out, double* frame_out, void* stream) {
    if (!s) return fail(LAPF_ERR_INVALID, "sampler is NULL");
    if (!s->bm) return fail(LAPF_ERR_INVALID, "batch means are not enabled (lapf_sampler_batchmeans_enable)");
    cudaStream_t st = (cudaStream_t)stream;
    if (walker_out) CU(cudaMemcpyAsync(walker_out, s->bm, bm_state_bytes(s), cudaMemcpyDeviceToDevice, st));
    if (frame_out) {
        const int64_t n_rows = rows_upto(s->count, s->cfg.burn_in, s->cfg.thin);
        batchmeans_reduce_kernel<<<s->cfg.problem.n_frames, 256, 0, st>>>(s->bm, s->moments, s->sk_mom, s->walker_of,
                                                                        s->frame_start, s->P, s->bm_c, s->bm_levels,
                                                                        s->bm_rows, n_rows, frame_out);
        CU(cudaGetLastError());
        s->launches++;
    }
    return LAPF_OK;
}

int lapf_sampler_draws_enable(lapf_sampler* s, int32_t per_walker, void* stream) {
    if (!s) return fail(LAPF_ERR_INVALID, "sampler is NULL");
    if (per_walker < 1 || per_walker > 65536) return fail(LAPF_ERR_INVALID, "draws need per_walker in [1, 65536]");
    if (s->dr_val) return fail(LAPF_ERR_INVALID, "draws are already enabled");
    if (rows_upto(s->count, s->cfg.burn_in, s->cfg.thin) > 0)
        return fail(LAPF_ERR_INVALID, "draws must be enabled before the first recorded row");
    s->dr_k = per_walker;
    const int rc = enable_parts(s, {{(void**)&s->dr_val, draws_val_bytes(s), 0xFF}, {(void**)&s->dr_row, draws_row_bytes(s), 0xFF}},
                                true, (cudaStream_t)stream, [] { return LAPF_OK; });
    if (rc) s->dr_k = 0;
    return rc;
}

int lapf_sampler_draws(lapf_sampler* s, double* values_out, int64_t* rows_out, void* stream) {
    if (!s) return fail(LAPF_ERR_INVALID, "sampler is NULL");
    if (!s->dr_val) return fail(LAPF_ERR_INVALID, "draws are not enabled (lapf_sampler_draws_enable)");
    cudaStream_t st = (cudaStream_t)stream;
    if (values_out) CU(cudaMemcpyAsync(values_out, s->dr_val, draws_val_bytes(s), cudaMemcpyDeviceToDevice, st));
    if (rows_out) CU(cudaMemcpyAsync(rows_out, s->dr_row, draws_row_bytes(s), cudaMemcpyDeviceToDevice, st));
    return LAPF_OK;
}

int lapf_sampler_set_frame_widths(lapf_sampler* s, const double* widths, void* stream) {
    if (!s) return fail(LAPF_ERR_INVALID, "sampler is NULL");
    const int F = s->cfg.problem.n_frames, P = s->P;
    std::vector<double> h((size_t)F * P);
    for (int f = 0; f < F; ++f)
        for (int j = 0; j < P; ++j) {
            const double v = widths ? widths[(size_t)f * P + j] : s->widths[j];
            if (!(v >= 0.0) || !std::isfinite(v))
                return fail(LAPF_ERR_INVALID, "widths[%d][%d] = %g is not a valid jump width", f, j, v);
            h[(size_t)f * P + j] = v;
        }
    cudaStream_t st = (cudaStream_t)stream;
    auto put = [&]() -> int {
        CU(cudaMemcpyAsync(s->fw, h.data(), fw_bytes(s), cudaMemcpyHostToDevice, st));
        CU(cudaStreamSynchronize(st));   // `h` is pageable and lives on this stack frame
        return LAPF_OK;
    };
    if (s->fw) return put();   // later calls replace the widths and keep the snapshot
    return enable_parts(s, {{(void**)&s->fw, fw_bytes(s), kKeep}, {(void**)&s->fw_snap, fw_snap_bytes(s), 0}}, true, st, put);
}

int lapf_sampler_set_priors(lapf_sampler* s, const double* table, void* stream) {
    if (!s || !table) return fail(LAPF_ERR_INVALID, "sampler/table is NULL");
    const int F = s->cfg.problem.n_frames, P = s->P;
    const size_t n = (size_t)F * P * 4;
    std::vector<double> h(2 * n);                        // {lo, hi, mu, h} for the kernels, then the table as given
    for (int f = 0; f < F; ++f)
        for (int j = 0; j < P; ++j) {
            const double* e = table + ((size_t)f * P + j) * 4;
            const double lo = e[0], hi = e[1], mu = e[2], sg = e[3];
            if (lo != lo || hi != hi || mu != mu || sg != sg)
                return fail(LAPF_ERR_INVALID, "prior of frame %d, parameter %d has a nan entry", f, j);
            if (lo > hi) return fail(LAPF_ERR_INVALID, "prior of frame %d, parameter %d: lo %g > hi %g", f, j, lo, hi);
            if (!(sg > 0.0)) return fail(LAPF_ERR_INVALID, "prior of frame %d, parameter %d: sigma %g <= 0", f, j, sg);
            if (std::isfinite(sg) && !std::isfinite(mu))
                return fail(LAPF_ERR_INVALID, "prior of frame %d, parameter %d: mu %g is not finite and sigma %g is", f, j,
                            mu, sg);
            const double hh = std::isinf(sg) ? 0.0 : 0.5 / (sg * sg);
            if (!std::isfinite(hh))
                return fail(LAPF_ERR_INVALID, "prior of frame %d, parameter %d: sigma %g is too small", f, j, sg);
            double* d = h.data() + ((size_t)f * P + j) * 4;
            d[0] = lo; d[1] = hi; d[2] = mu; d[3] = hh;
            memcpy(h.data() + n + ((size_t)f * P + j) * 4, e, 4 * sizeof(double));
        }
    cudaStream_t st = (cudaStream_t)stream;
    double* tmp = nullptr;
    CU(cudaMallocAsync((void**)&tmp, 2 * prior_bytes(s), st));
    cudaError_t e = cudaMemcpyAsync(tmp, h.data(), 2 * prior_bytes(s), cudaMemcpyHostToDevice, st);
    int rc = e == cudaSuccess ? prior_check(s, s->state, P + 1, tmp, "priors refused", st)   // synchronises: `h` is settled
                              : fail(LAPF_ERR_CUDA, "copy of the priors failed: %s", cudaGetErrorString(e));
    auto put = [&]() -> int {
        CU(cudaMemcpyAsync(s->pr, tmp, prior_bytes(s), cudaMemcpyDeviceToDevice, st));
        CU(cudaMemcpyAsync(s->pr_given, tmp + n, prior_bytes(s), cudaMemcpyDeviceToDevice, st));
        return LAPF_OK;
    };
    if (!rc) rc = s->pr ? put()             // later calls replace the table
                        : enable_parts(s, {{(void**)&s->pr, prior_bytes(s), kKeep}, {(void**)&s->pr_given, prior_bytes(s), kKeep}},
                                       true, st, put);
    cudaFreeAsync(tmp, st);
    return rc;
}

int lapf_sampler_priors(lapf_sampler* s, double* out, void* stream) {
    if (!s || !out) return fail(LAPF_ERR_INVALID, "sampler/out is NULL");
    if (!s->pr) return fail(LAPF_ERR_INVALID, "priors are not on (lapf_sampler_set_priors)");
    CU(cudaMemcpyAsync(out, s->pr_given, prior_bytes(s), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return LAPF_OK;
}

int lapf_sampler_frame_widths(lapf_sampler* s, double* out, void* stream) {
    if (!s || !out) return fail(LAPF_ERR_INVALID, "sampler/out is NULL");
    if (!s->fw) return fail(LAPF_ERR_INVALID, "per-frame widths are not on (lapf_sampler_set_frame_widths)");
    CU(cudaMemcpyAsync(out, s->fw, fw_bytes(s), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return LAPF_OK;
}

int lapf_sampler_frame_counts(lapf_sampler* s, int64_t* out, void* stream) {
    if (!s || !out) return fail(LAPF_ERR_INVALID, "sampler/out is NULL");
    frame_counts_kernel<<<s->cfg.problem.n_frames, 32 * s->P, 0, (cudaStream_t)stream>>>(
        s->tries, s->accepts, s->walker_of, s->frame_start, s->P, (long long*)out);
    CU(cudaGetLastError());
    s->launches++;
    return LAPF_OK;
}

int lapf_sampler_adapt_widths(lapf_sampler* s, const int64_t* counts, double target, void* stream) {
    if (!s || !counts) return fail(LAPF_ERR_INVALID, "sampler/counts is NULL");
    if (!s->fw) return fail(LAPF_ERR_INVALID, "per-frame widths are not on (lapf_sampler_set_frame_widths)");
    if (!(target > 0.0 && target < 1.0)) return fail(LAPF_ERR_INVALID, "target acceptance %g is not in (0, 1)", target);
    const int n = s->cfg.problem.n_frames * s->P;
    adapt_widths_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>((const long long*)counts, s->fw_snap, s->fw, n,
                                                                           target);
    CU(cudaGetLastError());
    s->launches++;
    return LAPF_OK;
}

int lapf_frame_outside(const float* frames, int32_t n_frames, int32_t fy, int32_t fx, const int32_t* cut, int32_t ny,
                       int32_t nx, double satlevel, double readnoise, double* outside_out, void* stream) {
    if (!frames || !cut || !outside_out || n_frames <= 0 || fy <= 0 || fx <= 0 || ny <= 0 || nx <= 0)
        return fail(LAPF_ERR_INVALID, "bad arguments to lapf_frame_outside");
    int rc = require_device();
    if (rc) return rc;
    keep_pool_memory();
    cudaStream_t st = (cudaStream_t)stream;
    const int rows_per_tile = 16, tiles = (fy + rows_per_tile - 1) / rows_per_tile;
    if (n_frames > 65535) return fail(LAPF_ERR_INVALID, "lapf_frame_outside handles at most 65535 frames per call");
    double* partial = nullptr;
    CU(cudaMallocAsync((void**)&partial, sizeof(double) * (size_t)n_frames * tiles * 3, st));
    outside_partial_kernel<<<dim3((unsigned)tiles, (unsigned)n_frames), 256, 0, st>>>(
        frames, fy, fx, cut, ny, nx, 0.8 * satlevel, readnoise * readnoise, rows_per_tile, partial);
    CU(cudaGetLastError());
    outside_reduce_kernel<<<(3 * n_frames + 127) / 128, 128, 0, st>>>(partial, n_frames, tiles, outside_out);
    CU(cudaGetLastError());
    CU(cudaFreeAsync(partial, st));
    return LAPF_OK;
}

int lapf_chain_drain(const void* device_src, void* pinned_dst, size_t nbytes, void* compute_stream, void* copy_stream) {
    if (!device_src || !pinned_dst) return fail(LAPF_ERR_INVALID, "NULL buffer");
    cudaEvent_t ev;
    CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    cudaError_t e = cudaEventRecord(ev, (cudaStream_t)compute_stream);
    if (e == cudaSuccess) e = cudaStreamWaitEvent((cudaStream_t)copy_stream, ev, 0);
    if (e == cudaSuccess) e = cudaMemcpyAsync(pinned_dst, device_src, nbytes, cudaMemcpyDeviceToHost, (cudaStream_t)copy_stream);
    cudaEventDestroy(ev);
    if (e != cudaSuccess) return fail(LAPF_ERR_CUDA, "chain drain failed: %s", cudaGetErrorString(e));
    return LAPF_OK;
}

int lapf_write_chain_csv(const char* path, const double* rows, int64_t n_rows, int32_t n_cols, int64_t row_stride,
                         int32_t flags) {
    const bool leading_nan_row = (flags & LAPF_CSV_LEADING_NAN_ROW) != 0;
    const bool append = (flags & LAPF_CSV_APPEND) != 0;
    if (!path || (!rows && n_rows > 0) || n_cols <= 0 || n_rows < 0)
        return fail(LAPF_ERR_INVALID, "bad arguments to lapf_write_chain_csv");
    FILE* fp = fopen(path, append ? "ab" : "wb");
    if (!fp) return fail(LAPF_ERR_INVALID, "cannot open %s for writing", path);
    std::string buf;
    buf.reserve(1 << 20);
    auto put = [&](double v) {
        if (std::isnan(v)) { buf += "nan"; return; }
        if (std::isinf(v)) { buf += v > 0 ? "inf" : "-inf"; return; }
        char tmp[40];
        auto r = std::to_chars(tmp, tmp + sizeof(tmp), v);   // shortest round-trip, like repr(float)
        buf.append(tmp, r.ptr);
    };
    if (leading_nan_row) {   // the seed column of apf_step2.py:278-279
        for (int c = 0; c < n_cols; ++c) { if (c) buf += ','; buf += "nan"; }
        buf += "\r\n";
    }
    bool ok = true;
    for (int64_t r = 0; r < n_rows && ok; ++r) {
        const double* row = rows + r * row_stride;
        for (int c = 0; c < n_cols; ++c) { if (c) buf += ','; put(row[c]); }
        buf += "\r\n";   // csv.writer default line terminator
        if (buf.size() > (1 << 20) - 1024) {
            ok = fwrite(buf.data(), 1, buf.size(), fp) == buf.size();
            buf.clear();
        }
    }
    if (ok && !buf.empty()) ok = fwrite(buf.data(), 1, buf.size(), fp) == buf.size();
    ok = (fclose(fp) == 0) && ok;
    return ok ? LAPF_OK : fail(LAPF_ERR_INVALID, "short write to %s", path);
}

// cuTensorMapEncodeTiled through the runtime's driver entry-point lookup (no link against libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
        cudaGetLastError();
    }
    return fn;
}

int lapf_frame_prep(const float* frames, int32_t n_frames, int32_t fy, int32_t fx, const int32_t* origin,
                    int32_t ny, int32_t nx, double satlevel, double readnoise, float* data_out,
                    float* weight_out, void* stream) {
    if (!frames || !origin || !data_out || !weight_out || n_frames <= 0 || fy <= 0 || fx <= 0 || ny <= 0 || nx <= 0)
        return fail(LAPF_ERR_INVALID, "bad arguments to lapf_frame_prep");
    int rc = require_device();
    if (rc) return rc;
    // Cut-outs through the TMA unit when a tensor map can describe the frames (rows 16-byte aligned, a box
    // of at most 256 pixels a side, at most 65535 frames per launch); the plain kernel otherwise (and with
    // LAPF_NO_TMA_PREP set).  Same arithmetic, same bits.
    EncodeTiledFn enc = getenv("LAPF_NO_TMA_PREP") ? nullptr : encode_tiled();
    if (enc && fx % 4 == 0 && nx % 4 == 0 && nx + 4 <= 256 && ((uintptr_t)frames & 15) == 0 && n_frames <= 65535 &&
        (size_t)kPrepRows * (nx + 4) * sizeof(float) <= 48 * 1024) {
        alignas(64) CUtensorMap tmap;
        const cuuint64_t dims[3] = {(cuuint64_t)fx, (cuuint64_t)fy, (cuuint64_t)n_frames};
        const cuuint64_t strides[2] = {(cuuint64_t)fx * sizeof(float), (cuuint64_t)fx * fy * sizeof(float)};
        const cuuint32_t box[3] = {(cuuint32_t)(nx + 4), (cuuint32_t)kPrepRows, 1u};
        const cuuint32_t estr[3] = {1u, 1u, 1u};
        if (enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(frames), dims, strides, box, estr,
                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS) {
            const dim3 grid((unsigned)((ny + kPrepRows - 1) / kPrepRows), (unsigned)n_frames);
            frame_prep_tma_kernel<<<grid, 256, (size_t)kPrepRows * (nx + 4) * sizeof(float), (cudaStream_t)stream>>>(
                tmap, fy, fx, origin, ny, nx, 0.8 * satlevel, readnoise * readnoise, data_out, weight_out);
            CU(cudaGetLastError());
            return LAPF_OK;
        }
    }
    const int64_t n = (int64_t)n_frames * ny * nx;
    frame_prep_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        frames, n_frames, fy, fx, origin, ny, nx, 0.8 * satlevel, readnoise * readnoise, data_out, weight_out);
    CU(cudaGetLastError());
    return LAPF_OK;
}

int lapf_philox_draws(uint64_t seed, uint64_t walker_id, uint64_t first_update, int32_t n, int32_t nparam,
                      int32_t* index_out, double* normal_out, double* log_uniform_out, void* stream) {
    if (n < 0 || nparam <= 0 || !index_out || !normal_out || !log_uniform_out)
        return fail(LAPF_ERR_INVALID, "bad arguments to lapf_philox_draws");
    if (n == 0) return LAPF_OK;
    int rc = require_device();
    if (rc) return rc;
    philox_draws_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(seed, walker_id, first_update, n, nparam,
                                                                          index_out, normal_out, log_uniform_out);
    CU(cudaGetLastError());
    return LAPF_OK;
}

int lapf_measure_peaks(double* out4) {
    if (!out4) return fail(LAPF_ERR_INVALID, "out is NULL");
    int rc = require_device();
    if (rc) return rc;
    int dev = 0, sms = 0, khz = 0;
    CU(cudaGetDevice(&dev));
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    CU(cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, dev));
    float* d = nullptr;
    CU(cudaMalloc((void**)&d, 64));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    const int blocks = sms * 8, threads = 256, iters = 4096;
    const double ops = (double)blocks * threads * (double)iters * 64.0;
    float ms = 0.f;
    double best[2] = {0, 0};
    for (int which = 0; which < 2; ++which) {
        for (int rep = 0; rep < 4; ++rep) {   // first repetition is the warm-up
            CU(cudaEventRecord(e0));
            if (which == 0) peak_ex2_kernel<<<blocks, threads>>>(d, iters);
            else peak_ffma_kernel<<<blocks, threads>>>(d, iters, 0.999f, 0.001f);
            CU(cudaEventRecord(e1));
            CU(cudaEventSynchronize(e1));
            CU(cudaGetLastError());
            CU(cudaEventElapsedTime(&ms, e0, e1));
            if (rep > 0) best[which] = std::max(best[which], ops / (ms * 1e-3));
        }
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d);
    out4[0] = best[0];
    out4[1] = best[1];
    out4[2] = khz / 1000.0;
    out4[3] = sms;
    return LAPF_OK;
}

}  // extern "C"
