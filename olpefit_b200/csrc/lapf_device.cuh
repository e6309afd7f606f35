// Device-side building blocks of the LAPF step-2 hot path for sm_100a.
//
//   Layout<NB>      parameter-vector index map (apf_step2.py:108; 3body/apf_step2_3body.py:266-288)
//   Coef<NB>        per-proposal coefficients of the K = 2*NB elliptical Gaussians, culling
//                   segments, safe-range flag; CoefImg its shared-memory image
//   warp_chi2<>     fused model / residual / square / reduce over one stamp by ONE warp
//                   (replaces build_analytical_model + chi_squared, apf_step2.py:78-137):
//                   block table + column table -> factorised loop (row_steps_fast: one exponential
//                   per 2x4-pixel block and component) or plain loop (row_steps: one per pixel)
//   tmem_*          tensor memory as a per-lane pixel store (tcgen05.alloc / st / ld)
//   philox / draws  counter-based random stream (replaces numpy's global MT, apf_step2.py:64,68,143,302)
//
// Numerics (SURVEY.md appendix D): pixel terms in FP32 with stamp-local coordinates, ex2.approx
// with coefficients pre-scaled by -log2(e); FP32 partial sums of a few rows are folded into an FP64
// accumulator; everything that crosses lanes, the stored chi-square and the Metropolis
// difference are FP64.  The pixel->lane map and the reduction tree are fixed, so chi-square is
// a pure function of the parameter vector.
#pragma once
#ifndef LAPF_LOOP_UNROLL
#define LAPF_LOOP_UNROLL 2   /* row steps per trip of the factorised loop (measured: 2 is 2 % faster than 1 or 4) */
#endif
#include <cstdint>
#include <cuda_runtime.h>

namespace lapf {

constexpr float kLog2e = 1.4426950408889634f;
constexpr int kLoopUnroll = LAPF_LOOP_UNROLL;
constexpr unsigned kFull = 0xffffffffu;

template <int NB>
struct Layout {
    static constexpr int NOBJ = NB;
    static constexpr int P = 3 * NB + 10;   // 16 / 19
    static constexpr int K = 2 * NB;        // Gaussian components: (narrow, wide) per object
    static constexpr int I_DX = 2 * NB, I_DY = 2 * NB + 1;
    static constexpr int I_AMP = 2 * NB + 2;
    static constexpr int I_RATIO = 3 * NB + 2, I_BKGD = 3 * NB + 3;
    static constexpr int I_SX = 3 * NB + 4, I_SY = 3 * NB + 5, I_SX2 = 3 * NB + 6, I_SY2 = 3 * NB + 7;
    static constexpr int I_TH = 3 * NB + 8, I_TH2 = 3 * NB + 9;
};

// ---------------------------------------------------------------------------------------------
// PTX helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));   // one MUFU.EX2
    return y;
}

__device__ __forceinline__ double shfl_f64(double v, int src) {
    int lo = __double2loint(v), hi = __double2hiint(v);
    lo = __shfl_sync(kFull, lo, src);
    hi = __shfl_sync(kFull, hi, src);
    return __hiloint2double(hi, lo);
}

__device__ __forceinline__ double shfl_xor_f64(double v, int mask) {
    int lo = __double2loint(v), hi = __double2hiint(v);
    lo = __shfl_xor_sync(kFull, lo, mask);
    hi = __shfl_xor_sync(kFull, hi, mask);
    return __hiloint2double(hi, lo);
}

__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) v += shfl_xor_f64(v, off);
    return v;   // identical in every lane: xor-butterfly adds the same pairs everywhere
}

// warp_sum_f64 of the lane values (double)p[0..31], worked out by ONE thread from the 32 values in
// shared memory (16-byte aligned).  Lane 0 of the butterfly adds p[0] + p[16], then the partner
// 8, 4, 2, 1 lanes away; this is that tree, operand for operand, so the result is bit-identical.
__device__ __forceinline__ double warp_sum_f64_of(const float* __restrict__ p) {
    double v[16];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float4 a = reinterpret_cast<const float4*>(p)[q], b = reinterpret_cast<const float4*>(p)[q + 4];
        v[4 * q] = (double)a.x + (double)b.x; v[4 * q + 1] = (double)a.y + (double)b.y;
        v[4 * q + 2] = (double)a.z + (double)b.z; v[4 * q + 3] = (double)a.w + (double)b.w;
    }
#pragma unroll
    for (int off = 8; off >= 1; off >>= 1)
#pragma unroll
        for (int l = 0; l < off; ++l) v[l] += v[l + off];
    return v[0];
}

// mbarrier + 1-D TMA bulk copy (global -> shared), used to stage a stamp once per frame.
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes,
                                             uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// Tensor memory (TMEM) as a per-lane, read-only pixel store.  The sampler never uses the tensor
// cores, so their 256 KB of TMEM per SM are free: every lane keeps ITS pixels of the staged stamp
// (prepared data and weight of the 8 columns x NY/RG rows it always works on) in the TMEM lane it
// is allowed to read -- lane 32 (warp % 4) + lane id, shape .32x32b -- and fetches the 16 values
// of a row step with one tcgen05.ld instead of four LDS.128.  That takes 2 KB per warp and row
// step off the shared-memory pipe, which the factorised loop would otherwise saturate.
__device__ __forceinline__ void tmem_alloc(uint32_t* slot_in_smem, uint32_t ncols) {   // one warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_in_smem)), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t base, uint32_t ncols) {          // the same warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void tmem_st16(uint32_t addr, const float (&v)[16]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
                 ::"r"(addr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
                   "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
                   "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])), "r"(__float_as_uint(v[8])),
                   "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
                   "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])),
                   "r"(__float_as_uint(v[15]))
                 : "memory");
}
// issue the load of 16 consecutive columns; the registers are valid only after tmem_ld16_wait
__device__ __forceinline__ void tmem_ld16_issue(uint32_t addr, uint32_t (&r)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(addr));
}
__device__ __forceinline__ void tmem_st8(uint32_t addr, const float (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 ::"r"(addr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
                   "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
                   "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
                 : "memory");
}
__device__ __forceinline__ void tmem_ld8_issue(uint32_t addr, uint32_t (&r)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(addr));
}
__device__ __forceinline__ void tmem_ld8_wait(uint32_t (&r)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]));
}
// the operands tie every later use of the registers to the wait
__device__ __forceinline__ void tmem_ld16_wait(uint32_t (&r)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                   "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]));
}

// ---------------------------------------------------------------------------------------------
// Coefficients
// ---------------------------------------------------------------------------------------------
template <int NB>
struct Coef {
    static constexpr int K = 2 * NB;
    float x0[K], y0[K], amp[K];   // component 2o = narrow core of object o, 2o+1 = its wide wing
    float sa[2], sb[2], sc[2];    // shape 0 = narrow, 1 = wide; a, b, c of A.1 times -log2(e)
    float floor;
    // far-field culling (set_cull -> set_segments): per column panel the row steps
    //   [0, seg0) floor only, [seg0, seg1) wide wings, [seg1, seg2) all, [seg2, seg3) wings, rest floor only
    // and the component evaluations (pixels x components) they add up to
    int seg[2][4];
    unsigned nexp;
    // the factorised pixel loop (row_steps_fast) is safe for this vector (set_fast)
    bool fast;
};

// a, b, c of astropy Gaussian2D.evaluate (SURVEY appendix A.1), pre-scaled so that the
// exponential is a bare ex2:  G = A * 2^(sa*dx^2 + sb*dx*dy + sc*dy^2).
//
// Coefficients, the safe-range test and the culling bounds are inlined into several kernels (the
// stateless operator, the team sampler, the batched sampler), whose chi-squares must agree bit for
// bit.  Plain `a * b + c` leaves it to the compiler whether to contract into an FMA, and it decides
// per inlined copy (a build of the two-vectors-per-pass operator contracted `a - a * ratio` in one
// kernel only: 1.5 % of the trial chi-squares differed in the last bits).  So every sum of products
// here is spelled with rounding intrinsics, which are never contracted.
template <int NB>
__device__ __forceinline__ void set_shape_sc(Coef<NB>& cf, int which, float sx, float sy, float s, float c) {
    const float ivx = __fdiv_rn(1.0f, __fmul_rn(sx, sx)), ivy = __fdiv_rn(1.0f, __fmul_rn(sy, sy));
    const float cc = __fmul_rn(c, c), ss = __fmul_rn(s, s);
    cf.sa[which] = __fmul_rn(-0.5f * kLog2e, __fmaf_rn(cc, ivx, __fmul_rn(ss, ivy)));
    cf.sb[which] = __fmul_rn(__fmul_rn(-kLog2e, __fmul_rn(s, c)), __fsub_rn(ivx, ivy));     // sin(2t)/2 = s*c
    cf.sc[which] = __fmul_rn(-0.5f * kLog2e, __fmaf_rn(ss, ivx, __fmul_rn(cc, ivy)));
}

template <int NB>
__device__ __forceinline__ void set_shape(Coef<NB>& cf, int which, float sx, float sy, float th) {
    float s, c;
    sincosf(th, &s, &c);
    set_shape_sc<NB>(cf, which, sx, sy, s, c);
}

// Per-warp staging of one (trial) parameter vector as FP32 in shared memory.  Lane j < P holds
// parameter j in FP64 frame coordinates; positions are converted to stamp-local coordinates in
// FP64 before rounding to FP32 (SURVEY appendix D.1).  Layout of tf[]:
//   tf[j], j < P            parameter j (positions: local)
//   tf[P + j], j < 2*NB     centre coordinate j of the WIDE component: position j + dx or dy
// Every conversion is done once, by the owning lane; afterwards all lanes read tf[] as broadcasts.
template <int NB>
__device__ __forceinline__ void stage_trial(float* tf, int lane, double mine, double oxd, double oyd) {
    using L = Layout<NB>;
    const double dxv = shfl_f64(mine, L::I_DX), dyv = shfl_f64(mine, L::I_DY);
    __syncwarp();   // readers of the previous vector are done
    if (lane < 2 * NB) {
        const double base = mine - ((lane & 1) ? oyd : oxd);
        tf[lane] = (float)base;
        tf[L::P + lane] = (float)(base + ((lane & 1) ? dyv : dxv));
    } else if (lane < L::P) {
        tf[lane] = (float)mine;
    }
    __syncwarp();
}

// Centres and amplitudes from the staged vector (build_2d_gaussian, apf_step2.py:95-101).
template <int NB>
__device__ __forceinline__ void load_centres_amps(Coef<NB>& cf, const float* tf) {
    using L = Layout<NB>;
    const float ratio = tf[L::I_RATIO], bkgd = tf[L::I_BKGD];
#pragma unroll
    for (int o = 0; o < NB; ++o) {
        cf.x0[2 * o] = tf[2 * o];
        cf.y0[2 * o] = tf[2 * o + 1];
        cf.x0[2 * o + 1] = tf[L::P + 2 * o];
        cf.y0[2 * o + 1] = tf[L::P + 2 * o + 1];
        const float a = __fsub_rn(tf[L::I_AMP + o], bkgd);   // :95
        const float aw = __fmul_rn(a, ratio);                // :96
        cf.amp[2 * o] = __fsub_rn(a, aw);                    // :97 (two roundings, never an FMA: see set_shape_sc)
        cf.amp[2 * o + 1] = aw;
    }
}
// the floor of the model is parameter floor_index of the staged vector (apf_step2.py:119-120)

template <int NB>
__device__ __forceinline__ void load_shape(Coef<NB>& cf, int which, const float* tf) {
    using L = Layout<NB>;
    if (which)
        set_shape<NB>(cf, 1, tf[L::I_SX2], tf[L::I_SY2], tf[L::I_TH2]);
    else
        set_shape<NB>(cf, 0, tf[L::I_SX], tf[L::I_SY], tf[L::I_TH]);
}

// Shared-memory image of a Coef: 16-byte slots, an ODD number of them per walker, so that both the
// one-walker-per-lane accesses of the batched sampler and its broadcast reads are conflict-free
// 128-bit transactions.  At least 32 floats: once its pass has read it, the batched sampler reuses a
// walker's image for the pass's 32 lane partials of chi-square.
template <int NB, int PANELS>
struct CoefImg {
    static constexpr int K = 2 * NB;
    static constexpr int WORDS = 3 * K + 7 + 4 * PANELS + 3;   // x0 y0 amp | sa sb sc floor | segments | nexp fast slot
    static constexpr int V4 = ((WORDS + 3) / 4 > 8 ? (WORDS + 3) / 4 : 8) | 1;
    static constexpr int STRIDE = 4 * V4;             // floats per walker
};

// `slot`: which of the resident stamps (TMEM pixel-store slots of the batched sampler) the vector is evaluated on
template <int NB, int PANELS>
__device__ __forceinline__ void store_coef(float* __restrict__ dst, const Coef<NB>& cf, int slot = 0) {
    constexpr int K = 2 * NB;
    using I = CoefImg<NB, PANELS>;
    float v[I::STRIDE];
#pragma unroll
    for (int i = 0; i < I::STRIDE; ++i) v[i] = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) { v[k] = cf.x0[k]; v[K + k] = cf.y0[k]; v[2 * K + k] = cf.amp[k]; }
#pragma unroll
    for (int c = 0; c < 2; ++c) { v[3 * K + c] = cf.sa[c]; v[3 * K + 2 + c] = cf.sb[c]; v[3 * K + 4 + c] = cf.sc[c]; }
    v[3 * K + 6] = cf.floor;
#pragma unroll
    for (int p = 0; p < PANELS; ++p)
#pragma unroll
        for (int q = 0; q < 4; ++q) v[3 * K + 7 + 4 * p + q] = __int_as_float(cf.seg[p][q]);
    v[3 * K + 7 + 4 * PANELS] = __uint_as_float(cf.nexp);
    v[3 * K + 8 + 4 * PANELS] = __int_as_float(cf.fast ? 1 : 0);
    v[3 * K + 9 + 4 * PANELS] = __int_as_float(slot);
#pragma unroll
    for (int q = 0; q < I::V4; ++q)
        reinterpret_cast<float4*>(dst)[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
}

template <int NB, int PANELS>
__device__ __forceinline__ void load_coef(Coef<NB>& cf, const float* __restrict__ src, int* slot = nullptr) {
    constexpr int K = 2 * NB;
    using I = CoefImg<NB, PANELS>;
    float v[I::STRIDE];
#pragma unroll
    for (int q = 0; q < I::V4; ++q) {
        const float4 t = reinterpret_cast<const float4*>(src)[q];
        v[4 * q] = t.x; v[4 * q + 1] = t.y; v[4 * q + 2] = t.z; v[4 * q + 3] = t.w;
    }
#pragma unroll
    for (int k = 0; k < K; ++k) { cf.x0[k] = v[k]; cf.y0[k] = v[K + k]; cf.amp[k] = v[2 * K + k]; }
#pragma unroll
    for (int c = 0; c < 2; ++c) { cf.sa[c] = v[3 * K + c]; cf.sb[c] = v[3 * K + 2 + c]; cf.sc[c] = v[3 * K + 4 + c]; }
    cf.floor = v[3 * K + 6];
#pragma unroll
    for (int p = 0; p < PANELS; ++p)
#pragma unroll
        for (int q = 0; q < 4; ++q) cf.seg[p][q] = __float_as_int(v[3 * K + 7 + 4 * p + q]);
    cf.nexp = __float_as_uint(v[3 * K + 7 + 4 * PANELS]);
    cf.fast = __float_as_int(v[3 * K + 8 + 4 * PANELS]) != 0;
    if (slot) *slot = __float_as_int(v[3 * K + 9 + 4 * PANELS]);
}

// Coefficients of a parameter vector given in FP64 frame coordinates, by ONE thread: the same
// conversions as stage_trial + load_centres_amps + load_shape, so the numbers are the ones the
// cooperative path produces.  v[] must be indexed with constants only (registers).
template <int NB>
__device__ __forceinline__ void coef_from_vector(Coef<NB>& cf, const double (&v)[Layout<NB>::P], double floor_v,
                                                 double oxd, double oyd) {
    using L = Layout<NB>;
    float tf[L::P + 2 * NB];
#pragma unroll
    for (int j = 0; j < L::P; ++j) {
        if (j < 2 * NB) {
            const double base = v[j] - ((j & 1) ? oyd : oxd);
            tf[j] = (float)base;
            tf[L::P + j] = (float)(base + ((j & 1) ? v[L::I_DY] : v[L::I_DX]));
        } else {
            tf[j] = (float)v[j];
        }
    }
    load_centres_amps<NB>(cf, tf);
    cf.floor = (float)floor_v;
    set_shape<NB>(cf, 0, tf[L::I_SX], tf[L::I_SY], tf[L::I_TH]);
    set_shape<NB>(cf, 1, tf[L::I_SX2], tf[L::I_SY2], tf[L::I_TH2]);
}

// ---------------------------------------------------------------------------------------------
// The pixel loop: one warp evaluates chi-square of one parameter vector over an NY x NX stamp.
//
// Lane geometry.  Columns are processed in panels of PW = min(NX, 64).  A WARP STEP covers RG rows
// of a panel (4 rows x 64 columns, or 8 rows x 32 columns): lane (b, a) owns the 2 x 4 pixel BLOCK
// of rows 2b, 2b+1 of the step and columns 4a .. 4a+3 of the panel -- 8 pixels, two 128-bit loads
// per plane (16 lanes read 256 contiguous bytes of a row: conflict-free).  The column offsets of a
// lane never change, so everything that depends on them lives in registers for the whole panel.
// ---------------------------------------------------------------------------------------------
// WPP = 2 (32-pixel stamps, whole-warp passes): TWO parameter vectors per pass, one per half warp.  A
// 32-pixel row needs only 8 column anchors, so a half warp (8 anchors x 2 block rows, 4 rows per
// warp step, 8 steps) covers the stamp, and everything a pass does once -- coefficient load, block
// table (which leaves 16 lanes idle otherwise), reduction, loop control -- serves two walkers.
template <int NX, int WPP = 1>
struct Geo {
    static constexpr int PW = NX >= 64 ? 64 : 32;
    static constexpr int PANELS = NX / PW;
    static constexpr int GPR = PW / 4;        // 4-pixel column groups across a panel: 16 / 8
    static constexpr int LPW = 32 / WPP;      // lanes that work on one parameter vector
    static constexpr int BPS = LPW / GPR;     // 2-row blocks per warp step: 2 / 4 (2 with two vectors per pass)
    static constexpr int RG = 2 * BPS;        // rows per warp step: 4 / 8 (4)
    static_assert(NX % PW == 0 && (NX == 32 || NX % 64 == 0), "unsupported stamp width");
    static_assert(WPP == 1 || (WPP == 2 && NX == 32), "two vectors per pass: 32-pixel stamps only");
};

// Block table: everything that depends on the rows only, computed ONCE per proposal by the warp
// (one 2-row block per lane) instead of once per step by every lane.  One entry of Tab::RS floats
// per block, with yb the centre of its two rows and dyb_k = yb - y0_k:
//   [4q .. 4q + 3]            sb dyb_ka, sb dyb_kb, sc dyb_ka^2, sc dyb_kb^2   piece q < NB: the components
//                             ka = Tab::ka(q), kb = Tab::kb(q), each with the sb, sc of its own class
//   [2K + 8c .. 2K + 8c + 7]  T_c,ij = 2^(j (sb dyb_c + i sb) + 2 i sc dyb_c + sc / 4)   shape class c,
//                             i = -1/2 then +1/2 (row), j = -3/2, -1/2, 1/2, 3/2 (column)
// The first terms give the exponent of component k at the centre of a lane's block,
//   q0 = fma(dxa, fma(sa, dxa, sb*dyb), sc*dyb^2),        dxa = anchor column - x0_k;
// T moves it to the 8 pixels of the block (see row_steps_fast).  Pieces 0 and 1 are the two objects'
// components of class 0 and of class 1: they share sa, so one packed FMA pair (fma.rn.f32x2, rounded
// per element like fma.rn.f32) works out both exponents.  y0_c is the centre of the class's
// FIRST component; the other components of the class fold their offset into the lane constants.
// The entry is padded to 28 floats so the blocks of a warp step read distinct banks.
template <int NB>
struct Tab {
    static constexpr int K = 2 * NB;
    static constexpr int RS = 28;
    static constexpr int OFF_T = 2 * K;
    static_assert(NB == 2 || NB == 3, "pieces 0, 1: class 0, 1 of objects 0 and 1; piece 2: object 2");
    static_assert(OFF_T + 16 <= RS && OFF_T % 4 == 0, "block table entry layout");
    __host__ __device__ static constexpr int ka(int q) { return q < 2 ? q : 4; }
    __host__ __device__ static constexpr int kb(int q) { return q < 2 ? q + 2 : 5; }
};

// A table covers TR rows of the stamp; taller stamps are walked table by table ("half").  A team
// member (TEAM warps share one walker, warp tw takes every TEAM-th warp step) only builds the
// blocks of the steps it evaluates.
template <int NY, int TEAM = 1>
struct Rows {
    static constexpr int TR = NY < 64 ? NY : 64;       // rows per table
    static constexpr int HALVES = NY / TR;
    static constexpr int NBLK = TR / 2 / TEAM;         // blocks a warp builds
    static_assert(NY % TR == 0 && (TR / 2) % TEAM == 0, "unsupported stamp height");
};

// per-warp shared-memory scratch of the pixel loop: the block table, then the column table
// (coop_consts: [component][row of the block][anchor][4 column offsets])
template <int NB, int NX, int NY, int TEAM = 1, int WPP = 1>
struct Scratch {
    // block table of one vector (two vectors per pass: 8 floats apart in the banks, so the four blocks
    // a warp step reads -- 2 block rows x 2 vectors -- are one conflict-free wavefront)
    // (a team member's table: its share of the blocks of ONE panel over the whole height, see team_chi2)
    static constexpr int TEAM_NBLK = NY * Geo<NX>::PANELS / (2 * TEAM);
    static constexpr int TAB1 = (TEAM > 1 ? TEAM_NBLK : Rows<NY, TEAM>::NBLK) * Tab<NB>::RS + (WPP > 1 ? 8 : 0);
    static constexpr int TAB = WPP * TAB1;
    static constexpr int CT = 2 * NB * 2 * Geo<NX>::GPR * 4;      // column table of one panel and vector
    static constexpr int FLOATS = TAB + WPP * CT;                  // one warp on its own (TEAM = 1)
    // a team: every member's block table, then ONE column table for all panels, worked out by the team together
    static constexpr int TEAM_FLOATS = TEAM * TAB + Geo<NX>::PANELS * CT;
};

// A block's entry is 2 + K/2 independent 16-byte pieces (K/2 anchor pieces, 4 (class, row)
// factor quadruples).  Team members, whose tables have 8 blocks or fewer, spread the pieces of a
// block over 4 lanes, with the same instruction stream in every lane (the piece is picked with
// selects): a quarter of the instructions and of the serialised MUFUs on the latency path of an
// update.  (Whole-warp passes keep one block per lane: on 32-pixel stamps, the only case with lanes
// to spare, the split was not faster.)
template <int NB, int NX, int TR, int TEAM, int WPP = 1>
__device__ __forceinline__ void build_row_table(float* __restrict__ rt, const Coef<NB>& cf, int lane, int row0, int tw) {
    using G = Geo<NX, WPP>;
    using T = Tab<NB>;
    constexpr int K = 2 * NB;
    constexpr int NQ = K / 2;                         // component pairs (narrow, wide) = objects
    constexpr int NBLK = TR / 2 / TEAM;
#ifdef LAPF_EXP_SPLIT   /* experiment only: the configuration of the wrong-chi-square build of DESIGN.md 10 (whole-warp
                           tables spread over two lanes); with the round-1 sources it reproduces the failure */
    constexpr int SPLIT = NBLK >= 32 ? 1 : (NBLK >= 16 ? 2 : (TEAM == 1 ? 2 : 4));
#else
    constexpr int SPLIT = (TEAM == 1 || NBLK >= 32) ? 1 : (NBLK >= 16 ? 2 : 4);
#endif
    __syncwarp();   // readers of the previous table are done
    if (WPP > 1) rt += (lane / G::LPW) * (NBLK * T::RS + 8);      // the table of this half warp's vector (Scratch::TAB1)
#pragma unroll
    for (int j0 = 0; j0 < NBLK * SPLIT; j0 += G::LPW) {
        const int idx = j0 + lane % G::LPW;
        if ((NBLK * SPLIT) % G::LPW == 0 || idx < NBLK * SPLIT) {
            const int jb = idx / SPLIT, part = idx % SPLIT;   // local block: warp step jb / BPS of this warp, block jb % BPS
            const int step = (jb / G::BPS) * TEAM + tw;
            const float yb = (float)(row0 + step * G::RG + 2 * (jb % G::BPS)) + 0.5f;
            float4* o = reinterpret_cast<float4*>(rt + jb * T::RS);
            // anchor pieces q = part, part + SPLIT, ...: (sb dyb, sc dyb^2) of components T::ka(q), T::kb(q)
#pragma unroll
            for (int q0 = 0; q0 < NQ; q0 += SPLIT) {
                const int q = q0 + part;
                if (NQ % SPLIT == 0 || q < NQ) {
                    float y0a = cf.y0[T::ka(q0)], y0b = cf.y0[T::kb(q0)];
                    float sba = cf.sb[T::ka(q0) & 1], sbb = cf.sb[T::kb(q0) & 1];
                    float sca = cf.sc[T::ka(q0) & 1], scb = cf.sc[T::kb(q0) & 1];
#pragma unroll
                    for (int t = 1; t < SPLIT; ++t)
                        if (q0 + t < NQ && part == t) {
                            const int ka = T::ka(q0 + t), kb = T::kb(q0 + t);
                            y0a = cf.y0[ka]; y0b = cf.y0[kb];
                            sba = cf.sb[ka & 1]; sbb = cf.sb[kb & 1]; sca = cf.sc[ka & 1]; scb = cf.sc[kb & 1];
                        }
                    const float yda = __fsub_rn(yb, y0a), ydb = __fsub_rn(yb, y0b);
                    o[q] = make_float4(__fmul_rn(sba, yda), __fmul_rn(sbb, ydb),
                                       __fmul_rn(__fmul_rn(sca, yda), yda), __fmul_rn(__fmul_rn(scb, ydb), ydb));
                }
            }
            // factor quadruples pr = 2 c + ii = part, part + SPLIT, ...
            const float2 jlo = make_float2(-1.5f, -0.5f), jhi = make_float2(0.5f, 1.5f);
#pragma unroll
            for (int p0 = 0; p0 < 4; p0 += SPLIT) {
                const int pr = p0 + part;
                const bool c = (pr >> 1) != 0, hi = (pr & 1) != 0;
                const float sbc = c ? cf.sb[1] : cf.sb[0], scc = c ? cf.sc[1] : cf.sc[0];
                const float yd = __fsub_rn(yb, c ? cf.y0[1] : cf.y0[0]);
                const float p = __fmul_rn(sbc, yd);             // sb_c * dyb_c
                const float sy = __fmul_rn(__fmul_rn(scc, yd), 2.f);
                const float g = __fmul_rn(0.25f, scc);
                const float i = hi ? 0.5f : -0.5f;
                const float pj = __fmaf_rn(i, sbc, p), base = __fmaf_rn(i, sy, g);
                const float2 pj2 = make_float2(pj, pj), b2 = make_float2(base, base);
                const float2 alo = __ffma2_rn(jlo, pj2, b2), ahi = __ffma2_rn(jhi, pj2, b2);
                o[T::OFF_T / 4 + pr] = make_float4(ex2_approx(alo.x), ex2_approx(alo.y), ex2_approx(ahi.x), ex2_approx(ahi.y));
            }
        }
    }
    __syncwarp();
}

// Far-field culling.  |A_k| 2^(q) <= |A_k| 2^(kappa dy^2) for every pixel of a row at distance dy
// from the component's centre (kappa = sc - sb^2/(4 sa), the exponent maximised over dx), and the
// same with the roles of x and y swapped for a column panel.  A component whose bound over a whole
// row step (or panel) is below tau = 2^-27 |floor| is skipped there: the components of a class are
// added to the pixel as ONE term (see row_steps_fast), and up to four terms below tau sum to less
// than half an ulp of a model value that is at least the floor, so the FMA that would add them
// rounds them away: no MUFU, no FFMA, and (for non-negative amplitudes) bit-identical results.  Rows are
// culled per CLASS (all narrow cores / all wide wings): the active rows of a class are one interval
// of row steps, so a panel is walked as at most five segments (none, wings, all, wings, none), each
// a tight loop without per-row tests.  On a 128-pixel stamp the cores matter in ~1/4 of the rows and
// the wings in ~2/3.  The decision is a pure function of the coefficients (chi-square stays a
// function of the parameter vector); a nan/inf in them disables culling so it reaches chi-square.
template <int NX, int NY>
__device__ __forceinline__ void cull_one(float a, float x0, float y0, float sa, float sb, float sc, float floor_v,
                                         int& lo, int& hi, uint32_t& pm) {
    using G = Geo<NX>;
    constexpr int STEPS = NY / G::RG;
    constexpr uint32_t kAllPans = (1u << G::PANELS) - 1u;
    // approximate log2 / divide / sqrt are fine here: the radius gets a whole pixel of slack
    const float tau = __fmul_rn(0x1p-27f, fabsf(floor_v));
    const float L = __log2f(__fdividef(fabsf(a), tau));    // bits of headroom above tau
    lo = 0; hi = STEPS - 1;                                // default: everything (also for nan / inf)
    pm = kAllPans;
    if (L <= 0.f) {                                        // below tau everywhere
        lo = STEPS; hi = -1; pm = 0u;
    } else {
        const float sb2 = __fmul_rn(sb, sb);
        const float ky = __fsub_rn(sc, __fdividef(sb2, __fmul_rn(4.f, sa))), kx = __fsub_rn(sa, __fdividef(sb2, __fmul_rn(4.f, sc)));   // both < 0
        const float Y = __fadd_rn(__fsqrt_rn(__fdividef(L, -ky)), 1.f), X = __fadd_rn(__fsqrt_rn(__fdividef(L, -kx)), 1.f);
        if (Y < 1e6f && fabsf(y0) < 1e6f) {
            constexpr float kInvRG = 1.f / (float)G::RG;       // a power of two
            lo = max(0, (int)ceilf(__fmul_rn(__fsub_rn(__fsub_rn(y0, Y), (float)(G::RG - 1)), kInvRG)));
            hi = min(STEPS - 1, (int)floorf(__fmul_rn(__fadd_rn(y0, Y), kInvRG)));
            if (lo > hi) { lo = STEPS; hi = -1; }
        }
        if (G::PANELS > 1 && X < 1e6f && fabsf(x0) < 1e6f) {
            pm = 0u;
#pragma unroll
            for (int p = 0; p < G::PANELS; ++p)
                if (__fadd_rn(x0, X) >= (float)(p * G::PW) && __fsub_rn(x0, X) <= (float)(p * G::PW + G::PW - 1)) pm |= 1u << p;
        }
    }
}

// From the class intervals to the segments of every panel (the wing interval is widened to contain
// the core interval: evaluating a component where it is not needed is harmless).  The plain loop
// and team members (whose update time is set by the warp with the busiest rows) evaluate densely.
// Needs cf.fast.
template <int NB, int NX, int NY, int TEAM>
__device__ __forceinline__ void set_segments(Coef<NB>& cf, const int (&lo)[2], const int (&hi)[2], const uint32_t (&pm)[2]) {
    using G = Geo<NX>;
    constexpr int STEPS = NY / G::RG;
    unsigned n = 0;
#pragma unroll
    for (int pan = 0; pan < G::PANELS; ++pan) {
        const bool n_on = ((pm[0] >> pan) & 1u) && lo[0] <= hi[0];
        const bool w_on = ((pm[1] >> pan) & 1u) && lo[1] <= hi[1];
        int nlo = n_on ? lo[0] : STEPS, nhi1 = n_on ? hi[0] + 1 : STEPS;
        int wlo = w_on ? lo[1] : nlo, whi1 = w_on ? hi[1] + 1 : nhi1;
        wlo = min(wlo, nlo);
        whi1 = max(whi1, nhi1);
        if (!n_on) { nlo = whi1; nhi1 = whi1; }
        if (!cf.fast || TEAM > 1) { wlo = 0; nlo = 0; nhi1 = STEPS; whi1 = STEPS; }
        cf.seg[pan][0] = wlo; cf.seg[pan][1] = nlo; cf.seg[pan][2] = nhi1; cf.seg[pan][3] = whi1;
        n += (unsigned)((nhi1 - nlo) + (whi1 - wlo));
    }
    cf.nexp = (unsigned)(G::PW * G::RG * NB) * n;
}

// cooperative form: lane k < K works out component k, the hulls are formed with shuffles
template <int NB, int NX, int NY, int TEAM = 1>
__device__ __forceinline__ void set_cull(Coef<NB>& cf, int lane) {
    using G = Geo<NX>;
    constexpr int K = 2 * NB;
    constexpr int STEPS = NY / G::RG;
    float a = cf.amp[0], x0 = cf.x0[0], y0 = cf.y0[0];
#pragma unroll
    for (int k = 1; k < K; ++k)
        if (lane == k) { a = cf.amp[k]; x0 = cf.x0[k]; y0 = cf.y0[k]; }
    const int sh = lane & 1;
    const float sa = sh ? cf.sa[1] : cf.sa[0], sb = sh ? cf.sb[1] : cf.sb[0], sc = sh ? cf.sc[1] : cf.sc[0];
    int lo, hi;
    uint32_t pm;
    cull_one<NX, NY>(a, x0, y0, sa, sb, sc, cf.floor, lo, hi, pm);
    if (lane >= K) { lo = STEPS; hi = -1; pm = 0u; }       // neutral element
    // hull over the components of each class: lanes of equal parity (xor 2, 4 keeps the parity)
#pragma unroll
    for (int off = 2; off <= 4; off <<= 1) {
        lo = min(lo, __shfl_xor_sync(kFull, lo, off));
        hi = max(hi, __shfl_xor_sync(kFull, hi, off));
        pm |= __shfl_xor_sync(kFull, pm, off);
    }
    int clo[2], chi[2];
    uint32_t cpm[2];
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        clo[c] = __shfl_sync(kFull, lo, c);
        chi[c] = __shfl_sync(kFull, hi, c);
        cpm[c] = __shfl_sync(kFull, pm, c);
    }
    set_segments<NB, NX, NY, TEAM>(cf, clo, chi, cpm);
}

// one-thread form (the batched sampler prepares one walker per lane): same decisions
template <int NB, int NX, int NY>
__device__ __forceinline__ void set_cull_serial(Coef<NB>& cf) {
    constexpr int K = 2 * NB;
    constexpr int STEPS = NY / Geo<NX>::RG;
    int clo[2] = {STEPS, STEPS}, chi[2] = {-1, -1};
    uint32_t cpm[2] = {0u, 0u};
#pragma unroll
    for (int k = 0; k < K; ++k) {
        int lo, hi;
        uint32_t pm;
        cull_one<NX, NY>(cf.amp[k], cf.x0[k], cf.y0[k], cf.sa[k & 1], cf.sb[k & 1], cf.sc[k & 1], cf.floor, lo, hi, pm);
        clo[k & 1] = min(clo[k & 1], lo);
        chi[k & 1] = max(chi[k & 1], hi);
        cpm[k & 1] |= pm;
    }
    set_segments<NB, NX, NY, 1>(cf, clo, chi, cpm);
}

template <int NB, int NX, int NY, int TEAM = 1>
__device__ __forceinline__ void no_cull(Coef<NB>& cf) {
    const int clo[2] = {0, 0}, chi[2] = {NY / Geo<NX>::RG - 1, NY / Geo<NX>::RG - 1};
    const uint32_t cpm[2] = {0xffffffffu, 0xffffffffu};
    set_segments<NB, NX, NY, TEAM>(cf, clo, chi, cpm);
}

// The factorised pixel loop multiplies factors whose exponents can be large although their sum is
// not.  It is used only when, for every pixel of the stamp, the lane constants' exponent
// |j (sa (2 dxa + j) + sb dy0) + i (sb dxa + 2 sc dy0)| and the block factors' exponent
// |j sb (dyb + i) + 2 i sc dyb + sc / 4| stay below 40 -- no factor overflows or underflows on its
// own -- and when an anchor exponential that underflows (q0 < -126) implies that its eight pixels
// are below 2^-46 |A| <= 2^-25 |floor|.  Anything else, nan and inf included, takes the plain loop
// (one exponential per pixel and component).  The decision is a function of the coefficients only
// and is the same in every lane.
template <int NX, int NY>
__device__ __forceinline__ bool fast_one(float a, float x0, float y0, float yref, float sa, float sb, float sc,
                                         float floor_v) {
    const float dxm = __fadd_rn(fabsf(__fsub_rn(x0, 0.5f * NX)), 0.5f * NX);      // >= |anchor - x0| for every anchor column
    const float dym = __fadd_rn(fabsf(__fsub_rn(yref, 0.5f * NY)), 0.5f * NY);    // >= |block centre - y0_c| for every block
    const float dy0 = fabsf(__fsub_rn(yref, y0));
    const float asa = fabsf(sa), asb = fabsf(sb), asc = fabsf(sc);
    // argc = 1.5 (|sa| (2 dxm + 1.5) + |sb| dy0) + 0.5 (|sb| dxm + 2 |sc| dy0);  argt = 1.5 |sb| (dym + 0.5) + |sc| (dym + 0.25)
    const float c1 = __fmaf_rn(asa, __fmaf_rn(2.f, dxm, 1.5f), __fmul_rn(asb, dy0));
    const float c2 = __fmaf_rn(asb, dxm, __fmul_rn(__fmul_rn(2.f, asc), dy0));
    const float argc = __fmaf_rn(1.5f, c1, __fmul_rn(0.5f, c2));
    const float argt = __fmaf_rn(__fmul_rn(1.5f, asb), __fadd_rn(dym, 0.5f), __fmul_rn(asc, __fadd_rn(dym, 0.25f)));
    return argc <= 40.f && argt <= 40.f && asc <= 1e30f &&
           fabsf(a) <= __fmul_rn(0x1p21f, fabsf(floor_v)) && fabsf(a) <= 1e12f;    // all false on nan
}

template <int NB, int NX, int NY>
__device__ __forceinline__ void set_fast(Coef<NB>& cf, int lane) {
    constexpr int K = 2 * NB;
    float a = cf.amp[0], x0 = cf.x0[0], y0 = cf.y0[0];
#pragma unroll
    for (int k = 1; k < K; ++k)
        if (lane == k) { a = cf.amp[k]; x0 = cf.x0[k]; y0 = cf.y0[k]; }
    const int sh = lane & 1;
    const float sa = sh ? cf.sa[1] : cf.sa[0], sb = sh ? cf.sb[1] : cf.sb[0], sc = sh ? cf.sc[1] : cf.sc[0];
    const bool ok = fast_one<NX, NY>(a, x0, y0, sh ? cf.y0[1] : cf.y0[0], sa, sb, sc, cf.floor);
    cf.fast = __all_sync(kFull, ok || lane >= K);
}

template <int NB, int NX, int NY>
__device__ __forceinline__ void set_fast_serial(Coef<NB>& cf) {
    constexpr int K = 2 * NB;
    bool ok = true;
#pragma unroll
    for (int k = 0; k < K; ++k)
        ok = ok && fast_one<NX, NY>(cf.amp[k], cf.x0[k], cf.y0[k], cf.y0[k & 1], cf.sa[k & 1], cf.sb[k & 1],
                                    cf.sc[k & 1], cf.floor);
    cf.fast = ok;
}

// Warp steps [i0, i1) of one panel for the component classes KIND says (0: none, the model is the
// floor; 1: wide wings only; 2: all components).  chi-square terms are added to the four FP32
// accumulators s0, s1 in step order, whatever the segmentation (so culling does not regroup sums).
// PREP = true: the planes hold d*sqrt(w) and -sqrt(w) (the sampler converts a stamp once after
// staging it); PREP = false: raw data / weight planes, converted per pixel.  Both give
// bit-identical chi-square: the residual is always  r = fma(-sqrt(w), m, d*sqrt(w)),  chi2 += r*r.
struct StepPtrs {          // where the next warp step of this lane lives
    const float* rp;       // block table entry
    const float* dp;       // data plane, first row of the block at the lane's columns
    const float* wp;       // weight plane, same
    float* mp;             // model output (STORE only), same
    uint32_t tm;           // TMEM address of the lane's values (TM only)
    float row;             // first row of the block (plain loop only)
};

// model of 8 pixels (pairs: row 0 px 0-1, row 0 px 2-3, row 1 px 0-1, row 1 px 2-3) -> (optional
// store) -> residuals -> chi-square accumulators
template <int NX, bool STORE, bool PREP>
__device__ __forceinline__ void finish_step(const float2 (&m)[4], const float4& d0, const float4& d1,
                                            const float4& w0, const float4& w1, float* mp, float2& s0, float2& s1,
                                            bool keep = true) {
    if (STORE && keep) {
        *reinterpret_cast<float4*>(mp) = make_float4(m[0].x, m[0].y, m[1].x, m[1].y);
        *reinterpret_cast<float4*>(mp + NX) = make_float4(m[2].x, m[2].y, m[3].x, m[3].y);
    }
    float2 dv[4] = {make_float2(d0.x, d0.y), make_float2(d0.z, d0.w), make_float2(d1.x, d1.y),
                    make_float2(d1.z, d1.w)};
    float2 wv[4] = {make_float2(w0.x, w0.y), make_float2(w0.z, w0.w), make_float2(w1.x, w1.y),
                    make_float2(w1.z, w1.w)};
    if (!PREP) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float rx = sqrtf(wv[j].x), ry = sqrtf(wv[j].y);
            dv[j] = make_float2(dv[j].x * rx, dv[j].y * ry);
            wv[j] = make_float2(-rx, -ry);
        }
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const float2 ra = __ffma2_rn(wv[j], m[j], dv[j]);
        const float2 rb = __ffma2_rn(wv[2 + j], m[2 + j], dv[2 + j]);
        s0 = __ffma2_rn(ra, ra, s0);
        s1 = __ffma2_rn(rb, rb, s1);
    }
}

// ---- plain loop: one exponential per pixel and component -------------------------------------
// q = fma(dx, fma(sa, dx, sb*dy), sc*dy^2), e = ex2(q), m = fma(A, e, m) per pixel and component,
// issued as packed FFMA2 (fma.rn.f32x2, new on sm_100: two adjacent pixels per instruction, scalar
// coefficients as broadcast operands) -- 3 FFMA2 + 2 MUFU.EX2 per pixel PAIR and component:
// SFU-bound.  Kept for parameter vectors set_fast turns away; it takes no table (the row terms are
// worked out per row on the spot).
template <int NB, int NX, int NY, bool STORE, bool PREP, int WPP = 1, int TM = 0>
__device__ __forceinline__ void row_steps(const Coef<NB>& cf, const float2 (&xd)[2 * NB][2], float2& s0, float2& s1,
                                          int& i, int i1, StepPtrs& sp, bool keep = true) {
    using G = Geo<NX, WPP>;
    constexpr int K = 2 * NB;
    static_assert(TM == 0 || TM == 1, "the plain loop reads both planes from one place");
    const float* dp = sp.dp;
    const float* wp = sp.wp;
    float* mp = sp.mp;
    float row = sp.row;
    uint32_t tm = sp.tm;
#pragma unroll 1
    for (; i < i1; ++i) {
        float4 d0, d1, w0, w1;
        if (TM == 1) {      // the step's 16 values from the TMEM pixel store (same layout as row_steps_fast)
            uint32_t tv[16];
            tmem_ld16_issue(tm, tv);
            tmem_ld16_wait(tv);
            d0 = make_float4(__uint_as_float(tv[0]), __uint_as_float(tv[1]), __uint_as_float(tv[2]), __uint_as_float(tv[3]));
            d1 = make_float4(__uint_as_float(tv[4]), __uint_as_float(tv[5]), __uint_as_float(tv[6]), __uint_as_float(tv[7]));
            w0 = make_float4(__uint_as_float(tv[8]), __uint_as_float(tv[9]), __uint_as_float(tv[10]), __uint_as_float(tv[11]));
            w1 = make_float4(__uint_as_float(tv[12]), __uint_as_float(tv[13]), __uint_as_float(tv[14]), __uint_as_float(tv[15]));
            tm += 16;
        } else {
            d0 = *reinterpret_cast<const float4*>(dp);
            d1 = *reinterpret_cast<const float4*>(dp + NX);
            w0 = *reinterpret_cast<const float4*>(wp);
            w1 = *reinterpret_cast<const float4*>(wp + NX);
        }
        float2 m[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) m[j] = make_float2(cf.floor, cf.floor);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const float2 sa2 = make_float2(cf.sa[k & 1], cf.sa[k & 1]);
            const float2 am2 = make_float2(cf.amp[k], cf.amp[k]);
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const float yd = __fsub_rn(__fadd_rn(row, (float)r), cf.y0[k]);
                const float by = __fmul_rn(cf.sb[k & 1], yd), cy = __fmul_rn(__fmul_rn(cf.sc[k & 1], yd), yd);
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const float2 t = __ffma2_rn(sa2, xd[k][j], make_float2(by, by));
                    const float2 q = __ffma2_rn(xd[k][j], t, make_float2(cy, cy));
                    const float2 e = make_float2(ex2_approx(q.x), ex2_approx(q.y));
                    m[2 * r + j] = __ffma2_rn(am2, e, m[2 * r + j]);
                }
            }
        }
        finish_step<NX, STORE, PREP>(m, d0, d1, w0, w1, mp, s0, s1, keep);
        if (STORE) mp += G::RG * NX;
        dp += G::RG * NX;
        wp += G::RG * NX;
        row += (float)G::RG;
    }
    sp.dp = dp; sp.wp = wp; sp.mp = mp; sp.row = row; sp.tm = tm;
}

// ---- factorised loop -------------------------------------------------------------------------
// The exponent is a quadratic form, so around the centre (xa, yb) of a lane's 2 x 4 block, with
// i in {-1/2, 1/2} (row), j in {-3/2, -1/2, 1/2, 3/2} (column), dxa_k = xa - x0_k, dyb_k = yb - y0_k,
//     q_k(xa + j, yb + i) = q_k(xa, yb) + j sa (2 dxa_k + j) + sb (i dxa_k + j dyb_k + i j)
//                                        + i sc (2 dyb_k + i),
// and dyb_k = dyb_c + (y0_c - y0_k) with c the first component of k's shape class, so
//     A_k 2^q_k(xa + j, yb + i) = E_k * C_k,ij * T_c,ij
//     E_k    = 2^q_k(xa, yb)                            ONE MUFU.EX2 per block and component
//     C_k,ij = A_k 2^(j (sa (2 dxa_k + j) + sb dy0_k) + i (sb dxa_k + 2 sc dy0_k))   lane constant (registers),
//                                                       dy0_k = y0_c - y0_k
//     T_c,ij = 2^(j sb (dyb_c + i) + 2 i sc dyb_c + sc / 4)                          block table, shared by the class
// and a class adds  T_c,ij * sum_k C_k,ij E_k  to the pixel: per pixel pair NB + 1 packed
// operations for NB components, plus 2 FMA (one packed FMA pair serves the two objects' components
// of a class) + 1 MUFU per component for the anchor.  A warp step of 8 pixels x 4 components is 36
// packed FP32 instructions and 4 MUFU (plain loop: 56 packed and 32 MUFU): the loop is bound by FP32
// issue, not by the SFU.
template <int NB>
struct LaneK {
    static constexpr int K = 2 * NB;
    float dxa[K];        // anchor offset to the centre of component k
    float2 C[K][4];      // pixel pairs: row 0 (-3/2,-1/2), row 0 (1/2,3/2), row 1 (-3/2,-1/2), row 1 (1/2,3/2)
};

// The 8 lane constants C_k,ij of one component at one anchor column (dxa = anchor - x0_k), rows
// i = -1/2 (lo) and +1/2 (hi), columns j = -3/2, -1/2, 1/2, 3/2.
__device__ __forceinline__ void block_consts(float amp, float dxa, float dy0, float sa, float sb, float sc,
                                             float4& lo, float4& hi) {
    const float u = __fmul_rn(sb, dy0), d2 = __fmul_rn(2.f, dxa);
    const float v = __fmaf_rn(sb, dxa, __fmul_rn(2.f, __fmul_rn(sc, dy0)));
    const float2 u2 = make_float2(u, u), sa2 = make_float2(sa, sa), d22 = make_float2(d2, d2);
    const float2 jlo = make_float2(-1.5f, -0.5f), jhi = make_float2(0.5f, 1.5f);
    const float2 xlo = __fmul2_rn(jlo, __ffma2_rn(sa2, __fadd2_rn(d22, jlo), u2));
    const float2 xhi = __fmul2_rn(jhi, __ffma2_rn(sa2, __fadd2_rn(d22, jhi), u2));
    const float hv = 0.5f * v;
    const float2 m2 = make_float2(-hv, -hv), p2 = make_float2(hv, hv);
    const float2 a0 = __fadd2_rn(xlo, m2), a1 = __fadd2_rn(xhi, m2), b0 = __fadd2_rn(xlo, p2), b1 = __fadd2_rn(xhi, p2);
    lo = make_float4(__fmul_rn(amp, ex2_approx(a0.x)), __fmul_rn(amp, ex2_approx(a0.y)), __fmul_rn(amp, ex2_approx(a1.x)),
                     __fmul_rn(amp, ex2_approx(a1.y)));
    hi = make_float4(__fmul_rn(amp, ex2_approx(b0.x)), __fmul_rn(amp, ex2_approx(b0.y)), __fmul_rn(amp, ex2_approx(b1.x)),
                     __fmul_rn(amp, ex2_approx(b1.y)));
}

template <int NB, int NX>
__device__ __forceinline__ void read_consts(LaneK<NB>& lk, const float* __restrict__ ct, const Coef<NB>& cf, int lane, int pan);

// The C_k,ij of the GPR anchors of a panel (columns 4a + 1.5), worked out once per proposal by the
// warp -- one (anchor, component) pair per lane and round -- and handed round through the column
// table ct[k][row of the block][a][4]; every lane then reads the 8K values of its own anchor.
template <int NB, int NX, int WPP = 1>
__device__ __forceinline__ void coop_consts(LaneK<NB>& lk, float* __restrict__ ct, const Coef<NB>& cf, int lane, int pan) {
    using G = Geo<NX, WPP>;
    constexpr int K = 2 * NB;
    __syncwarp();   // readers of the previous column table are done
    if (WPP > 1) ct += (lane / G::LPW) * (K * 2 * G::GPR * 4);     // the table of this half warp's vector (Scratch::CT)
#pragma unroll
    for (int t0 = 0; t0 < G::GPR * K; t0 += G::LPW) {
        const int t = t0 + lane % G::LPW;
        if ((G::GPR * K) % G::LPW == 0 || t < G::GPR * K) {
            const int a = t % G::GPR, kk = t / G::GPR;
            float amp = cf.amp[0], x0 = cf.x0[0], y0 = cf.y0[0];
#pragma unroll
            for (int k = 1; k < K; ++k)
                if (kk == k) { amp = cf.amp[k]; x0 = cf.x0[k]; y0 = cf.y0[k]; }
            const int c = kk & 1;
            const float sa = c ? cf.sa[1] : cf.sa[0], sb = c ? cf.sb[1] : cf.sb[0], sc = c ? cf.sc[1] : cf.sc[0];
            const float dy0 = (c ? cf.y0[1] : cf.y0[0]) - y0;           // exactly 0 for the class's first component
            float4 lo, hi;
            block_consts(amp, ((float)(pan * G::PW + 4 * a) + 1.5f) - x0, dy0, sa, sb, sc, lo, hi);
            reinterpret_cast<float4*>(ct)[(kk * 2) * G::GPR + a] = lo;
            reinterpret_cast<float4*>(ct)[(kk * 2 + 1) * G::GPR + a] = hi;
        }
    }
    __syncwarp();
    read_consts<NB, NX>(lk, ct, cf, lane, pan);
}

// TEAM > 1: the column tables of ALL panels, once per proposal, by the whole team -- one (panel,
// component, anchor) triple per thread.  Every member used to work out the constants of its own
// anchor (own_consts: 8K exponentials per lane and panel, the same 16 anchors in every warp and in
// both block rows: 32x redundant, and what kept the XU pipe busy in the team kernels); now the
// team's 32 TEAM threads share the work and a named barrier hands the table over.  Same
// block_consts, same inputs: same bits as coop_consts / own_consts.
template <int NB, int NX, int TEAM>
__device__ __forceinline__ void team_consts(float* __restrict__ ct, const Coef<NB>& cf, int tid) {
    using G = Geo<NX>;
    constexpr int K = 2 * NB;
    constexpr int TASKS = G::PANELS * K * G::GPR;
#pragma unroll
    for (int t0 = 0; t0 < TASKS; t0 += TEAM * 32) {
        const int t = t0 + tid;
        if (TASKS % (TEAM * 32) == 0 || t < TASKS) {
            const int a = t % G::GPR, kk = (t / G::GPR) % K, pan = t / (G::GPR * K);
            float amp = cf.amp[0], x0 = cf.x0[0], y0 = cf.y0[0];
#pragma unroll
            for (int k = 1; k < K; ++k)
                if (kk == k) { amp = cf.amp[k]; x0 = cf.x0[k]; y0 = cf.y0[k]; }
            const int c = kk & 1;
            const float sa = c ? cf.sa[1] : cf.sa[0], sb = c ? cf.sb[1] : cf.sb[0], sc = c ? cf.sc[1] : cf.sc[0];
            const float dy0 = (c ? cf.y0[1] : cf.y0[0]) - y0;
            float4 lo, hi;
            block_consts(amp, ((float)(pan * G::PW + 4 * a) + 1.5f) - x0, dy0, sa, sb, sc, lo, hi);
            float4* base = reinterpret_cast<float4*>(ct) + pan * (K * 2 * G::GPR);
            base[(kk * 2) * G::GPR + a] = lo;
            base[(kk * 2 + 1) * G::GPR + a] = hi;
        }
    }
}

// The same numbers without the exchange: every lane works out the 8K constants of its own anchor
// (4x the arithmetic, but no shared-memory round trip) -- for team members, where the latency of
// one update is what counts.
template <int NB, int NX>
__device__ __forceinline__ void own_consts(LaneK<NB>& lk, const Coef<NB>& cf, int lane, int pan) {
    using G = Geo<NX>;
    constexpr int K = 2 * NB;
    const float xa = (float)(pan * G::PW + 4 * (lane % G::GPR)) + 1.5f;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const int c = k & 1;
        lk.dxa[k] = xa - cf.x0[k];
        float4 lo, hi;
        block_consts(cf.amp[k], lk.dxa[k], cf.y0[c] - cf.y0[k], cf.sa[c], cf.sb[c], cf.sc[c], lo, hi);
        lk.C[k][0] = make_float2(lo.x, lo.y); lk.C[k][1] = make_float2(lo.z, lo.w);
        lk.C[k][2] = make_float2(hi.x, hi.y); lk.C[k][3] = make_float2(hi.z, hi.w);
    }
}

template <int NB, int NX>
__device__ __forceinline__ void read_consts(LaneK<NB>& lk, const float* __restrict__ ct, const Coef<NB>& cf, int lane, int pan) {
    using G = Geo<NX>;
    constexpr int K = 2 * NB;
    const int mine = lane % G::GPR;
    const float xa = (float)(pan * G::PW + 4 * mine) + 1.5f;
#pragma unroll
    for (int k = 0; k < K; ++k) {
#pragma unroll
        for (int ii = 0; ii < 2; ++ii) {
            const float4 v = reinterpret_cast<const float4*>(ct)[(k * 2 + ii) * G::GPR + mine];
            lk.C[k][2 * ii] = make_float2(v.x, v.y);
            lk.C[k][2 * ii + 1] = make_float2(v.z, v.w);
        }
        lk.dxa[k] = xa - cf.x0[k];
    }
}

template <int NB, int NX, int NY, bool STORE, bool PREP, int KIND, int TM = 0, int WPP = 1>
__device__ __forceinline__ void row_steps_fast(const Coef<NB>& cf, const LaneK<NB>& lk, float2& s0, float2& s1,
                                               int& i, int i1, StepPtrs& sp, bool keep = true) {
    using G = Geo<NX, WPP>;
    using T = Tab<NB>;
    constexpr int K = 2 * NB;
    const float* rp = sp.rp;
    const float* dp = sp.dp;
    const float* wp = sp.wp;
    float* mp = sp.mp;
    uint32_t tm = sp.tm;
#pragma unroll kLoopUnroll
    for (; i < i1; ++i) {
        float4 d0, d1, w0, w1;
        uint32_t tv[16];
        if (TM == 1) {
            tmem_ld16_issue(tm, tv);
        } else if (TM == 2) {
            tmem_ld8_issue(tm, tv);
            d0 = *reinterpret_cast<const float4*>(dp);
            d1 = *reinterpret_cast<const float4*>(dp + NX);
        } else {
            d0 = *reinterpret_cast<const float4*>(dp);
            d1 = *reinterpret_cast<const float4*>(dp + NX);
            w0 = *reinterpret_cast<const float4*>(wp);
            w1 = *reinterpret_cast<const float4*>(wp + NX);
        }
        float2 m[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) m[j] = make_float2(cf.floor, cf.floor);
        if (KIND > 0) {
#pragma unroll
            for (int c = (KIND == 2 ? 0 : 1); c < 2; ++c) {
                const float4 T0 = reinterpret_cast<const float4*>(rp + T::OFF_T)[2 * c];
                const float4 T1 = reinterpret_cast<const float4*>(rp + T::OFF_T)[2 * c + 1];
                // anchor exponents of the class: objects 0 and 1 as one packed pair (table piece c), object 2 on its own
                float ea[NB];
                {
                    const float4 r = reinterpret_cast<const float4*>(rp)[c];
                    const float2 dx = make_float2(lk.dxa[c], lk.dxa[2 + c]);
                    const float2 q = __ffma2_rn(dx, __ffma2_rn(make_float2(cf.sa[c], cf.sa[c]), dx, make_float2(r.x, r.y)),
                                                make_float2(r.z, r.w));
                    ea[0] = ex2_approx(q.x);
                    ea[1] = ex2_approx(q.y);
                }
                if (NB > 2) {
                    const float4 r = reinterpret_cast<const float4*>(rp)[2];
                    const float dx = lk.dxa[4 + c];
                    ea[NB - 1] = ex2_approx(__fmaf_rn(dx, __fmaf_rn(cf.sa[c], dx, c ? r.y : r.x), c ? r.w : r.z));
                }
                float2 u[4];
#pragma unroll
                for (int o = 0; o < NB; ++o) {
                    const int k = 2 * o + c;
                    const float2 e2 = make_float2(ea[o], ea[o]);
#pragma unroll
                    for (int p = 0; p < 4; ++p)
                        u[p] = (o == 0) ? __fmul2_rn(lk.C[k][p], e2) : __ffma2_rn(lk.C[k][p], e2, u[p]);
                }
                m[0] = __ffma2_rn(make_float2(T0.x, T0.y), u[0], m[0]); m[1] = __ffma2_rn(make_float2(T0.z, T0.w), u[1], m[1]);
                m[2] = __ffma2_rn(make_float2(T1.x, T1.y), u[2], m[2]); m[3] = __ffma2_rn(make_float2(T1.z, T1.w), u[3], m[3]);
            }
        }
        if (TM == 1) {
            tmem_ld16_wait(tv);
            d0 = make_float4(__uint_as_float(tv[0]), __uint_as_float(tv[1]), __uint_as_float(tv[2]), __uint_as_float(tv[3]));
            d1 = make_float4(__uint_as_float(tv[4]), __uint_as_float(tv[5]), __uint_as_float(tv[6]), __uint_as_float(tv[7]));
            tm += 16;
        } else if (TM == 2) {
            tmem_ld8_wait(tv);
            tm += 8;
        }
        if (TM) {
            w0 = make_float4(__uint_as_float(tv[8]), __uint_as_float(tv[9]), __uint_as_float(tv[10]), __uint_as_float(tv[11]));
            w1 = make_float4(__uint_as_float(tv[12]), __uint_as_float(tv[13]), __uint_as_float(tv[14]), __uint_as_float(tv[15]));
        }
        finish_step<NX, STORE, PREP>(m, d0, d1, w0, w1, mp, s0, s1, keep);
        if (STORE) mp += G::RG * NX;
        rp += G::BPS * T::RS;
        dp += G::RG * NX;
        wp += G::RG * NX;
    }
    sp.rp = rp; sp.dp = dp; sp.wp = wp; sp.mp = mp; sp.tm = tm;
}

// This lane's FP32 partial of chi-square over one panel of one table ("half") of the stamp, by ONE
// warp, with the block table of that half already built in `scratch` (if cf.fast).  The column
// table goes to the scratch behind it.
template <int NB, int NX, int NY, bool STORE, bool PREP, int TM = 0>
__device__ __forceinline__ float panel_chi2(const Coef<NB>& cf, float* __restrict__ scratch,
                                            const float* __restrict__ d, const float* __restrict__ w,
                                            float* __restrict__ model_out, int lane, int half, int pan, uint32_t tmem) {
    using G = Geo<NX>;
    using T = Tab<NB>;
    using R = Rows<NY, 1>;
    constexpr int K = 2 * NB;
    constexpr int TR = R::TR;
    constexpr int STEPS = TR / G::RG;            // warp steps per table (per panel)
    static_assert(TM == 0 || PREP, "the TMEM pixel store holds prepared stamps");
    static_assert(TM != 1 || (R::HALVES == 1 && G::PANELS == 1), "both planes fit the 512 TMEM columns up to 64 x 64 pixels");
    constexpr int TM_STEP = TM == 1 ? 16 : 8;     // TMEM columns per warp step
    static_assert(TR % G::RG == 0, "unsupported stamp height");
    const float* rt = scratch;
    float* ct = scratch + Scratch<NB, NX, NY>::TAB;
    const int a = lane % G::GPR, b = lane / G::GPR;
    const int off0 = (half * TR + 2 * b) * NX + pan * G::PW + 4 * a;   // the lane's block of warp step 0
    // segments of this panel, clipped to the warp steps of this table:
    //   [0,wlo) none, [wlo,nlo) wings, [nlo,nhi1) all, [nhi1,whi1) wings, [whi1,STEPS) none
    const bool p1 = G::PANELS > 1 && pan > 0;   // (constant indices keep the coefficients in registers)
    int wlo = p1 ? cf.seg[1][0] : cf.seg[0][0], nlo = p1 ? cf.seg[1][1] : cf.seg[0][1];
    int nhi1 = p1 ? cf.seg[1][2] : cf.seg[0][2], whi1 = p1 ? cf.seg[1][3] : cf.seg[0][3];
    if (R::HALVES > 1) {
        const int base = half * STEPS;
        wlo = min(max(wlo - base, 0), STEPS); nlo = min(max(nlo - base, 0), STEPS);
        nhi1 = min(max(nhi1 - base, 0), STEPS); whi1 = min(max(whi1 - base, 0), STEPS);
    }
    float2 s0 = make_float2(0.f, 0.f), s1 = make_float2(0.f, 0.f);
    if (cf.fast) {
        LaneK<NB> lk;
        coop_consts<NB, NX>(lk, ct, cf, lane, pan);
        // contiguous steps: the pointers run through the segments
        StepPtrs sp{rt + b * T::RS, d + off0, w + off0, STORE ? model_out + off0 : nullptr,
                    tmem + (uint32_t)((half * G::PANELS + pan) * STEPS * TM_STEP), 0.f};
        int i = 0;
        if (NX < 64) {
            // 32-pixel stamps have no far field (set_cull is never called for them)
            row_steps_fast<NB, NX, NY, STORE, PREP, 2, TM>(cf, lk, s0, s1, i, STEPS, sp);
        } else {
            row_steps_fast<NB, NX, NY, STORE, PREP, 0, TM>(cf, lk, s0, s1, i, wlo, sp);
            row_steps_fast<NB, NX, NY, STORE, PREP, 1, TM>(cf, lk, s0, s1, i, nlo, sp);
            row_steps_fast<NB, NX, NY, STORE, PREP, 2, TM>(cf, lk, s0, s1, i, nhi1, sp);
            row_steps_fast<NB, NX, NY, STORE, PREP, 1, TM>(cf, lk, s0, s1, i, whi1, sp);
            row_steps_fast<NB, NX, NY, STORE, PREP, 0, TM>(cf, lk, s0, s1, i, STEPS, sp);
        }
    } else {
        float2 xd[K][2];   // column offsets of the lane's pixel pairs (0,1) and (2,3)
        const float fa = (float)(pan * G::PW + 4 * a);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const float2 nx0 = make_float2(-cf.x0[k], -cf.x0[k]);
            xd[k][0] = __fadd2_rn(make_float2(fa, fa + 1.f), nx0);
            xd[k][1] = __fadd2_rn(make_float2(fa + 2.f, fa + 3.f), nx0);
        }
#pragma unroll 1
        for (int st = 0; st < STEPS; ++st) {
            const int so = st * G::RG * NX;
            StepPtrs sp{nullptr, d + off0 + so, w + off0 + so, STORE ? model_out + off0 + so : nullptr,
                        TM == 1 ? tmem + (uint32_t)(st * 16) : 0u, (float)(half * TR + st * G::RG + 2 * b)};
            int i = 0;
            row_steps<NB, NX, NY, STORE, PREP, 1, (TM == 1 ? 1 : 0)>(cf, xd, s0, s1, i, 1, sp);
        }
    }
    // at most 16 steps x 8 pixels over 4 accumulators
    return (s0.x + s0.y) + (s1.x + s1.y);
}

// chi-square of one parameter vector over the stamp by ONE warp (a team member's share: team_chi2).
// Builds the block and column tables in `scratch` (Scratch<NB, NX, NY>::FLOATS
// floats of this warp's own shared memory) itself.  `exps` counts the component evaluations
// (pixels x components) the far-field culling left to do.
template <int NB, int NX, int NY, bool STORE, bool PREP, int TEAM = 1, int TM = 0>
__device__ __forceinline__ double warp_chi2(const Coef<NB>& cf, float* __restrict__ scratch,
                                            const float* __restrict__ d, const float* __restrict__ w,
                                            float* __restrict__ model_out, int lane, int tw = 0,
                                            unsigned* exps = nullptr, uint32_t tmem = 0) {
    static_assert(TEAM == 1, "whole-warp passes only");
    using G = Geo<NX>;
    using R = Rows<NY, TEAM>;
    double acc = 0.0;
    if (exps) *exps += cf.nexp;
#pragma unroll 1
    for (int half = 0; half < R::HALVES; ++half) {
        if (cf.fast) build_row_table<NB, NX, R::TR, TEAM>(scratch, cf, lane, half * R::TR, tw);
#pragma unroll 1
        for (int pan = 0; pan < G::PANELS; ++pan)     // FP32 partial sums of one panel -> FP64
            acc += (double)panel_chi2<NB, NX, NY, STORE, PREP, TM>(cf, scratch, d, w, model_out, lane, half, pan, tmem);
    }
    return warp_sum_f64(acc);
}

// One-table, one-panel stamps: this lane's partial of warp_chi2, unreduced.  The caller reduces
// (warp_sum_f64, or warp_sum_f64_of on the 32 partials gathered in shared memory) and counts cf.nexp.
template <int NB, int NX, int NY, int TM>
__device__ __forceinline__ float lane_chi2(const Coef<NB>& cf, float* __restrict__ scratch, const float* __restrict__ d,
                                           const float* __restrict__ w, int lane, uint32_t tmem) {
    static_assert(Geo<NX>::PANELS == 1 && Rows<NY, 1>::HALVES == 1, "one table, one panel");
    if (cf.fast) build_row_table<NB, NX, NY, 1>(scratch, cf, lane, 0, 0);
    return panel_chi2<NB, NX, NY, false, true, TM>(cf, scratch, d, w, nullptr, lane, 0, 0, tmem);
}

// TEAM > 1: this warp's share of chi-square of one parameter vector (the caller adds the TEAM partials
// in a fixed order).  Warp tw works on ONE column panel (tw % PANELS) and on every (TEAM / PANELS)-th
// warp step of it over the whole height of the stamp: one block table (its own steps only), one read
// of the lane constants from the team's column table (team_consts), one run of MY steps.  (Round 1
// gave a member every TEAM-th step of every panel and table half: on a 128-pixel stamp with 16 warps
// that was four single-step loops, each with its own table build or constant read.)
template <int NB, int NX, int NY, int TEAM>
__device__ __forceinline__ double team_chi2(const Coef<NB>& cf, float* __restrict__ rt, const float* __restrict__ d,
                                            const float* __restrict__ w, int lane, int tw, unsigned* exps,
                                            const float* __restrict__ team_ct) {
    using G = Geo<NX>;
    using T = Tab<NB>;
    constexpr int K = 2 * NB;
    constexpr int RGROUPS = TEAM / G::PANELS;      // warps that share a panel
    constexpr int TSTEPS = NY / G::RG;             // warp steps of a panel
    constexpr int MY = TSTEPS / RGROUPS;           // ... of this warp
    static_assert(TEAM > 1 && TEAM % G::PANELS == 0 && RGROUPS > 1 && TSTEPS % RGROUPS == 0, "unsupported team size");
    static_assert(MY * G::BPS == Scratch<NB, NX, NY, TEAM>::TEAM_NBLK, "table size");
    const int pan = tw % G::PANELS, rgp = tw / G::PANELS;
    const int a = lane % G::GPR, b = lane / G::GPR;
    const int off0 = (2 * b) * NX + pan * G::PW + 4 * a;   // the lane's block of warp step 0
    if (exps) *exps += cf.nexp;
    float2 s0 = make_float2(0.f, 0.f), s1 = make_float2(0.f, 0.f);
    if (cf.fast) {
        // blocks jb of the table: warp step (jb / BPS) * RGROUPS + rgp, block jb % BPS
        build_row_table<NB, NX, NY, RGROUPS>(rt, cf, lane, 0, rgp);
        LaneK<NB> lk;
        read_consts<NB, NX>(lk, team_ct + pan * Scratch<NB, NX, NY, TEAM>::CT, cf, lane, pan);   // team_consts wrote it
#pragma unroll(MY < 4 ? MY : 2)
        for (int m = 0; m < MY; ++m) {
            const int so = (m * RGROUPS + rgp) * G::RG * NX;
            StepPtrs sp{rt + (m * G::BPS + b) * T::RS, d + off0 + so, w + off0 + so, nullptr, 0u, 0.f};
            int i = 0;
            row_steps_fast<NB, NX, NY, false, true, 2>(cf, lk, s0, s1, i, 1, sp);
        }
    } else {
        float2 xd[K][2];   // column offsets of the lane's pixel pairs (0,1) and (2,3)
        const float fa = (float)(pan * G::PW + 4 * a);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const float2 nx0 = make_float2(-cf.x0[k], -cf.x0[k]);
            xd[k][0] = __fadd2_rn(make_float2(fa, fa + 1.f), nx0);
            xd[k][1] = __fadd2_rn(make_float2(fa + 2.f, fa + 3.f), nx0);
        }
#pragma unroll 1
        for (int m = 0; m < MY; ++m) {
            const int st = m * RGROUPS + rgp;
            const int so = st * G::RG * NX;
            StepPtrs sp{nullptr, d + off0 + so, w + off0 + so, nullptr, 0u, (float)(st * G::RG + 2 * b)};
            int i = 0;
            row_steps<NB, NX, NY, false, true>(cf, xd, s0, s1, i, 1, sp);
        }
    }
    return warp_sum_f64((double)((s0.x + s0.y) + (s1.x + s1.y)));
}

// Two parameter vectors per pass on a 32-pixel stamp (Geo<NX, 2>): every lane holds the coefficients
// of ITS half warp's vector; tables, lane constants, loop and reduction are shared instruction
// streams.  Returns, in every lane, chi-square of the vector of the lane's half warp.  A vector
// outside the safe range of the factorised loop (set_fast) takes the plain loop as it would alone:
// if the two halves disagree both loops run and each half keeps its own result, so chi-square and
// model image stay pure functions of the vector, whatever it is paired with.
template <int NB, int NX, int NY, bool STORE, bool PREP, int TM = 0>
__device__ __forceinline__ double warp_chi2_pair(const Coef<NB>& cf, float* __restrict__ scratch,
                                                 const float* __restrict__ d, const float* __restrict__ w,
                                                 float* __restrict__ model_out, int lane, unsigned* exps = nullptr,
                                                 uint32_t tmem = 0) {
    using G = Geo<NX, 2>;
    using T = Tab<NB>;
    using S = Scratch<NB, NX, NY, 1, 2>;
    constexpr int K = 2 * NB;
    constexpr int STEPS = NY / G::RG;
    static_assert(NX == 32 && NY == 32 && G::PANELS == 1, "two vectors per pass: 32 x 32 stamps");
    static_assert(TM == 0 || PREP, "the TMEM pixel store holds prepared stamps");
    const int wl = lane % G::LPW, h = lane / G::LPW, a = wl % G::GPR, b = wl / G::GPR;
    float* rt = scratch;
    float* ct = scratch + S::TAB;
    if (exps) *exps += cf.nexp;
    const bool run_fast = __any_sync(kFull, cf.fast), run_plain = __any_sync(kFull, !cf.fast);
    const int off0 = (2 * b) * NX + 4 * a;        // the lane's block of warp step 0
    float2 s0 = make_float2(0.f, 0.f), s1 = make_float2(0.f, 0.f);
    if (run_fast) {
        build_row_table<NB, NX, NY, 1, 2>(rt, cf, lane, 0, 0);
        LaneK<NB> lk;
        coop_consts<NB, NX, 2>(lk, ct, cf, lane, 0);
        float2 f0 = make_float2(0.f, 0.f), f1 = make_float2(0.f, 0.f);
        StepPtrs sp{rt + h * S::TAB1 + b * T::RS, d + off0, w + off0, STORE ? model_out + off0 : nullptr, tmem, 0.f};
        int i = 0;
        row_steps_fast<NB, NX, NY, STORE, PREP, 2, TM, 2>(cf, lk, f0, f1, i, STEPS, sp, cf.fast);
        if (cf.fast) { s0 = f0; s1 = f1; }
    }
    if (run_plain) {
        float2 xd[K][2];
        const float fa = (float)(4 * a);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const float2 nx0 = make_float2(-cf.x0[k], -cf.x0[k]);
            xd[k][0] = __fadd2_rn(make_float2(fa, fa + 1.f), nx0);
            xd[k][1] = __fadd2_rn(make_float2(fa + 2.f, fa + 3.f), nx0);
        }
        float2 p0 = make_float2(0.f, 0.f), p1 = make_float2(0.f, 0.f);
#pragma unroll 1
        for (int st = 0; st < STEPS; ++st) {
            const int so = st * G::RG * NX;
            StepPtrs sp{nullptr, d + off0 + so, w + off0 + so, STORE ? model_out + off0 + so : nullptr,
                        TM == 1 ? tmem + (uint32_t)(st * 16) : 0u, (float)(st * G::RG + 2 * b)};
            int i = 0;
            row_steps<NB, NX, NY, STORE, PREP, 2, (TM == 1 ? 1 : 0)>(cf, xd, p0, p1, i, 1, sp, !cf.fast);
        }
        if (!cf.fast) { s0 = p0; s1 = p1; }
    }
    double acc = (double)((s0.x + s0.y) + (s1.x + s1.y));
#pragma unroll
    for (int off = G::LPW / 2; off >= 1; off >>= 1) acc += shfl_xor_f64(acc, off);     // within the half warp
    return acc;
}

// Copy of the prepared stamp into the TMEM pixel store: called by warps 0..3 (one per TMEM lane
// quadrant) after prep_stamp; warp step i of the lane goes to columns 16 i .. 16 i + 15 in the
// order the loop consumes them (data row 0, data row 1, weight row 0, weight row 1).
template <int NX, int NY, int WPP = 1>
__device__ __forceinline__ void tmem_fill_stamp(uint32_t tmem_base, const float* __restrict__ sd,
                                                const float* __restrict__ sw, int warp, int lane) {
    using G = Geo<NX, WPP>;
    static_assert(G::PANELS == 1, "one panel");
    const int a = (lane % G::LPW) % G::GPR, b = (lane % G::LPW) / G::GPR;      // both half warps hold the same pixels
    const uint32_t addr = tmem_base + ((uint32_t)(32 * warp) << 16);
#pragma unroll 1
    for (int i = 0; i < NY / G::RG; ++i) {
        const int o = (i * G::RG + 2 * b) * NX + 4 * a;
        const float4 d0 = *reinterpret_cast<const float4*>(sd + o);
        const float4 d1 = *reinterpret_cast<const float4*>(sd + o + NX);
        const float4 w0 = *reinterpret_cast<const float4*>(sw + o);
        const float4 w1 = *reinterpret_cast<const float4*>(sw + o + NX);
        const float v[16] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w, w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
        tmem_st16(addr + 16 * i, v);
    }
    tmem_wait_st();
}

// 128-pixel stamps: only the weight plane fits (8 columns per warp step, 2 tables x 2 panels x 16
// steps = 512 columns, the whole TMEM); the data plane stays in shared memory.  Same order as the
// loop nest of warp_chi2: table, panel, warp step.
template <int NX, int NY>
__device__ __forceinline__ void tmem_fill_weights(uint32_t tmem_base, const float* __restrict__ sw, int warp, int lane) {
    using G = Geo<NX>;
    using R = Rows<NY, 1>;
    constexpr int STEPS = R::TR / G::RG;
    static_assert(R::HALVES * G::PANELS * STEPS * 8 <= 512, "weight plane exceeds the TMEM columns");
    const int a = lane % G::GPR, b = lane / G::GPR;
    const uint32_t addr = tmem_base + ((uint32_t)(32 * warp) << 16);
#pragma unroll 1
    for (int hp = 0; hp < R::HALVES * G::PANELS; ++hp) {
        const int half = hp / G::PANELS, pan = hp % G::PANELS;
#pragma unroll 1
        for (int i = 0; i < STEPS; ++i) {
            const int o = (half * R::TR + i * G::RG + 2 * b) * NX + pan * G::PW + 4 * a;
            const float4 w0 = *reinterpret_cast<const float4*>(sw + o);
            const float4 w1 = *reinterpret_cast<const float4*>(sw + o + NX);
            const float v[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
            tmem_st8(addr + (uint32_t)((hp * STEPS + i) * 8), v);
        }
    }
    tmem_wait_st();
}

// In-place conversion of a staged stamp to (d*sqrt(w), -sqrt(w)); called by the whole CTA.
__device__ __forceinline__ void prep_stamp(float* __restrict__ sd, float* __restrict__ sw, int n) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float r = sqrtf(sw[i]);
        sw[i] = -r;
        sd[i] *= r;
    }
}

// ---------------------------------------------------------------------------------------------
// Random stream
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kPhiloxM0 = 0xD2511F53u, kPhiloxM1 = 0xCD9E8D57u;
constexpr uint32_t kPhiloxW0 = 0x9E3779B9u, kPhiloxW1 = 0xBB67AE85u;
constexpr uint32_t kPhiloxTag = 0x4C415046u;   // 'LAPF'

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t hi0 = __umulhi(kPhiloxM0, c.x), lo0 = kPhiloxM0 * c.x;
        const uint32_t hi1 = __umulhi(kPhiloxM1, c.z), lo1 = kPhiloxM1 * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += kPhiloxW0;
        k.y += kPhiloxW1;
    }
    return c;
}

// The draws of update t of one walker, in the reference's order: parameter index
// (apf_step2.py:302), one standard normal (:64/:68), one uniform (:143).
struct Draw {
    int k;        // parameter index
    double z;     // standard normal
    double lnu;   // log of the uniform (-inf when the uniform is 0)
};

// Per-warp sampler scratch in shared memory: the staged trial vector, the random numbers of the
// next 32 updates (one update per lane, read back as broadcasts) and the shapes of the current
// state.  Keeping these out of registers leaves the register file to the pixel loop.
struct WarpScratch {
    float tf[32];        // staged trial vector (stage_trial)
    double step[32];     // proposal step of update slot i: w*z, or 10^(w*z) for log10 parameters
    double lnu[32];      // log of the accept/reject uniform of update slot i
    int k[32];           // parameter index of update slot i
    int dslot[32];       // posterior draws: reservoir slot (or -1) of the recorded row r at [r & 31]
    float shape[8];      // sa0 sb0 sc0 - sa1 sb1 sc1 -  of the CURRENT state
    float trig[4];       // sin, cos of theta (narrow), sin, cos of theta2 (wide) of the CURRENT state
};

__device__ __forceinline__ Draw make_draw(uint64_t seed, uint64_t walker_id, uint64_t t, int nparam) {
    const uint4 r = philox4x32_10(
        make_uint4((uint32_t)t, (uint32_t)(t >> 32), (uint32_t)(seed >> 32), kPhiloxTag),
        make_uint2((uint32_t)seed, (uint32_t)walker_id));
    Draw d;
    d.k = (int)__umulhi(r.x, (uint32_t)nparam);
    // Box-Muller from two full 32-bit words: |z| reaches 6.66 sigma
    const double u1 = ((double)r.y + 1.0) * 0x1p-32;         // (0, 1]
    const double u2 = (double)r.z * 0x1p-32;                 // [0, 1)
    d.z = sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
    // the accept/reject uniform carries 53 bits like numpy's rand() (apf_step2.py:143): the fourth
    // word and the low 21 bits of the first, whose high bits picked the parameter
    const uint64_t m = ((uint64_t)r.w << 21) | (uint64_t)(r.x & 0x1FFFFFu);
    const double u = (double)m * 0x1p-53;                    // [0, 1)
    d.lnu = log(u);                                          // -inf for u = 0 (probability 2^-53)
    return d;
}

// Posterior draws (DESIGN.md 4, "Posterior draws"): the reservoir slot that recorded row n of walker
// walker_id takes among K, or -1 -- algorithm R.  Rows n < K fill slot n; row n >= K replaces slot
// j = mulhi64(r, n + 1) if j < K, r the 64-bit word of its own Philox stream (tag 'LAPR', so the
// update stream is untouched).  Integer-only, so the host restates it bit for bit; mulhi64 without
// rejection favours some j by at most (n + 1) / 2^64.
constexpr uint32_t kPhiloxTagDraws = 0x4C415052u;   // 'LAPR'

__device__ __forceinline__ int draw_slot(uint64_t seed, uint64_t walker_id, uint64_t n, int K) {
    if (n < (uint64_t)K) return (int)n;
    const uint4 r = philox4x32_10(
        make_uint4((uint32_t)n, (uint32_t)(n >> 32), (uint32_t)(seed >> 32), kPhiloxTagDraws),
        make_uint2((uint32_t)seed, (uint32_t)walker_id));
    const uint64_t j = __umul64hi(((uint64_t)r.y << 32) | r.x, n + 1);
    return j < (uint64_t)K ? (int)j : -1;
}

}  // namespace lapf
