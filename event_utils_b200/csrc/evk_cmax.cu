// evk_cmax.cu -- fused contrast-maximisation evaluation on B200:
//   warp -> bounds mask -> bilinear IWE (+ Jacobian-weighted derivative images) -> Gaussian
//   blur -> variance objective and its analytic gradient, one pass over the events.
//
// Semantics (reference):
//   linvel_warp.warp              lib/contrast_max/warps.py:51-61        (f64)
//   events_bounds_mask            lib/util/event_util.py:26-27           (f64)
//   get_iwe                       lib/contrast_max/objectives.py:184-192
//   events_to_image_drv           lib/representations/image.py:179-217   (f64 -> f32 cast, splat)
//   interpolate_to_derivative_img lib/representations/image.py:131-135
//   variance_objective            lib/contrast_max/objectives.py:231-236, 251-264
//   warp_events_flow_torch + IWE  lib/transforms/optic_flow.py:37-44, lib/visualization/draw_flow.py:18-21
//
// B200 design (DESIGN.md section 4):
//   * ONE pass over the events.  The accumulator is an array of 32-byte BLOCKS, one per pixel:
//     block (y,x) = {I_TL, I_TR, I_BL, I_BR, a, b, c, d} collects every event whose bilinear
//     footprint is anchored at (y,x) (each pixel therefore lives in four blocks; a gather kernel
//     folds them).  The 2x2 IWE footprint of an event is ONE red.global.add.v4.f32
//     (REDG.E.ADD.F32x4); the 8 derivative taps have only 4 free values (the taps of a derivative
//     image come in +/- pairs, image.py:131-135), so both derivative images are ONE more vector
//     reduction: 1 RED per event for f, 2 for f and g, instead of 4 / 12 scalar ones.  Measured:
//     every scatter kernel on B200 costs ~0.25 ms per RED lane-operation per 50 M events,
//     whatever its width (scalar, v2, v4) and whether or not lanes share a sector -- the count of
//     reduction operations is what has to be minimised.  The accumulator (181*241*32 B = 1.4 MB
//     per replica, R <= 8 replicas against same-address serialisation) never leaves L2.
//   * ON-CHIP IWE (round 2, large event counts): the whole 181x241 image of warped events is 174 KB -- it
//     fits in ONE SM's shared memory.  cmax_onchip_kernel runs one 1024-thread CTA per SM, each with a
//     PRIVATE fixed-point image in shared memory; the four bilinear taps are native integer shared-memory
//     atomics (ATOMS.ADD; measured: 4 per event are hidden under the HBM read of the events, while f32
//     shared atomics are CAS loops and L2 reductions cost ~0.3 ms per 50 M).  Fixed point = value * 2^22 in
//     a biased u32 cell; the RETURNING atomic tells the thread whether ITS add wrapped the 32-bit cell and
//     that thread carries +-2^10 out to the global accumulator, so the sum is exact integer arithmetic with
//     no overflow whatever the stream (per-tap quantisation 2^-23, below f32 rounding of the reference's
//     own accumulation).  Events with |p*mask| > 1 or non-finite weights take the global f32 path.  At
//     the end every CTA converts its image to f32 in place and adds it to a planar global image with TMA
//     bulk reductions (cp.reduce.async.bulk.global.shared::cta.add.f32, SASS UBLKRED) -- "finished tiles
//     leave through TMA".  The derivative images do not fit next to the IWE (3 x 174 KB), so with the
//     gradient their four free values per event remain ONE vector reduction to the L2 block accumulator.
//   * The reference blurs both derivative images and multiplies by the un-blurred IWE.  The
//     reflect-boundary Gaussian is self-adjoint, so  sum(2(I-mu) * G(D_k)) == sum(G(2(I-mu)) * D_k)
//     and G(2(I-mu)) = 2(G(I)-mu): ONE blur of ONE image (which f needs anyway) serves f and g.
//   * scipy blurs the (2,H,W) derivative stack along its length-2 axis as well
//     (objectives.py:253), mixing the two gradient components by [[a,b],[b,a]]; applied to the
//     two scalars at the end (host supplies a,b).
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "evk_common.cuh"

namespace evk {

constexpr int kMaxRadius = 64;
constexpr int kMaxReplicas = 8;
constexpr int kMaxCandidates = 32;  // parameter points per batched evaluation
constexpr int kBlockFloats = 8;   // one 32-byte block (= one L2 sector) per pixel: {I_TL, I_TR, I_BL, I_BR, a, b, c, d}

struct BlurTaps {
    int r;
    double w[kMaxRadius + 1];  // w[k] = weight at distance k (symmetric)
};

struct CmaxArgs {
    const void *x, *y, *t, *p;
    int64_t n;
    double vx, vy, t_ref;  // linvel
    double p_scale;        // polarity multiplier (objectives.py:225 uses 100)
    const float *flow;     // dense flow [2][Hs][Ws]
    const float2 *flow_uv; // the same, interleaved {u,v} per pixel (built per call in the workspace)
    float flow_t0;
    int Hm, Wm;  // bounds-mask size (img_size)
    int Hc, Wc;  // canvas = sensor + 1
    int abs_polarity;
    int replicas;
    float *acc;  // [R][Hc*Wc][8]
    int vec16;      // on-chip path: all four event arrays are 16-byte aligned
    float *planar;  // on-chip path: planar f32 image [npix padded to 4] the CTAs' shared-memory images are reduced into
    unsigned long long *oob;
    double params[8];  // rotation (cx, cy, omega) / xyztheta (vx, vy, vz, omega)
};

enum { WARP_LINVEL_F64 = 0, WARP_LINVEL_F32 = 1, WARP_FLOW_F32 = 2, WARP_ROT_F64 = 3, WARP_ROT_F32 = 4, WARP_XYZT_F64 = 5, WARP_XYZT_F32 = 6 };
__host__ __device__ constexpr bool is_model(int w) { return w >= WARP_ROT_F64; }

// bilinear splat of weight w (and derivative weight a) at (xf, yf) on the canvas:
// image.py:199-207 (IWE) and :131-135 (derivative images) with w1 = [a;0], w2 = [0;a].
// PAIR: two adjacent lanes carry the SAME event; lane parity `xt` picks the x tap (x0 or x0+1) and
// the lane issues the two row taps of that column.  The two lanes of a pair then write 32
// contiguous bytes (pixels x0, x0+1 of the interleaved accumulator) in the same instruction, which
// the LSU merges into one L2 request per row: half the L2 tag look-ups of the one-lane-per-event
// form (the measured limiter, lts__t_tag_requests ~75 % of peak).
struct Taps {
    int x0, x1, y0, y1;
    float wm;     // masked weight (|wm| <= 1 is the fast-path condition of the on-chip image)
    float4 ti;    // IWE taps TL, TR, BL, BR
    float4 td;    // free values of the derivative taps: a = am*oy, b = am*dy, c = am*ox, d = am*dx
};

// The arithmetic of one bilinear splat (image.py:199-207, :131-135), shared by the two accumulator back ends.
// Returns false when the event contributes nothing (out of the canvas -> counted, or all-zero weights).
template <bool GRAD>
__device__ __forceinline__ bool splat_taps(const CmaxArgs &A, float xf, float yf, float w, float a, bool clip, unsigned &oob, Taps &T)
{
    const float clipx = (float)(A.Wc - 1), clipy = (float)(A.Hc - 1);
    float m2 = 1.0f;
    if (clip) m2 = (xf >= clipx ? 0.0f : 1.0f) * (yf >= clipy ? 0.0f : 1.0f);
    const float pxf = floorf(xf), pyf = floorf(yf);
    const float dx = __fsub_rn(xf, pxf), dy = __fsub_rn(yf, pyf);
    int upx, upy;
    if (!trunc_checked(__fmul_rn(pxf, m2), upx) || !trunc_checked(__fmul_rn(pyf, m2), upy) ||
        !wrap_int_index(upx, A.Wc, T.x0) || !wrap_int_index(upx + 1, A.Wc, T.x1) ||
        !wrap_int_index(upy, A.Hc, T.y0) || !wrap_int_index(upy + 1, A.Hc, T.y1)) { ++oob; return false; }
    const float wm = __fmul_rn(w, m2);
    const float am = GRAD ? __fmul_rn(a, wm) : 0.0f;  // jacobian * masked_ps (image.py:211-212)
    if (wm == 0.0f && am == 0.0f) return false;
    const float ox = __fsub_rn(1.0f, dx), oy = __fsub_rn(1.0f, dy);
    const float wl = __fmul_rn(wm, ox), wr = __fmul_rn(wm, dx);
    T.wm = wm;
    // tap order inside a block: TL (y0,x0), TR (y0,x1), BL (y1,x0), BR (y1,x1)
    T.ti = make_float4(__fmul_rn(wl, oy), __fmul_rn(wr, oy), __fmul_rn(wl, dy), __fmul_rn(wr, dy));
    // image.py:131-135 with w1 = [am;0], w2 = [0;am]:
    //   D0 taps = am*{-oy, +oy, -dy, +dy}   -> TL = -TR, BL = -BR : two free values a = am*oy, b = am*dy
    //   D1 taps = am*{-ox, -dx, +ox, +dx}   -> TL = -BL, TR = -BR : two free values c = am*ox, d = am*dx
    // (negation is exact and commutes with the sums, so accumulating a,b,c,d and restoring the
    // signs in the fold gives the same images) -> both derivative images are ONE vector reduction.
    T.td = make_float4(0.f, 0.f, 0.f, 0.f);
    if (GRAD) T.td = make_float4(__fmul_rn(am, oy), __fmul_rn(am, dy), __fmul_rn(am, ox), __fmul_rn(am, dx));
    return true;
}

// taps -> the global block accumulator.  WANT_I / WANT_D select the image taps and the derivative values.
template <bool WANT_I, bool WANT_D>
__device__ __forceinline__ void emit_global(const CmaxArgs &A, float *acc, const Taps &T)
{
    if (T.x1 == T.x0 + 1 && T.y1 == T.y0 + 1) {
        float *blk = acc + ((int64_t)T.y0 * A.Wc + T.x0) * kBlockFloats;
        if (WANT_I) red_add4(blk, T.ti);
        if (WANT_D) red_add4(blk + 4, T.td);
        return;
    }
    // wrapped footprint (negative coordinates, only reachable without the bounds mask): every tap
    // becomes the TL tap of its own pixel's block (TL of D0 is -a, TL of D1 is -c)
    const float vi[4] = {T.ti.x, T.ti.y, T.ti.z, T.ti.w};
    const float v0[4] = {-T.td.x, T.td.x, -T.td.y, T.td.y}, v1[4] = {-T.td.z, -T.td.w, T.td.z, T.td.w};
    const int ys[4] = {T.y0, T.y0, T.y1, T.y1}, xs[4] = {T.x0, T.x1, T.x0, T.x1};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        float *bk = acc + ((int64_t)ys[k] * A.Wc + xs[k]) * kBlockFloats;
        if (WANT_I && vi[k] != 0.0f) red_add(bk, vi[k]);
        if (WANT_D && v0[k] != 0.0f) red_add(bk + 4, -v0[k]);
        if (WANT_D && v1[k] != 0.0f) red_add(bk + 6, -v1[k]);
    }
}

// bilinear splat of weight w (and derivative weight a) at (xf, yf) on the canvas, L2 back end
template <bool GRAD>
__device__ __forceinline__ void splat(const CmaxArgs &A, float *acc, float xf, float yf, float w, float a,
                                      bool clip, unsigned &oob)
{
    Taps T;
    if (!splat_taps<GRAD>(A, xf, yf, w, a, clip, oob, T)) return;
    emit_global<true, GRAD>(A, acc, T);
}

// ---- on-chip back end: the IWE lives in the CTA's shared memory as biased fixed point ----------------
constexpr int kFixBits = 22;
constexpr float kFixScale = (float)(1 << kFixBits);
constexpr float kFixCarry = (float)(1u << (32 - kFixBits));   // value of one 2^32 wrap of a cell
constexpr unsigned kFixBias = 0x80000000u;

__device__ __forceinline__ unsigned atoms_add_ret(unsigned *cell, unsigned v)
{
    unsigned old;
    asm volatile("atom.relaxed.cta.shared::cta.add.u32 %0, [%1], %2;" : "=r"(old) : "r"((unsigned)__cvta_generic_to_shared(cell)), "r"(v));
    return old;
}

// Did adding the signed increment q to the biased cell (old -> old + q mod 2^32) wrap the 32 bits?  A wrap flips the
// top bit TOWARDS the sign of q (carry: 1 -> 0 with q >= 0; borrow: 0 -> 1 with q < 0); the other top-bit flip is the
// true value crossing zero.  Bit 31 of the result is the answer; q == 0 never wraps.
__device__ __forceinline__ unsigned wrap_bit(unsigned old, unsigned q) { const unsigned nw = old + q; return (old ^ nw) & ~(nw ^ q); }

// The four taps of one event: four independent native shared-memory atomics, ONE rarely taken branch.
// A wrap of a cell is carried to the global accumulator (TL slot of the pixel's own block, which the fold
// adds to the pixel), so the total is exact integer arithmetic for any event count.
__device__ __forceinline__ void onchip_taps(unsigned *simg, float *acc, int p00, int p01, int p10, int p11, float4 ti)
{
    const unsigned q0 = (unsigned)__float2int_rn(__fmul_rn(ti.x, kFixScale));   // |tap| <= 1 -> |q| <= 2^22
    const unsigned q1 = (unsigned)__float2int_rn(__fmul_rn(ti.y, kFixScale));
    const unsigned q2 = (unsigned)__float2int_rn(__fmul_rn(ti.z, kFixScale));
    const unsigned q3 = (unsigned)__float2int_rn(__fmul_rn(ti.w, kFixScale));
    const unsigned o0 = atoms_add_ret(simg + p00, q0), o1 = atoms_add_ret(simg + p01, q1);
    const unsigned o2 = atoms_add_ret(simg + p10, q2), o3 = atoms_add_ret(simg + p11, q3);
    const unsigned w0 = wrap_bit(o0, q0), w1 = wrap_bit(o1, q1), w2 = wrap_bit(o2, q2), w3 = wrap_bit(o3, q3);
    if ((w0 | w1 | w2 | w3) >> 31) {
        if (w0 >> 31) red_add(acc + (int64_t)p00 * kBlockFloats, (int)q0 >= 0 ? kFixCarry : -kFixCarry);
        if (w1 >> 31) red_add(acc + (int64_t)p01 * kBlockFloats, (int)q1 >= 0 ? kFixCarry : -kFixCarry);
        if (w2 >> 31) red_add(acc + (int64_t)p10 * kBlockFloats, (int)q2 >= 0 ? kFixCarry : -kFixCarry);
        if (w3 >> 31) red_add(acc + (int64_t)p11 * kBlockFloats, (int)q3 >= 0 ? kFixCarry : -kFixCarry);
    }
}

template <bool GRAD>
__device__ __forceinline__ void splat_onchip(const CmaxArgs &A, float *acc, unsigned *simg, float xf, float yf, float w, float a,
                                             bool clip, unsigned &oob)
{
    Taps T;
    if (!splat_taps<GRAD>(A, xf, yf, w, a, clip, oob, T)) return;
    if (fabsf(T.wm) <= 1.0f) {      // false for NaN / inf as well
        const int r0 = T.y0 * A.Wc, r1 = T.y1 * A.Wc;
        onchip_taps(simg, acc, r0 + T.x0, r0 + T.x1, r1 + T.x0, r1 + T.x1, T.ti);
        if (GRAD) emit_global<false, true>(A, acc, T);
    } else {
        emit_global<true, GRAD>(A, acc, T);
    }
}

// One event's four components as loaded (f64 in parity mode, f32 otherwise).
template <int WARP> struct EvT { using type = float; };
template <> struct EvT<WARP_LINVEL_F64> { using type = double; };
template <> struct EvT<WARP_ROT_F64> { using type = double; };
template <> struct EvT<WARP_XYZT_F64> { using type = double; };

// ---- the rotation and xyztheta motion models (contrast_max/warps.py, include/evk.h) ----------------------
// d = t - t_ref (f64 parity mode) or the stored t - t_last (f32 fast mode); T is the event precision.
//   rotation  (cx, cy, omega), th = -omega d:  x' = cx + cos th (x - cx) - sin th (y - cy)
//                                              y' = cy + sin th (x - cx) + cos th (y - cy)
//             dx'/dp = (1 - cos th,  sin th,  d (y' - cy)),  dy'/dp = (-sin th, 1 - cos th, -d (x' - cx))
//   xyztheta  (vx, vy, vz, omega):  x' = x - d (vx + vz x - omega y),  y' = y - d (vy + vz y + omega x)
//             dx'/dp = (-d, 0, -d x, d y),  dy'/dp = (0, -d, -d y, -d x)
// The operation order is the numpy order of warps.py (the library is built without FMA contraction).
template <int WARP> struct Model {
    static constexpr bool rot = (WARP == WARP_ROT_F64 || WARP == WARP_ROT_F32);
    static constexpr int dims = rot ? 3 : 4;
    using T = typename EvT<WARP>::type;
};

template <int WARP, bool JAC>
__device__ __forceinline__ void model_warp(const CmaxArgs &A, typename Model<WARP>::T x, typename Model<WARP>::T y,
                                           typename Model<WARP>::T d, typename Model<WARP>::T &xw, typename Model<WARP>::T &yw,
                                           typename Model<WARP>::T *jx, typename Model<WARP>::T *jy)
{
    using T = typename Model<WARP>::T;
    if constexpr (Model<WARP>::rot) {
        const T cx = (T)A.params[0], cy = (T)A.params[1], om = (T)A.params[2];
        const T th = -(om * d);
        T s, c;
        if constexpr (sizeof(T) == 8) sincos(th, &s, &c); else sincosf(th, &s, &c);
        const T X = x - cx, Y = y - cy;
        xw = cx + c * X - s * Y;
        yw = cy + s * X + c * Y;
        if (JAC) {
            jx[0] = (T)1 - c; jx[1] = s; jx[2] = d * (yw - cy);
            jy[0] = -s; jy[1] = (T)1 - c; jy[2] = -(d * (xw - cx));
        }
    } else {
        const T vx = (T)A.params[0], vy = (T)A.params[1], vz = (T)A.params[2], om = (T)A.params[3];
        xw = x - d * (vx + vz * x - om * y);
        yw = y - d * (vy + vz * y + om * x);
        if (JAC) {
            jx[0] = -d; jx[1] = (T)0; jx[2] = -(d * x); jx[3] = d * y;
            jy[0] = (T)0; jy[1] = -d; jy[2] = -(d * y); jy[3] = -(d * x);
        }
    }
}

// The polarity, time offset, warp and bounds mask of one event of a model (as the linvel branch of cmax_event).
// Returns false when the mask drops the event.
template <int WARP, bool JAC>
__device__ __forceinline__ bool model_event(const CmaxArgs &A, typename Model<WARP>::T x, typename Model<WARP>::T y,
                                            typename Model<WARP>::T t, typename Model<WARP>::T &p, typename Model<WARP>::T &xw,
                                            typename Model<WARP>::T &yw, typename Model<WARP>::T *jx, typename Model<WARP>::T *jy)
{
    using T = typename Model<WARP>::T;
    if (A.p_scale != 1.0) p = p * (T)A.p_scale;
    if (A.abs_polarity) p = fabs(p);
    const T d = (sizeof(T) == 8) ? t - (T)A.t_ref : t;
    model_warp<WARP, JAC>(A, x, y, d, xw, yw, jx, jy);
    // event_util.py:26-27: keep iff 0 < x' <= Wm and 0 < y' <= Hm (NaN compares false -> kept)
    return !(xw <= (T)0 || xw > (T)A.Wm) && !(yw <= (T)0 || yw > (T)A.Hm);
}

template <int WARP>
struct Event {
    typename EvT<WARP>::type x, y, t, p;
};

template <int WARP>
__device__ __forceinline__ Event<WARP> load_event(const CmaxArgs &A, int64_t i)
{
    using T = typename EvT<WARP>::type;
    Event<WARP> e;
    e.x = ld_stream((const T *)A.x + i);
    e.y = ld_stream((const T *)A.y + i);
    e.t = ld_stream((const T *)A.t + i);
    e.p = ld_stream((const T *)A.p + i);
    return e;
}

__device__ __forceinline__ void ld_vec16(const float *p, float (&v)[4])
{
    const float4 q = ld_stream4(p);
    v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
}
__device__ __forceinline__ void ld_vec16(const double *p, double (&v)[2])
{
    const double2 q = ld_stream2(p);
    v[0] = q.x; v[1] = q.y;
}

template <int WARP, bool GRAD, bool ONCHIP = false>
__device__ __forceinline__ void cmax_event(const CmaxArgs &A, float *acc, const Event<WARP> &e, unsigned &oob, double cvx,
                                           double cvy, unsigned *simg = nullptr)
{
    if constexpr (is_model(WARP)) {
        // pass 1 of a model: the IWE only (the gradient is cmax_model_grad_kernel's second pass)
        typename Model<WARP>::T p = e.p, xw, yw;
        if (!model_event<WARP, false>(A, e.x, e.y, e.t, p, xw, yw, nullptr, nullptr)) return;
        if (ONCHIP) splat_onchip<false>(A, acc, simg, (float)xw, (float)yw, (float)p, 0.0f, true, oob);
        else splat<false>(A, acc, (float)xw, (float)yw, (float)p, 0.0f, true, oob);
        return;
    }
    if (WARP == WARP_LINVEL_F64) {
        const double x = e.x, y = e.y, t = e.t;
        double p = e.p;
        if (A.p_scale != 1.0) p = __dmul_rn(p, A.p_scale);
        if (A.abs_polarity) p = fabs(p);
        const double d = __dsub_rn(t, A.t_ref);
        const double xw = __dsub_rn(x, __dmul_rn(d, cvx));  // warps.py:52-54
        const double yw = __dsub_rn(y, __dmul_rn(d, cvy));
        // event_util.py:26-27: keep iff 0 < x' <= Wm and 0 < y' <= Hm (NaN compares false -> kept)
        const bool keep = !(xw <= 0.0 || xw > (double)A.Wm) && !(yw <= 0.0 || yw > (double)A.Hm);
        if (!keep) return;  // x,y,p,j all multiplied by 0: only exact zeros are added at (0,0)..(1,1)
        if (ONCHIP) splat_onchip<GRAD>(A, acc, simg, (float)xw, (float)yw, (float)p, (float)(-d), true, oob);
        else splat<GRAD>(A, acc, (float)xw, (float)yw, (float)p, (float)(-d), true, oob);  // image.py:180-183 casts
    } else if (WARP == WARP_LINVEL_F32) {
        const float x = e.x, y = e.y;
        const float d = e.t;  // already t - t_ref
        float p = e.p;
        if (A.p_scale != 1.0) p = __fmul_rn(p, (float)A.p_scale);
        if (A.abs_polarity) p = fabsf(p);
        const float vx = (float)cvx, vy = (float)cvy;
        const float xw = __fsub_rn(x, __fmul_rn(d, vx)), yw = __fsub_rn(y, __fmul_rn(d, vy));
        const bool keep = !(xw <= 0.0f || xw > (float)A.Wm) && !(yw <= 0.0f || yw > (float)A.Hm);
        if (!keep) return;
        if (ONCHIP) splat_onchip<GRAD>(A, acc, simg, xw, yw, p, -d, true, oob);
        else splat<GRAD>(A, acc, xw, yw, p, -d, true, oob);
    } else {
        // optic_flow.py:37-44 then events_to_image_torch(..., interpolation='bilinear') defaults
        const float xe = e.x, ye = e.y, te = e.t;
        float p = e.p;
        if (A.abs_polarity) p = fabsf(p);
        const int H = A.Hc - 1, W = A.Wc - 1;
        const float wm1 = (float)(W - 1), hm1 = (float)(H - 1);
        const float gx = __fsub_rn(__fmul_rn(__fdiv_rn(xe, wm1), 2.0f), 1.0f);
        const float gy = __fsub_rn(__fmul_rn(__fdiv_rn(ye, hm1), 2.0f), 1.0f);
        const float ix = __fmul_rn(__fdiv_rn(__fadd_rn(gx, 1.0f), 2.0f), wm1);
        const float iy = __fmul_rn(__fdiv_rn(__fadd_rn(gy, 1.0f), 2.0f), hm1);
        float u = 0.0f, v = 0.0f;
        if (fabsf(ix) < 1.0e9f && fabsf(iy) < 1.0e9f) {
            const float fx = floorf(ix), fy = floorf(iy);
            const int x0 = (int)fx, y0 = (int)fy;
            const float xs = fx + 1.0f, ys = fy + 1.0f;
            const float nw = __fmul_rn(__fsub_rn(xs, ix), __fsub_rn(ys, iy));
            const float ne = __fmul_rn(__fsub_rn(ix, fx), __fsub_rn(ys, iy));
            const float sw = __fmul_rn(__fsub_rn(xs, ix), __fsub_rn(iy, fy));
            const float se = __fmul_rn(__fsub_rn(ix, fx), __fsub_rn(iy, fy));
            const float4 top = flow_row<true>(A.flow, A.flow_uv, H, W, y0, x0), bot = flow_row<true>(A.flow, A.flow_uv, H, W, y0 + 1, x0);
            u = __fadd_rn(u, __fmul_rn(top.x, nw)); v = __fadd_rn(v, __fmul_rn(top.y, nw));
            u = __fadd_rn(u, __fmul_rn(top.z, ne)); v = __fadd_rn(v, __fmul_rn(top.w, ne));
            u = __fadd_rn(u, __fmul_rn(bot.x, sw)); v = __fadd_rn(v, __fmul_rn(bot.y, sw));
            u = __fadd_rn(u, __fmul_rn(bot.z, se)); v = __fadd_rn(v, __fmul_rn(bot.w, se));
        }
        const float d = __fsub_rn(te, A.flow_t0);
        if (ONCHIP) splat_onchip<false>(A, acc, simg, __fadd_rn(xe, __fmul_rn(u, d)), __fadd_rn(ye, __fmul_rn(v, d)), p, 0.0f, true, oob);
        else splat<false>(A, acc, __fadd_rn(xe, __fmul_rn(u, d)), __fadd_rn(ye, __fmul_rn(v, d)), p, 0.0f, true, oob);
    }
}

// The event pass.  Memory-level parallelism matters as much as the reductions here: each thread
// first issues the loads of kBatch events (16 independent loads in flight), then warps and
// splats them (a load -> compute -> red chain per event ran at ~0.9 ms / 50 M events whatever
// the number of reductions).
constexpr int kBatch = 4;

template <int WARP, bool GRAD>
__global__ void __launch_bounds__(256) cmax_scatter_kernel(const CmaxArgs A)
{
    unsigned oob = 0;
    float *acc = A.acc + (int64_t)(blockIdx.x % A.replicas) * A.Hc * A.Wc * kBlockFloats;
    const int64_t stride = (int64_t)gridDim.x * 256;
    int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    for (; i + (kBatch - 1) * stride < A.n; i += kBatch * stride) {
        Event<WARP> ev[kBatch];
#pragma unroll
        for (int k = 0; k < kBatch; ++k) ev[k] = load_event<WARP>(A, i + k * stride);
#pragma unroll
        for (int k = 0; k < kBatch; ++k) cmax_event<WARP, GRAD>(A, acc, ev[k], oob, A.vx, A.vy);
    }
    for (; i < A.n; i += stride) cmax_event<WARP, GRAD>(A, acc, load_event<WARP>(A, i), oob, A.vx, A.vy);
    flush_oob(A.oob, oob);
}

// The on-chip event pass: one persistent 1024-thread CTA per SM, private fixed-point IWE in shared memory.
constexpr int kOnchipThreads = 1024;
constexpr int kBulkFloats = 4096;   // 16 KB per TMA bulk reduction

template <int WARP, bool GRAD>
__global__ void __launch_bounds__(kOnchipThreads, 1) cmax_onchip_kernel(const CmaxArgs A)
{
    extern __shared__ __align__(128) unsigned simg[];   // [npad] biased fixed point, then f32 in place
    const int npix = A.Hc * A.Wc, npad = (npix + 3) & ~3;
    for (int i = threadIdx.x; i < npad; i += kOnchipThreads) simg[i] = kFixBias;
    __syncthreads();
    unsigned oob = 0;
    // derivative reductions and carries go to the L2 block accumulator (replicas against same-address serialisation)
    float *acc = A.acc + (int64_t)(blockIdx.x % A.replicas) * A.Hc * A.Wc * kBlockFloats;
    const int64_t stride = (int64_t)gridDim.x * kOnchipThreads;
    int64_t i = (int64_t)blockIdx.x * kOnchipThreads + threadIdx.x;
    if (A.vec16) {
        // 16-byte loads: 4 f32 events / 2 f64 events per vector, two vectors of every array in flight per thread
        using T = typename EvT<WARP>::type;
        constexpr int EPV = 16 / (int)sizeof(T);
        const int64_t nv = A.n / EPV;
        const T *px = (const T *)A.x, *py = (const T *)A.y, *pt = (const T *)A.t, *pp = (const T *)A.p;
        for (int64_t v = i; v < nv; v += 2 * stride) {
            const bool two = v + stride < nv;
            const int64_t v2 = two ? v + stride : v;
            T ex[2][EPV], ey[2][EPV], et[2][EPV], ep[2][EPV];
            ld_vec16(px + v * EPV, ex[0]); ld_vec16(py + v * EPV, ey[0]); ld_vec16(pt + v * EPV, et[0]); ld_vec16(pp + v * EPV, ep[0]);
            ld_vec16(px + v2 * EPV, ex[1]); ld_vec16(py + v2 * EPV, ey[1]); ld_vec16(pt + v2 * EPV, et[1]); ld_vec16(pp + v2 * EPV, ep[1]);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                if (h == 1 && !two) break;
#pragma unroll
                for (int k = 0; k < EPV; ++k) {
                    Event<WARP> e;
                    e.x = ex[h][k]; e.y = ey[h][k]; e.t = et[h][k]; e.p = ep[h][k];
                    cmax_event<WARP, GRAD, true>(A, acc, e, oob, A.vx, A.vy, simg);
                }
            }
        }
        for (int64_t j = nv * EPV + i; j < A.n; j += stride) cmax_event<WARP, GRAD, true>(A, acc, load_event<WARP>(A, j), oob, A.vx, A.vy, simg);
    } else {
        constexpr int kB = sizeof(typename EvT<WARP>::type) == 8 ? 2 : 4;   // loads in flight per thread (64-register budget at 1024 threads)
        for (; i + (kB - 1) * stride < A.n; i += kB * stride) {
            Event<WARP> ev[kB];
#pragma unroll
            for (int k = 0; k < kB; ++k) ev[k] = load_event<WARP>(A, i + k * stride);
#pragma unroll
            for (int k = 0; k < kB; ++k) cmax_event<WARP, GRAD, true>(A, acc, ev[k], oob, A.vx, A.vy, simg);
        }
        for (; i < A.n; i += stride) cmax_event<WARP, GRAD, true>(A, acc, load_event<WARP>(A, i), oob, A.vx, A.vy, simg);
    }
    flush_oob(A.oob, oob);
    __syncthreads();
    // fixed point -> f32 in place (an int32 sum rounds to f32 once, like a float accumulator's final value)
    float *fimg = reinterpret_cast<float *>(simg);
    for (int j = threadIdx.x; j < npad; j += kOnchipThreads)
        fimg[j] = __fmul_rn((float)(int)(simg[j] - kFixBias), 1.0f / kFixScale);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the TMA engine
    __syncthreads();
    // the finished image leaves through TMA: bulk add-reductions of 16 KB pieces into the planar global image
    if ((threadIdx.x & 31) == 0) {
        for (int c = threadIdx.x >> 5; c * kBulkFloats < npad; c += kOnchipThreads / 32) {
            const int off = c * kBulkFloats;
            const int cnt = (npad - off < kBulkFloats) ? (npad - off) : kBulkFloats;
            const unsigned src = (unsigned)__cvta_generic_to_shared(fimg + off);
            asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f32 [%0], [%1], %2;" ::"l"(
                             __cvta_generic_to_global(A.planar + off)), "r"(src), "r"(cnt * 4) : "memory");
        }
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // shared memory must outlive the engine's reads
    }
}

// ---- pass 2 of a model: the gradient in gather form -------------------------------------------------
// g_k = -c sum_j M[k][j] sum_pix W D_j, and the derivative images D_j are sums of per-event taps
// (image.py:131-135 with w1 = jx p, w2 = jy p), so by adjointness
//   sum_pix W D_j = sum_events p (jx_j Sx + jy_j Sy),   Sx = oy (W_TR - W_TL) + dy (W_BR - W_BL),
//                                                        Sy = ox (W_BL - W_TL) + dx (W_BR - W_TR)
// for the event's 2x2 footprint.  W (the blurred weight image of the objective, f32) sits in shared memory; the
// events are streamed a second time and every event costs four shared-memory loads and `dims` f64 FMAs -- no
// reductions, whatever the number of parameters.  One persistent CTA per SM.
constexpr int kGradThreads = 512;

template <int WARP>
__device__ __forceinline__ void grad_event(const CmaxArgs &A, const float *sw, typename Model<WARP>::T x, typename Model<WARP>::T y,
                                           typename Model<WARP>::T t, typename Model<WARP>::T p, double (&acc)[Model<WARP>::dims])
{
    using T = typename Model<WARP>::T;
    constexpr int D = Model<WARP>::dims;
    T xw, yw, jx[D], jy[D];
    if (!model_event<WARP, true>(A, x, y, t, p, xw, yw, jx, jy)) return;
    // the same f32 footprint as splat_taps (image.py:180-207); clipped events have zero weight, events outside
    // the canvas were counted by pass 1 (the evaluation then fails)
    const float xf = (float)xw, yf = (float)yw;
    if (xf >= (float)(A.Wc - 1) || yf >= (float)(A.Hc - 1)) return;
    const float pxf = floorf(xf), pyf = floorf(yf);
    int x0, y0;
    if (!trunc_checked(pxf, x0) || !trunc_checked(pyf, y0) || x0 < 0 || y0 < 0 || x0 + 1 >= A.Wc || y0 + 1 >= A.Hc) return;
    const float dx = __fsub_rn(xf, pxf), dy = __fsub_rn(yf, pyf);
    const float ox = __fsub_rn(1.0f, dx), oy = __fsub_rn(1.0f, dy);
    const float *r0 = sw + y0 * A.Wc + x0, *r1 = r0 + A.Wc;
    const double tl = r0[0], tr = r0[1], bl = r1[0], br = r1[1];
    const double sx = (double)oy * (tr - tl) + (double)dy * (br - bl);
    const double sy = (double)ox * (bl - tl) + (double)dx * (br - tr);
    const double pw = (double)(float)p;   // masked_ps after the f32 cast (image.py:180)
#pragma unroll
    for (int j = 0; j < D; ++j) acc[j] += pw * ((double)jx[j] * sx + (double)jy[j] * sy);
}

template <int WARP>
__global__ void __launch_bounds__(kGradThreads, 1) cmax_model_grad_kernel(const CmaxArgs A, const float *__restrict__ W, double *gk)
{
    using T = typename Model<WARP>::T;
    constexpr int D = Model<WARP>::dims;
    extern __shared__ __align__(16) float sw[];
    const int npix = A.Hc * A.Wc;
    for (int i = threadIdx.x; i < npix; i += kGradThreads) sw[i] = W[i];
    __syncthreads();
    double acc[D];
#pragma unroll
    for (int j = 0; j < D; ++j) acc[j] = 0.0;
    const int64_t stride = (int64_t)gridDim.x * kGradThreads;
    const int64_t i = (int64_t)blockIdx.x * kGradThreads + threadIdx.x;
    const T *px = (const T *)A.x, *py = (const T *)A.y, *pt = (const T *)A.t, *pp = (const T *)A.p;
    int64_t tail = i;
    if (A.vec16) {
        // 16-byte evict-first loads, two vectors of every array in flight per thread
        constexpr int EPV = 16 / (int)sizeof(T);
        const int64_t nv = A.n / EPV;
        for (int64_t v = i; v < nv; v += 2 * stride) {
            const bool two = v + stride < nv;
            const int64_t v2 = two ? v + stride : v;
            T ex[2][EPV], ey[2][EPV], et[2][EPV], ep[2][EPV];
            ld_vec16(px + v * EPV, ex[0]); ld_vec16(py + v * EPV, ey[0]); ld_vec16(pt + v * EPV, et[0]); ld_vec16(pp + v * EPV, ep[0]);
            ld_vec16(px + v2 * EPV, ex[1]); ld_vec16(py + v2 * EPV, ey[1]); ld_vec16(pt + v2 * EPV, et[1]); ld_vec16(pp + v2 * EPV, ep[1]);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                if (h == 1 && !two) break;
#pragma unroll
                for (int k = 0; k < EPV; ++k) grad_event<WARP>(A, sw, ex[h][k], ey[h][k], et[h][k], ep[h][k], acc);
            }
        }
        tail = nv * EPV + i;
    }
    for (int64_t j = tail; j < A.n; j += stride) grad_event<WARP>(A, sw, ld_stream(px + j), ld_stream(py + j), ld_stream(pt + j), ld_stream(pp + j), acc);
    // block reduction, one global add per CTA and parameter
    __shared__ double part[kGradThreads / 32][D];
#pragma unroll
    for (int j = 0; j < D; ++j) {
        double v = acc[j];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5][j] = v;
    }
    __syncthreads();
    if (threadIdx.x < D) {
        double s = 0.0;
        for (int w = 0; w < kGradThreads / 32; ++w) s += part[w][threadIdx.x];
        atomicAdd(gk + threadIdx.x, s);
    }
}

// get_iwe for a model on the device (objectives.py:184-190): warped, masked positions, polarities and Jacobians
// cast to f32 (image.py:179-183), ready for evk_image_drv_f32.  jx, jy: [dims][n].
template <int WARP>
__global__ void __launch_bounds__(256) cmax_model_warp_kernel(const CmaxArgs A, float *__restrict__ xo, float *__restrict__ yo,
                                                              float *__restrict__ po, float *__restrict__ jxo, float *__restrict__ jyo)
{
    using T = typename Model<WARP>::T;
    constexpr int D = Model<WARP>::dims;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < A.n; i += (int64_t)gridDim.x * 256) {
        T p = ((const T *)A.p)[i], xw, yw, jx[D], jy[D];
        const T m = model_event<WARP, true>(A, ((const T *)A.x)[i], ((const T *)A.y)[i], ((const T *)A.t)[i], p, xw, yw, jx, jy) ? (T)1 : (T)0;
        xo[i] = (float)(xw * m); yo[i] = (float)(yw * m); po[i] = (float)(p * m);
        if (jxo) {
#pragma unroll
            for (int j = 0; j < D; ++j) { jxo[(int64_t)j * A.n + i] = (float)(jx[j] * m); jyo[(int64_t)j * A.n + i] = (float)(jy[j] * m); }
        }
    }
}

// K candidate parameter points in ONE pass over the events (grid_search_initial evaluates 25 points per
// level, events_cmax.py:241-311): every event is loaded once and splatted into K accumulators.
struct Candidates {
    int n;
    double vx[kMaxCandidates], vy[kMaxCandidates];
};

template <int WARP, bool GRAD>
__global__ void __launch_bounds__(256) cmax_scatter_batch_kernel(const CmaxArgs A, const Candidates C)
{
    unsigned oob = 0;
    const int64_t acc_stride = (int64_t)A.Hc * A.Wc * kBlockFloats;
    const int64_t stride = (int64_t)gridDim.x * 256;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < A.n; i += 2 * stride) {
        const Event<WARP> e0 = load_event<WARP>(A, i);
        const bool has1 = i + stride < A.n;
        const Event<WARP> e1 = has1 ? load_event<WARP>(A, i + stride) : e0;
        for (int k = 0; k < C.n; ++k) {
            float *acc = A.acc + k * acc_stride;
            cmax_event<WARP, GRAD>(A, acc, e0, oob, C.vx[k], C.vy[k]);
            if (has1) cmax_event<WARP, GRAD>(A, acc, e1, oob, C.vx[k], C.vy[k]);
        }
    }
    flush_oob(A.oob, oob);
}

// ---- image-space tail (43.6 K pixels; negligible next to the event pass) ------------------
// sums[]: 0 sum(I)  1 sum(G)  2 sum(G^2)  3 sum(G*D0)  4 sum(G*D1)  5 sum(D0)  6 sum(D1)
// block-wide sum of v (all 256 threads participate), one atomicAdd(double) per block
__device__ __forceinline__ void block_add(double v, double *dst)
{
    __shared__ double part[8];
    const int lt = threadIdx.y * blockDim.x + threadIdx.x;   // blocks are 256 threads, 1-D or 32x8
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();  // protect `part` against the previous call's readers
    if ((lt & 31) == 0) part[lt >> 5] = v;
    __syncthreads();
    if (lt == 0) {
        double s = 0.0;
        for (int w = 0; w < 8; ++w) s += part[w];
        atomicAdd(dst, s);
    }
}

// CTA-wide sum in a FIXED order (shuffle tree, then the 8 warp sums left to right); valid on thread 0
__device__ __forceinline__ double block_sum_ordered(double v)
{
    __shared__ double part2[8];
    const int lt = threadIdx.y * blockDim.x + threadIdx.x;
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((lt & 31) == 0) part2[lt >> 5] = v;
    __syncthreads();
    double s = 0.0;
    if (lt == 0) for (int w = 0; w < 8; ++w) s += part2[w];
    return s;
}

// Blocks -> planar images.  Block (y,x) holds the 2x2 footprint anchored at (y,x) in tap order
// TL,TR,BL,BR, so pixel (y,x) collects TL of block (y,x), TR of (y,x-1), BL of (y-1,x) and BR of
// (y-1,x-1), over all replicas.
__global__ void __launch_bounds__(256) cmax_gather_kernel(const float *__restrict__ acc, const float *__restrict__ planar,
                                                          int replicas, int Hc, int Wc,
                                                          float *__restrict__ I, float *__restrict__ D0,
                                                          float *__restrict__ D1, float *__restrict__ iwe_out,
                                                          float *__restrict__ diwe_out, double *sums,
                                                          const unsigned long long *oob_in = nullptr, unsigned long long *oob_out = nullptr)
{
    const int npix = Hc * Wc;
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (oob_out && i == 0) *oob_out = *oob_in;
    float a = 0.f, b = 0.f, c = 0.f;
    if (i < npix) {
        const int y = i / Wc, x = i - y * Wc;
        if (planar) a = planar[i];      // the on-chip images (cmax_onchip_kernel); the blocks then hold carries / slow-path taps only
        for (int r = 0; r < replicas; ++r) {
            const float *base = acc + (int64_t)r * npix * kBlockFloats;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int by = y - (k >> 1), bx = x - (k & 1);
                if (by < 0 || bx < 0) continue;
                const float *blk = base + ((int64_t)by * Wc + bx) * kBlockFloats;
                a += blk[k];
                // D0 block = {-a, +a, -b, +b}, D1 block = {-c, -d, +c, +d} (see splat)
                b += (k == 0) ? -blk[4] : (k == 1) ? blk[4] : (k == 2) ? -blk[5] : blk[5];
                c += (k == 0) ? -blk[6] : (k == 1) ? -blk[7] : (k == 2) ? blk[6] : blk[7];
            }
        }
        I[i] = a; D0[i] = b; D1[i] = c;
        if (iwe_out) iwe_out[i] = a;
        if (diwe_out) { diwe_out[i] = b; diwe_out[npix + i] = c; }
    }
    block_add((double)a, sums + 0);
    block_add((double)b, sums + 5);
    block_add((double)c, sums + 6);
}

__device__ __forceinline__ int reflect_idx(int i, int n)
{
    if (n == 1) return 0;
    const int period = 2 * n;
    i %= period;
    if (i < 0) i += period;
    return i < n ? i : period - 1 - i;
}

// scipy applies axis 0 first and rounds the intermediate to f32
__global__ void __launch_bounds__(256) cmax_blur_axis0_kernel(const float *__restrict__ I, float *__restrict__ tmp,
                                                              int Hc, int Wc, const BlurTaps taps)
{
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= Hc * Wc) return;
    const int y = i / Wc, x = i - y * Wc;
    double acc = (double)I[i] * taps.w[0];
    for (int k = 1; k <= taps.r; ++k)
        acc += ((double)I[reflect_idx(y - k, Hc) * Wc + x] + (double)I[reflect_idx(y + k, Hc) * Wc + x]) * taps.w[k];
    tmp[i] = (float)acc;
}

__global__ void __launch_bounds__(256) cmax_blur_axis1_sums_kernel(const float *__restrict__ tmp, const float *__restrict__ I,
                                                                   const float *__restrict__ D0, const float *__restrict__ D1,
                                                                   int Hc, int Wc, const BlurTaps taps, int do_blur,
                                                                   double *sums)
{
    const int i = blockIdx.x * 256 + threadIdx.x;
    double g = 0.0, d0 = 0.0, d1 = 0.0;
    if (i < Hc * Wc) {
        if (do_blur) {
            const int y = i / Wc, x = i - y * Wc;
            const float *row = tmp + y * Wc;
            double acc = (double)row[x] * taps.w[0];
            for (int k = 1; k <= taps.r; ++k)
                acc += ((double)row[reflect_idx(x - k, Wc)] + (double)row[reflect_idx(x + k, Wc)]) * taps.w[k];
            g = (double)(float)acc;
        } else {
            g = (double)I[i];
        }
        d0 = (double)D0[i]; d1 = (double)D1[i];
    }
    block_add(g, sums + 1);
    block_add(g * g, sums + 2);
    block_add(g * d0, sums + 3);
    block_add(g * d1, sums + 4);
}

// result[0]=f  [1]=g0  [2]=g1  [3]=sum(IWE)  [4]=oob events  [5]=var  [6],[7] un-mixed 2-D gradient
__global__ void cmax_final_kernel(const double *sums, const unsigned long long *oob, int npix, double mix_a,
                                  double mix_b, int want_grad, double *result)
{
    const double P = (double)npix;
    const double mean_g = sums[1] / P;
    const double var = sums[2] / P - mean_g * mean_g;
    const double mu = sums[0] / P;
    // g2d_k = -mean( 2 (G(I) - mu) D_k )   (adjoint form of objectives.py:256-262)
    const double g0 = -2.0 * (sums[3] - mu * sums[5]) / P;
    const double g1 = -2.0 * (sums[4] - mu * sums[6]) / P;
    result[0] = -var;
    result[1] = want_grad ? (mix_a * g0 + mix_b * g1) : 0.0;
    result[2] = want_grad ? (mix_b * g0 + mix_a * g1) : 0.0;
    result[3] = sums[0];
    result[4] = (double)(*oob);
    result[5] = var;
    result[6] = g0;
    result[7] = g1;
}

// ---- generic objective tail (the reference's other objective functions, objectives.py:266-596) ---
// All of them are  f = reduce(phi(G))  with G = G_sigma * IWE and  g_k = -c * sum( w * (G3d * dIWE)_k )
// for a per-pixel weight image w.  The reflect Gaussian is self-adjoint, so sum(w * G(D_k)) ==
// sum(G(w) * D_k): ONE more blur (of w) replaces the reference's blur of the (2,H,W) stack.
//   SOS / RMS (objectives.py:266-357)  f = -mean(G^2)          w = 2*IWE (un-blurred), c = 1/P
//   SOE  (:358-400)                    f = -mean(exp(G))       w = exp(G),             c = 1/P
//   MOA  (:401-430)                    f = -max(G)             no gradient
//   ISOA (:431-477)                    f = +#(G > thresh)      w = [G > thresh],       c = 1
//   SOSA (:478-523)                    f = -sum(exp(-p G))     w = -p exp(-p G),       c = 1
enum { OBJ_VARIANCE = 0, OBJ_SOS = 1, OBJ_SOE = 2, OBJ_MOA = 3, OBJ_ISOA = 4, OBJ_SOSA = 5 };

__device__ __forceinline__ unsigned encode_ordered(float f)
{
    const unsigned b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__host__ __device__ __forceinline__ float decode_ordered(unsigned u)
{
    const unsigned b = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
#ifdef __CUDA_ARCH__
    return __uint_as_float(b);
#else
    float f; memcpy(&f, &b, 4); return f;
#endif
}

// axis-1 blur, result stored (the variance path only needs its sums and does not store it)
__global__ void __launch_bounds__(256) cmax_blur_axis1_store_kernel(const float *__restrict__ tmp, const float *__restrict__ I,
                                                                    int Hc, int Wc, const BlurTaps taps, int do_blur,
                                                                    float *__restrict__ G)
{
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= Hc * Wc) return;
    if (!do_blur) { G[i] = I[i]; return; }
    const int y = i / Wc, x = i - y * Wc;
    const float *row = tmp + y * Wc;
    double acc = (double)row[x] * taps.w[0];
    for (int k = 1; k <= taps.r; ++k)
        acc += ((double)row[reflect_idx(x - k, Wc)] + (double)row[reflect_idx(x + k, Wc)]) * taps.w[k];
    G[i] = (float)acc;
}

// gsums: 0 sum(G^2)  1 sum(exp(G))  2 sum(exp(-p G))  3 #(G > thresh)  4 sum(G)  5 sum(Gw*D0)  6 sum(Gw*D1)
__global__ void __launch_bounds__(256) cmax_obj_reduce_kernel(const float *__restrict__ G, const float *__restrict__ I, int npix,
                                                              int kind, double param, double *gsums, unsigned *gmax,
                                                              double *__restrict__ w)
{
    const int i = blockIdx.x * 256 + threadIdx.x;
    double g2 = 0.0, ge = 0.0, ga = 0.0, gc = 0.0, g1 = 0.0;
    float mx = -FLT_MAX;
    if (i < npix) {
        const float g = G[i];
        const double gd = (double)g;
        g1 = gd;
        g2 = kind == OBJ_VARIANCE ? gd * gd : (double)(g * g);   // variance: as cmax_blur_axis1_sums; np.mean(iwe*iwe): f32 product
        if (kind == OBJ_SOE) ge = exp(gd);              // np.exp(iwe.astype(np.double))
        if (kind == OBJ_SOSA) ga = exp(-param * gd);    // np.exp(-p*iwe.astype(np.double))
        if (kind == OBJ_ISOA) gc = (g > (float)param) ? 1.0 : 0.0;
        mx = g;
        double wi = 0.0;
        if (kind == OBJ_SOS) wi = (double)(I[i] * 2.0f);                                  // (iwe*2.0), un-blurred IWE
        else if (kind == OBJ_SOE) wi = ge;
        else if (kind == OBJ_ISOA) wi = gc;
        else if (kind == OBJ_SOSA) wi = -param * exp((double)(float)(-param * gd));       // exp((-p*iwe).astype(double)): f32 product first
        w[i] = wi;
    }
    block_add(g2, gsums + 0);
    if (kind == OBJ_SOE) block_add(ge, gsums + 1);
    if (kind == OBJ_SOSA) block_add(ga, gsums + 2);
    if (kind == OBJ_ISOA) block_add(gc, gsums + 3);
    block_add(g1, gsums + 4);
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) atomicMax(gmax, encode_ordered(mx));
}

__global__ void __launch_bounds__(256) cmax_blur_d_axis0_kernel(const double *__restrict__ w, double *__restrict__ wt, int Hc,
                                                                int Wc, const BlurTaps taps)
{
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= Hc * Wc) return;
    const int y = i / Wc, x = i - y * Wc;
    double acc = w[i] * taps.w[0];
    for (int k = 1; k <= taps.r; ++k) acc += (w[reflect_idx(y - k, Hc) * Wc + x] + w[reflect_idx(y + k, Hc) * Wc + x]) * taps.w[k];
    wt[i] = acc;
}

__global__ void __launch_bounds__(256) cmax_blur_d_axis1_dot_kernel(const double *__restrict__ wt, const double *__restrict__ w,
                                                                    const float *__restrict__ D0, const float *__restrict__ D1,
                                                                    int Hc, int Wc, const BlurTaps taps, int do_blur, double *gsums)
{
    const int i = blockIdx.x * 256 + threadIdx.x;
    double a = 0.0, b = 0.0;
    if (i < Hc * Wc) {
        double gw;
        if (do_blur) {
            const int y = i / Wc, x = i - y * Wc;
            const double *row = wt + y * Wc;
            gw = row[x] * taps.w[0];
            for (int k = 1; k <= taps.r; ++k) gw += (row[reflect_idx(x - k, Wc)] + row[reflect_idx(x + k, Wc)]) * taps.w[k];
        } else {
            gw = w[i];
        }
        a = gw * (double)D0[i];
        b = gw * (double)D1[i];
    }
    block_add(a, gsums + 5);
    block_add(b, gsums + 6);
}

// result: [0]=f [1],[2]=g [3]=sum(IWE) [4]=oob events [5]=var or aux [6],[7]=un-mixed gradient
//         [8]=mean(G^2) [9]=sum(exp(-p G)) [10]=max(G) [11]=#(G>thresh)
__global__ void cmax_obj_final_kernel(int kind, const double *gsums, const unsigned *gmax, const double *sums,
                                      const unsigned long long *oob, int npix, double mix_a, double mix_b, int want_grad,
                                      double *result)
{
    const double P = (double)npix;
    double f = 0.0, c = 0.0;
    const double mx = (double)decode_ordered(*gmax);
    if (kind == OBJ_SOS) { f = -gsums[0] / P; c = 1.0 / P; }
    else if (kind == OBJ_SOE) { f = -gsums[1] / P; c = 1.0 / P; }
    else if (kind == OBJ_MOA) { f = -mx; c = 0.0; }
    else if (kind == OBJ_ISOA) { f = gsums[3]; c = 1.0; }
    else if (kind == OBJ_SOSA) { f = -gsums[2]; c = 1.0; }
    const double u0 = -c * gsums[5], u1 = -c * gsums[6];
    const bool grad = want_grad && kind != OBJ_MOA;
    result[0] = f;
    result[1] = grad ? (mix_a * u0 + mix_b * u1) : 0.0;
    result[2] = grad ? (mix_b * u0 + mix_a * u1) : 0.0;
    result[3] = sums[0];
    result[4] = (double)(*oob);
    result[5] = gsums[4] / P;
    result[6] = u0;
    result[7] = u1;
    result[8] = gsums[0] / P;
    result[9] = gsums[2];
    result[10] = mx;
    result[11] = gsums[3];
}

// ---- tail of the models (any number K <= 8 of parameters): the weight image W, then f and K gradient entries ----
constexpr int kMaxDims = 8;
struct MixK { double m[kMaxDims][kMaxDims]; };   // scipy's blur along the length-K derivative-stack axis (objectives.py:253)

// variance: W = G(2(I - mu)) = 2(G(I) - mu)  (reflect blur: self-adjoint, keeps constants)
__global__ void __launch_bounds__(256) cmax_weight_variance_kernel(const float *__restrict__ G, const double *sums, int npix,
                                                                   float *__restrict__ W)
{
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= npix) return;
    const double mu = sums[0] / (double)npix;
    W[i] = (float)(2.0 * ((double)G[i] - mu));
}

// generic objectives: W = G(w), the axis-1 half of the blur of the per-pixel weight (cmax_blur_d_axis0_kernel is the other)
__global__ void __launch_bounds__(256) cmax_blur_d_axis1_store_kernel(const double *__restrict__ wt, const double *__restrict__ w,
                                                                      int Hc, int Wc, const BlurTaps taps, int do_blur, float *__restrict__ W)
{
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= Hc * Wc) return;
    double gw;
    if (do_blur) {
        const int y = i / Wc, x = i - y * Wc;
        const double *row = wt + y * Wc;
        gw = row[x] * taps.w[0];
        for (int k = 1; k <= taps.r; ++k) gw += (row[reflect_idx(x - k, Wc)] + row[reflect_idx(x + k, Wc)]) * taps.w[k];
    } else {
        gw = w[i];
    }
    W[i] = (float)gw;
}

// precomputed derivative images: gk[k] = sum_pix W D_k
__global__ void __launch_bounds__(256) cmax_dot_k_kernel(const float *__restrict__ W, const float *__restrict__ diwe, int K, int npix, double *gk)
{
    const int i = blockIdx.x * 256 + threadIdx.x;
    const double wi = i < npix ? (double)W[i] : 0.0;
    for (int k = 0; k < K; ++k) block_add(i < npix ? wi * (double)diwe[(int64_t)k * npix + i] : 0.0, gk + k);
}

// result: the 12 slots of cmax_obj_final_kernel (variance: [5] = var); grad: K entries
__global__ void cmax_model_final_kernel(int kind, int K, const MixK M, const double *gsums, const unsigned *gmax, const double *sums,
                                        const double *gk, const unsigned long long *oob, int npix, int want_grad, double *result,
                                        double *grad)
{
    const double P = (double)npix;
    double f = 0.0, c = 0.0;
    const double mx = (double)decode_ordered(*gmax);
    const double mean_g = gsums[4] / P;
    if (kind == OBJ_VARIANCE) { f = -(gsums[0] / P - mean_g * mean_g); c = 1.0 / P; }
    else if (kind == OBJ_SOS) { f = -gsums[0] / P; c = 1.0 / P; }
    else if (kind == OBJ_SOE) { f = -gsums[1] / P; c = 1.0 / P; }
    else if (kind == OBJ_MOA) { f = -mx; c = 0.0; }
    else if (kind == OBJ_ISOA) { f = gsums[3]; c = 1.0; }
    else if (kind == OBJ_SOSA) { f = -gsums[2]; c = 1.0; }
    const bool g_on = want_grad && kind != OBJ_MOA;
    double u[kMaxDims];
    for (int j = 0; j < kMaxDims; ++j) u[j] = (g_on && j < K) ? -c * gk[j] : 0.0;
    for (int k = 0; k < K; ++k) {
        double v = 0.0;
        for (int j = 0; j < K; ++j) v += M.m[k][j] * u[j];
        grad[k] = g_on ? v : 0.0;
    }
    result[0] = f;
    result[1] = K > 0 ? grad[0] : 0.0;
    result[2] = K > 1 ? grad[1] : 0.0;
    result[3] = sums[0];
    result[4] = (double)(*oob);
    result[5] = kind == OBJ_VARIANCE ? -f : mean_g;
    result[6] = u[0];
    result[7] = u[1];
    result[8] = gsums[0] / P;
    result[9] = gsums[2];
    result[10] = mx;
    result[11] = gsums[3];
}

// ---- fused variance tail: gather + both blur axes + all sums + the final scalars in ONE launch ---
// One CTA = an 8x32 tile of pixels.  It gathers the tile plus a halo of `r` pixels (reflected at the image
// border, like scipy's mode='reflect') straight from the block accumulator into shared memory, blurs
// vertically then horizontally with the same f64-accumulate / f32-store rounding as the separate kernels,
// reduces the seven sums, and the last CTA to finish (ticket counter) writes the result.  Replaces four
// launches (gather, blur axis 0, blur axis 1 + sums, final) -- at BFGS problem sizes (1e4..1e6 events) the
// evaluation is launch-bound.
constexpr int kTileY = 8, kTileX = 32, kFusedMaxR = 8;

// Sharded evaluation (one process per GPU): every rank's partial planar images [3][Hc*Wc] (I, D0, D1) live in symmetric
// memory; the tail of EVERY rank reads all of them through NVLink peer pointers and sums them on the fly (in rank order, so all
// ranks compute bit-identical f and g) -- the all-reduce is fused into the objective kernel, there is no NCCL call.
constexpr int kMaxCmaxPeers = 16;
struct CmaxPeers {
    const float *img[kMaxCmaxPeers];                  // [3][Hc*Wc] per rank
    const unsigned long long *oob[kMaxCmaxPeers];     // out-of-canvas events per rank
    int world;
};

__device__ __forceinline__ float gather_peers(const CmaxPeers &P, int Hc, int Wc, int y, int x, int comp)
{
    const int64_t npix = (int64_t)Hc * Wc, i = (int64_t)comp * npix + (int64_t)y * Wc + x;
    float v = 0.f;
    for (int r = 0; r < P.world; ++r) v += __ldcg(P.img[r] + i);       // peer loads bypass L1 (the data was written by another GPU)
    return v;
}

__device__ __forceinline__ float gather_pixel(const float *acc, const float *planar, int replicas, int Hc, int Wc, int y, int x, int comp)
{
    // comp 0: I, 1: D0, 2: D1 (see cmax_gather_kernel for the block / sign conventions)
    const int64_t npix = (int64_t)Hc * Wc;
    float v = (comp == 0 && planar) ? planar[(int64_t)y * Wc + x] : 0.f;
    for (int r = 0; r < replicas; ++r) {
        const float *base = acc + (int64_t)r * npix * kBlockFloats;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int by = y - (k >> 1), bx = x - (k & 1);
            if (by < 0 || bx < 0) continue;
            const float *blk = base + ((int64_t)by * Wc + bx) * kBlockFloats;
            if (comp == 0) v += blk[k];
            else if (comp == 1) v += (k == 0) ? -blk[4] : (k == 1) ? blk[4] : (k == 2) ? -blk[5] : blk[5];
            else v += (k == 0) ? -blk[6] : (k == 1) ? -blk[7] : (k == 2) ? blk[6] : blk[7];
        }
    }
    return v;
}

template <bool PEER>
__global__ void __launch_bounds__(kTileY *kTileX) cmax_fused_var_tail_kernel_t(const CmaxPeers PE, const float *__restrict__ acc, const float *__restrict__ planar, int replicas, int Hc, int Wc,
                                                                              const BlurTaps taps, int do_blur, int want_grad,
                                                                              double mix_a, double mix_b, float *__restrict__ iwe_out,
                                                                              float *__restrict__ diwe_out, double *sums,
                                                                              unsigned *ticket, const unsigned long long *oob,
                                                                              double *result, double *partials = nullptr)
{
    __shared__ float tileI[(kTileY + 2 * kFusedMaxR) * (kTileX + 2 * kFusedMaxR)];
    __shared__ float tileT[kTileY * (kTileX + 2 * kFusedMaxR)];
    // blockIdx.z = candidate index of a batched evaluation: its own accumulator, sums, ticket and result
    acc += (size_t)blockIdx.z * (size_t)Hc * Wc * kBlockFloats * replicas;
    sums += 8 * blockIdx.z;
    ticket += blockIdx.z;
    result += 12 * blockIdx.z;
    const int r = do_blur ? taps.r : 0;
    const int hw = kTileX + 2 * r, hh = kTileY + 2 * r;
    const int y0 = blockIdx.y * kTileY, x0 = blockIdx.x * kTileX;
    const int tid = threadIdx.y * kTileX + threadIdx.x;
    // 1. halo tile of the un-blurred IWE
    for (int j = tid; j < hh * hw; j += kTileY * kTileX) {
        const int ly = j / hw, lx = j - ly * hw;
        const int gy = reflect_idx(y0 - r + ly, Hc), gx = reflect_idx(x0 - r + lx, Wc);
        tileI[j] = PEER ? gather_peers(PE, Hc, Wc, gy, gx, 0) : gather_pixel(acc, planar, replicas, Hc, Wc, gy, gx, 0);
    }
    const int y = y0 + threadIdx.y, x = x0 + threadIdx.x;
    const bool inside = y < Hc && x < Wc;
    float vi = 0.f, d0 = 0.f, d1 = 0.f;
    if (inside) {
        d0 = PEER ? gather_peers(PE, Hc, Wc, y, x, 1) : gather_pixel(acc, nullptr, replicas, Hc, Wc, y, x, 1);
        d1 = PEER ? gather_peers(PE, Hc, Wc, y, x, 2) : gather_pixel(acc, nullptr, replicas, Hc, Wc, y, x, 2);
    }
    __syncthreads();
    if (inside) {
        vi = tileI[(threadIdx.y + r) * hw + threadIdx.x + r];
        const int64_t npix = (int64_t)Hc * Wc, i = (int64_t)y * Wc + x;
        if (iwe_out) iwe_out[i] = vi;
        if (diwe_out) { diwe_out[i] = d0; diwe_out[npix + i] = d1; }
    }
    double g = (double)vi;
    if (do_blur) {
        // 2. axis 0 (vertical), every column of the halo; rounded to f32 like scipy's intermediate array
        for (int j = tid; j < kTileY * hw; j += kTileY * kTileX) {
            const int ly = j / hw, lx = j - ly * hw;
            const float *col = tileI + (ly + r) * hw + lx;
            double a = (double)col[0] * taps.w[0];
            for (int k = 1; k <= r; ++k) a += ((double)col[-k * hw] + (double)col[k * hw]) * taps.w[k];
            tileT[j] = (float)a;
        }
        __syncthreads();
        // 3. axis 1 (horizontal)
        const float *row = tileT + threadIdx.y * hw + threadIdx.x + r;
        double a = (double)row[0] * taps.w[0];
        for (int k = 1; k <= r; ++k) a += ((double)row[-k] + (double)row[k]) * taps.w[k];
        g = (double)(float)a;
    }
    if (!inside) { g = 0.0; vi = 0.f; }
    // 4. the seven sums (same slots as the separate kernels)
    const int cta = blockIdx.y * gridDim.x + blockIdx.x, nctas = gridDim.x * gridDim.y;
    if (PEER) {
        // sharded evaluation: every rank must arrive at bit-identical f and g (a BFGS driver runs replicated), so the sums
        // are formed in a fixed order: per-CTA partials to memory, the last CTA adds them up CTA by CTA
        const double v[7] = {(double)vi, g, g * g, g * (double)d0, g * (double)d1, (double)d0, (double)d1};
#pragma unroll
        for (int k = 0; k < 7; ++k) {
            const double sk = block_sum_ordered(v[k]);
            if (tid == 0) partials[(size_t)cta * 8 + k] = sk;
        }
    } else {
        block_add((double)vi, sums + 0);
        block_add(g, sums + 1);
        block_add(g * g, sums + 2);
        block_add(g * (double)d0, sums + 3);
        block_add(g * (double)d1, sums + 4);
        block_add((double)d0, sums + 5);
        block_add((double)d1, sums + 6);
    }
    // 5. last CTA writes the result
    __shared__ bool last;
    if (tid == 0) {
        __threadfence();
        last = atomicAdd(ticket, 1u) == (unsigned)nctas - 1;
    }
    __syncthreads();
    if (last && tid == 0) {
        __threadfence();
        double s[7];
        if (PEER) {
            for (int k = 0; k < 7; ++k) s[k] = 0.0;
            for (int c = 0; c < nctas; ++c)
                for (int k = 0; k < 7; ++k) s[k] += __ldcg(partials + (size_t)c * 8 + k);
        } else {
            for (int k = 0; k < 7; ++k) s[k] = atomicAdd(sums + k, 0.0);   // read through L2
        }
        const double P = (double)Hc * (double)Wc;
        const double mean_g = s[1] / P, var = s[2] / P - mean_g * mean_g, mu = s[0] / P;
        const double g0 = -2.0 * (s[3] - mu * s[5]) / P, g1 = -2.0 * (s[4] - mu * s[6]) / P;
        result[0] = -var;
        result[1] = want_grad ? (mix_a * g0 + mix_b * g1) : 0.0;
        result[2] = want_grad ? (mix_b * g0 + mix_a * g1) : 0.0;
        result[3] = s[0];
        if (PEER) {
            unsigned long long bad = 0;
            for (int r = 0; r < PE.world; ++r) bad += __ldcg(PE.oob[r]);
            result[4] = (double)bad;
        } else {
            result[4] = (double)(*oob);
        }
        result[5] = var;
        result[6] = g0;
        result[7] = g1;
    }
}

struct CmaxWorkspace {
    float *planar;              // on-chip path: planar IWE the CTAs' shared-memory images are bulk-reduced into
    float *acc, *I, *D0, *D1, *tmp, *G;
    double *bsums;              // [kMaxCandidates][8] sums of a batched evaluation
    unsigned *btickets;         // [kMaxCandidates]
    double *w, *wt;             // generic objectives: per-pixel weight image and its axis-0 blur
    double *gsums;              // 8 doubles (generic objectives)
    unsigned *gmax;             // order-preserving encoding of max(G)
    double *sums;               // 8 doubles
    double *gk;                 // kMaxDims doubles: sum_pix W D_k of the model tail
    unsigned long long *oob;    // 1
};

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

static size_t carve(void *base, int Hs, int Ws, CmaxWorkspace *ws)
{
    const size_t npix = (size_t)(Hs + 1) * (Ws + 1);
    size_t off = 0;
    char *b = static_cast<char *>(base);
    auto take = [&](size_t bytes) { char *p = b ? b + off : nullptr; off += align_up(bytes, 256); return p; };
    // the small counters come first and are directly followed by the accumulator, so that ONE memset
    // zeroes counters + the R replicas an evaluation uses
    double *bsums = (double *)take(kMaxCandidates * 8 * sizeof(double));
    unsigned *btickets = (unsigned *)take(kMaxCandidates * sizeof(unsigned));
    double *gsums = (double *)take(8 * sizeof(double));
    unsigned *gmax = (unsigned *)take(sizeof(unsigned));
    double *sums = (double *)take(8 * sizeof(double));
    double *gk = (double *)take(kMaxDims * sizeof(double));
    unsigned long long *oob = (unsigned long long *)take(sizeof(unsigned long long));
    float *planar = (float *)take(((npix + 3) & ~(size_t)3) * sizeof(float));
    float *acc = (float *)take(npix * kBlockFloats * sizeof(float) * (kMaxCandidates > kMaxReplicas ? kMaxCandidates : kMaxReplicas));
    float *I = (float *)take(npix * sizeof(float));
    float *D0 = (float *)take(npix * sizeof(float));
    float *D1 = (float *)take(npix * sizeof(float));
    float *tmp = (float *)take(npix * sizeof(float));
    float *G = (float *)take(npix * sizeof(float));
    double *w = (double *)take(npix * sizeof(double));
    double *wt = (double *)take(npix * sizeof(double));
    if (ws) {
        ws->planar = planar; ws->acc = acc; ws->I = I; ws->D0 = D0; ws->D1 = D1; ws->tmp = tmp; ws->G = G; ws->w = w; ws->wt = wt;
        ws->gsums = gsums; ws->gmax = gmax; ws->sums = sums; ws->gk = gk; ws->oob = oob; ws->bsums = bsums; ws->btickets = btickets;
    }
    return off;
}

// channel-mix coefficients of scipy's blur along the length-2 stack axis (reflect):
// blurring the unit vector [1,0]: index i of the reflected signal equals 0 for i mod 4 in {0,3}.
static void mix_coeffs(const BlurTaps &t, double *a, double *b)
{
    double sa = 0.0, sb = 0.0;
    for (int k = -t.r; k <= t.r; ++k) {
        int i = k % 4;
        if (i < 0) i += 4;
        const double w = t.w[k < 0 ? -k : k];
        if (i == 0 || i == 3) sa += w; else sb += w;
    }
    *a = sa; *b = sb;
}

static int make_taps(double sigma, BlurTaps *t)
{
    int r = (int)(4.0 * sigma + 0.5);
    if (r > kMaxRadius) { set_error("evk_cmax: blur sigma %.3f needs radius %d > %d", sigma, r, kMaxRadius); return EVK_E_UNSUPPORTED; }
    t->r = r;
    double s = 0.0;
    for (int k = -r; k <= r; ++k) s += exp(-0.5 / (sigma * sigma) * (double)k * (double)k);
    for (int k = 0; k <= r; ++k) t->w[k] = exp(-0.5 / (sigma * sigma) * (double)k * (double)k) / s;
    return EVK_OK;
}

// image-space tail shared by the event entry points and the precomputed-image entry point
static int launch_tail(const CmaxWorkspace &ws, int Hc, int Wc, double sigma, unsigned flags, int objective, double obj_param,
                       bool grad, double *result, cudaStream_t st)
{
    const int npix = Hc * Wc;
    BlurTaps taps{};
    double mix_a = 1.0, mix_b = 0.0;
    const int do_blur = sigma > 0.0;
    if (do_blur) {
        int rc = make_taps(sigma, &taps);
        if (rc) return rc;
        if (!(flags & EVK_CMAX_NO_CHANNEL_MIX)) mix_coeffs(taps, &mix_a, &mix_b);
    }
    const int g = (npix + 255) / 256;
    if (do_blur) { prof_count(1); cmax_blur_axis0_kernel<<<g, 256, 0, st>>>(ws.I, ws.tmp, Hc, Wc, taps); }
    if (objective == OBJ_VARIANCE) {
        prof_count(2);
        cmax_blur_axis1_sums_kernel<<<g, 256, 0, st>>>(ws.tmp, ws.I, ws.D0, ws.D1, Hc, Wc, taps, do_blur, ws.sums);
        cmax_final_kernel<<<1, 1, 0, st>>>(ws.sums, ws.oob, npix, mix_a, mix_b, grad ? 1 : 0, result);
    } else {
        if (objective < OBJ_SOS || objective > OBJ_SOSA) { set_error("evk_cmax: unknown objective %d", objective); return EVK_E_ARG; }
        const bool g_needed = grad && objective != OBJ_MOA;
        prof_count(3);
        cmax_blur_axis1_store_kernel<<<g, 256, 0, st>>>(ws.tmp, ws.I, Hc, Wc, taps, do_blur, ws.G);
        cmax_obj_reduce_kernel<<<g, 256, 0, st>>>(ws.G, ws.I, npix, objective, obj_param, ws.gsums, ws.gmax, ws.w);
        if (g_needed) {
            prof_count(do_blur ? 2 : 1);
            if (do_blur) cmax_blur_d_axis0_kernel<<<g, 256, 0, st>>>(ws.w, ws.wt, Hc, Wc, taps);
            cmax_blur_d_axis1_dot_kernel<<<g, 256, 0, st>>>(ws.wt, ws.w, ws.D0, ws.D1, Hc, Wc, taps, do_blur, ws.gsums);
        }
        cmax_obj_final_kernel<<<1, 1, 0, st>>>(objective, ws.gsums, ws.gmax, ws.sums, ws.oob, npix, mix_a, mix_b, g_needed ? 1 : 0, result);
    }
    EVK_CUDA(cudaGetLastError());
    return EVK_OK;
}

// M[k][j] = sum_m w[|m|] [reflect(k + m, K) == j]: scipy's blur along the length-K stack axis, applied to the K
// gradient entries (mix_coeffs is the K = 2 case); the identity without blur or with EVK_CMAX_NO_CHANNEL_MIX
static void mix_matrix(const BlurTaps &t, int do_blur, unsigned flags, int K, MixK *M)
{
    memset(M, 0, sizeof(*M));
    const bool mix = do_blur && !(flags & EVK_CMAX_NO_CHANNEL_MIX);
    for (int k = 0; k < K; ++k) {
        if (!mix) { M->m[k][k] = 1.0; continue; }
        for (int m = -t.r; m <= t.r; ++m) {
            int i = k + m;
            const int period = 2 * K;
            if (K == 1) i = 0;
            else { i %= period; if (i < 0) i += period; if (i >= K) i = period - 1 - i; }
            M->m[k][i] += t.w[m < 0 ? -m : m];
        }
    }
}

// The model tail on the planar IWE in ws.I (sums[0] = its sum): blur, the objective's reductions, the weight image W
// (ws.tmp), then `pass2(W)` fills ws.gk[0..K) with sum_pix W D_k, and the final kernel writes f and the K entries.
template <typename Pass2>
static int model_tail(const CmaxWorkspace &ws, int Hc, int Wc, double sigma, unsigned flags, int objective, double obj_param,
                      bool want_grad, int K, Pass2 &&pass2, double *result, double *grad, cudaStream_t st)
{
    if (objective < OBJ_VARIANCE || objective > OBJ_SOSA) { set_error("evk_cmax: unknown objective %d", objective); return EVK_E_ARG; }
    const int npix = Hc * Wc;
    BlurTaps taps{};
    const int do_blur = sigma > 0.0;
    if (do_blur) {
        int rc = make_taps(sigma, &taps);
        if (rc) return rc;
    }
    MixK M;
    mix_matrix(taps, do_blur, flags, K, &M);
    const int g = (npix + 255) / 256;
    prof_count(do_blur ? 3 : 2);
    if (do_blur) cmax_blur_axis0_kernel<<<g, 256, 0, st>>>(ws.I, ws.tmp, Hc, Wc, taps);
    cmax_blur_axis1_store_kernel<<<g, 256, 0, st>>>(ws.tmp, ws.I, Hc, Wc, taps, do_blur, ws.G);
    cmax_obj_reduce_kernel<<<g, 256, 0, st>>>(ws.G, ws.I, npix, objective, obj_param, ws.gsums, ws.gmax, ws.w);
    const bool g_needed = want_grad && objective != OBJ_MOA;
    if (g_needed) {
        if (objective == OBJ_VARIANCE) {
            prof_count(1);
            cmax_weight_variance_kernel<<<g, 256, 0, st>>>(ws.G, ws.sums, npix, ws.tmp);
        } else {
            prof_count(do_blur ? 2 : 1);
            if (do_blur) cmax_blur_d_axis0_kernel<<<g, 256, 0, st>>>(ws.w, ws.wt, Hc, Wc, taps);
            cmax_blur_d_axis1_store_kernel<<<g, 256, 0, st>>>(ws.wt, ws.w, Hc, Wc, taps, do_blur, ws.tmp);
        }
        EVK_CUDA(cudaGetLastError());
        int rc = pass2(ws.tmp);
        if (rc) return rc;
    }
    prof_count(1);
    cmax_model_final_kernel<<<1, 1, 0, st>>>(objective, K, M, ws.gsums, ws.gmax, ws.sums, ws.gk, ws.oob, npix, g_needed ? 1 : 0, result, grad);
    EVK_CUDA(cudaGetLastError());
    return EVK_OK;
}

// event count from which the on-chip IWE pays (EVK_CMAX_ONCHIP_MIN overrides; measured crossover, DESIGN.md section 4)
static int64_t onchip_min_events()
{
    static int64_t v = -1;
    if (v < 0) {
        const char *e = getenv("EVK_CMAX_ONCHIP_MIN");
        v = (e && *e) ? atoll(e) : ((int64_t)4 << 20);
    }
    return v;
}

// partial_images != nullptr: stop after the event pass and leave this rank's planar I, D0, D1 ([3][Hc*Wc]) and its
// out-of-canvas count there (the sharded evaluation's first half; evk_cmax_peer_tail_f32 is the second)
template <int WARP>
static int run_cmax(CmaxArgs A, double sigma, unsigned flags, int objective, double obj_param, double *result,
                    float *iwe_out, float *diwe_out, void *workspace, size_t workspace_bytes, cudaStream_t st,
                    float *partial_images = nullptr, unsigned long long *partial_oob = nullptr, double *model_grad = nullptr)
{
    const int Hs = A.Hc - 1, Ws = A.Wc - 1;
    if (A.n < 0 || Hs < 1 || Ws < 1 || (!result && !partial_images) || !workspace) { set_error("evk_cmax: bad arguments"); return EVK_E_ARG; }
    if (((uintptr_t)workspace & 255) != 0) { set_error("evk_cmax: workspace must be 256-byte aligned"); return EVK_E_ARG; }
    CmaxWorkspace ws;
    const size_t need = carve(workspace, Hs, Ws, &ws);
    if (workspace_bytes < need) { set_error("evk_cmax: workspace of %zu bytes required, %zu given", need, workspace_bytes); return EVK_E_WORKSPACE; }
    const int npix = A.Hc * A.Wc;
    // a model's event pass forms the IWE only; its gradient is the second pass of model_tail
    const bool grad = (flags & EVK_CMAX_WANT_GRAD) != 0 && WARP != WARP_FLOW_F32 && !is_model(WARP);
    A.abs_polarity = (flags & EVK_CMAX_ABS_POLARITY) ? 1 : 0;
    // replicas spread same-address serialisation in L2; small problems do not need them
    int R = (int)(A.n / (1 << 20));
    R = R < 1 ? 1 : (R > kMaxReplicas ? kMaxReplicas : R);
    A.replicas = R;
    A.acc = ws.acc;
    A.oob = ws.oob;
    // on-chip IWE: worth its fixed cost (174 KB of shared memory initialised and bulk-reduced per CTA) for
    // large event sets only; EVK_VARIANT_SMEM_TILE / EVK_VARIANT_VECTOR_RED force one or the other
    const size_t onchip_smem = (((size_t)npix + 3) & ~(size_t)3) * sizeof(float);
    const unsigned variant = variant_of(flags);
    bool onchip = onchip_smem <= (size_t)200 * 1024 && A.n > 0 &&
                  (variant == EVK_VARIANT_SMEM_TILE || (variant == EVK_VARIANT_AUTO && A.n >= onchip_min_events()));
    if (variant == EVK_VARIANT_VECTOR_RED || variant == EVK_VARIANT_GLOBAL_RED) onchip = false;
    A.planar = onchip ? ws.planar : nullptr;
    A.vec16 = ((((uintptr_t)A.x | (uintptr_t)A.y | (uintptr_t)A.t | (uintptr_t)A.p) & 15) == 0) ? 1 : 0;
    const float *planar = A.planar;
    if (onchip && !grad) { R = 1; A.replicas = 1; }   // the blocks only receive carries and slow-path taps
    // counters (gsums, gmax, sums, oob), the planar image and the R accumulator replicas are contiguous: one memset
    EVK_CUDA(cudaMemsetAsync(ws.gsums, 0, (size_t)((char *)ws.acc - (char *)ws.gsums) + (size_t)R * npix * kBlockFloats * sizeof(float), st));
    if (WARP == WARP_FLOW_F32 && A.n > 0) {
        // the generic objectives' weight image (unused by the variance tail) holds the interleaved flow
        prof_count(1);
        launch_flow_interleave(A.flow, (int64_t)Hs * Ws, reinterpret_cast<float2 *>(ws.w), st);
        A.flow_uv = reinterpret_cast<const float2 *>(ws.w);
    }
    if (onchip) {
        ProfScope prof(st);
        prof_count(1);
        int64_t need_ctas = (A.n + kOnchipThreads * 8 - 1) / (kOnchipThreads * 8);
        const int g = (int)(need_ctas < num_sms() ? need_ctas : num_sms());
        if (grad) {
            EVK_CUDA(cudaFuncSetAttribute(cmax_onchip_kernel<WARP, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)onchip_smem));
            cmax_onchip_kernel<WARP, true><<<g, kOnchipThreads, onchip_smem, st>>>(A);
        } else {
            EVK_CUDA(cudaFuncSetAttribute(cmax_onchip_kernel<WARP, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)onchip_smem));
            cmax_onchip_kernel<WARP, false><<<g, kOnchipThreads, onchip_smem, st>>>(A);
        }
        EVK_CUDA(cudaGetLastError());
    } else if (A.n > 0) {
        ProfScope prof(st);
        prof_count(1);
        if (grad) cmax_scatter_kernel<WARP, true><<<grid_for(cmax_scatter_kernel<WARP, true>, 256, A.n, 256 * 4), 256, 0, st>>>(A);
        else cmax_scatter_kernel<WARP, false><<<grid_for(cmax_scatter_kernel<WARP, false>, 256, A.n, 256 * 4), 256, 0, st>>>(A);
    }
    if constexpr (is_model(WARP)) {
        prof_count(1);
        cmax_gather_kernel<<<(npix + 255) / 256, 256, 0, st>>>(ws.acc, planar, R, A.Hc, A.Wc, ws.I, ws.D0, ws.D1, nullptr, nullptr, ws.sums);
        auto pass2 = [&](const float *W) -> int {
            if (A.n == 0) return EVK_OK;
            const size_t smem = (size_t)npix * sizeof(float);
            if (smem > (size_t)227 * 1024) { set_error("evk_cmax: a %dx%d weight image does not fit in shared memory", A.Hc, A.Wc); return EVK_E_UNSUPPORTED; }
            EVK_CUDA(cudaFuncSetAttribute(cmax_model_grad_kernel<WARP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            const int64_t need_ctas = (A.n + kGradThreads * 8 - 1) / (kGradThreads * 8);
            const int g = (int)(need_ctas < num_sms() ? need_ctas : num_sms());
            ProfScope prof(st);
            prof_count(1);
            cmax_model_grad_kernel<WARP><<<g, kGradThreads, smem, st>>>(A, W, ws.gk);
            EVK_CUDA(cudaGetLastError());
            return EVK_OK;
        };
        return model_tail(ws, A.Hc, A.Wc, sigma, flags, objective, obj_param, (flags & EVK_CMAX_WANT_GRAD) != 0, Model<WARP>::dims,
                          pass2, result, model_grad, st);
    }
    if (partial_images) {
        prof_count(1);
        cmax_gather_kernel<<<(npix + 255) / 256, 256, 0, st>>>(ws.acc, planar, R, A.Hc, A.Wc, partial_images, partial_images + npix,
                                                                partial_images + 2 * (size_t)npix, nullptr, nullptr, ws.sums, ws.oob, partial_oob);
        EVK_CUDA(cudaGetLastError());
        return EVK_OK;
    }
    if (objective == OBJ_VARIANCE && (sigma <= 0.0 || (int)(4.0 * sigma + 0.5) <= kFusedMaxR)) {
        // launch-bound regime matters most here: gather + blur + sums + final in one kernel
        BlurTaps taps{};
        double mix_a = 1.0, mix_b = 0.0;
        const int do_blur = sigma > 0.0;
        if (do_blur) {
            int rc = make_taps(sigma, &taps);
            if (rc) return rc;
            if (!(flags & EVK_CMAX_NO_CHANNEL_MIX)) mix_coeffs(taps, &mix_a, &mix_b);
        }
        prof_count(1);
        dim3 tgrid((A.Wc + kTileX - 1) / kTileX, (A.Hc + kTileY - 1) / kTileY), tblock(kTileX, kTileY);
        cmax_fused_var_tail_kernel_t<false><<<tgrid, tblock, 0, st>>>(CmaxPeers{}, ws.acc, planar, R, A.Hc, A.Wc, taps, do_blur, grad ? 1 : 0, mix_a, mix_b, iwe_out,
                                                               diwe_out, ws.sums, ws.gmax, ws.oob, result);
        EVK_CUDA(cudaGetLastError());
        return EVK_OK;
    }
    prof_count(1);
    cmax_gather_kernel<<<(npix + 255) / 256, 256, 0, st>>>(ws.acc, planar, R, A.Hc, A.Wc, ws.I, ws.D0, ws.D1, iwe_out, diwe_out, ws.sums);
    return launch_tail(ws, A.Hc, A.Wc, sigma, flags, objective, obj_param, grad, result, st);
}

// precomputed planar iwe / diwe -> the planar working images + their sums (the block accumulator is
// bypassed: a block value stands for taps of TWO pixels, planar images cannot be packed into it)
__global__ void __launch_bounds__(256) cmax_planar_kernel(const float *__restrict__ iwe, const float *__restrict__ diwe,
                                                          int npix, float *__restrict__ I, float *__restrict__ D0,
                                                          float *__restrict__ D1, double *sums)
{
    const int i = blockIdx.x * 256 + threadIdx.x;
    float a = 0.f, b = 0.f, c = 0.f;
    if (i < npix) {
        a = iwe[i];
        if (diwe) { b = diwe[i]; c = diwe[npix + i]; }
        I[i] = a; D0[i] = b; D1[i] = c;
    }
    block_add((double)a, sums + 0);
    block_add((double)b, sums + 5);
    block_add((double)c, sums + 6);
}

}  // namespace evk

extern "C" {

size_t evk_cmax_workspace_bytes(int Hs, int Ws)
{
    if (Hs < 1 || Ws < 1) return 0;
    return evk::carve(nullptr, Hs, Ws, nullptr);
}

int evk_cmax_linvel_objective_f64(const double *x, const double *y, const double *t, const double *p, int64_t n,
                                  double p_scale, double vx, double vy, double t_ref, int Hm, int Wm, int Hs, int Ws,
                                  double sigma, unsigned flags, int objective, double obj_param, double *result,
                                  float *iwe_out, float *diwe_out, void *workspace, size_t workspace_bytes, void *stream)
{
    using namespace evk;
    if (n > 0 && (!x || !y || !t || !p)) { set_error("evk_cmax_linvel_objective_f64: null event array"); return EVK_E_ARG; }
    CmaxArgs A{};
    A.x = x; A.y = y; A.t = t; A.p = p; A.n = n;
    A.vx = vx; A.vy = vy; A.t_ref = t_ref; A.p_scale = p_scale;
    A.Hm = Hm; A.Wm = Wm; A.Hc = Hs + 1; A.Wc = Ws + 1;
    return run_cmax<WARP_LINVEL_F64>(A, sigma, flags, objective, obj_param, result, iwe_out, diwe_out, workspace,
                                     workspace_bytes, static_cast<cudaStream_t>(stream));
}

int evk_cmax_linvel_objective_f32(const float *x, const float *y, const float *t_rel, const float *p, int64_t n,
                                  float p_scale, float vx, float vy, int Hm, int Wm, int Hs, int Ws, double sigma,
                                  unsigned flags, int objective, double obj_param, double *result, float *iwe_out,
                                  float *diwe_out, void *workspace, size_t workspace_bytes, void *stream)
{
    using namespace evk;
    if (n > 0 && (!x || !y || !t_rel || !p)) { set_error("evk_cmax_linvel_objective_f32: null event array"); return EVK_E_ARG; }
    CmaxArgs A{};
    A.x = x; A.y = y; A.t = t_rel; A.p = p; A.n = n;
    A.vx = vx; A.vy = vy; A.t_ref = 0.0; A.p_scale = p_scale;
    A.Hm = Hm; A.Wm = Wm; A.Hc = Hs + 1; A.Wc = Ws + 1;
    return run_cmax<WARP_LINVEL_F32>(A, sigma, flags, objective, obj_param, result, iwe_out, diwe_out, workspace,
                                     workspace_bytes, static_cast<cudaStream_t>(stream));
}

int evk_cmax_linvel_variance_f64(const double *x, const double *y, const double *t, const double *p, int64_t n,
                                 double p_scale, double vx, double vy, double t_ref, int Hm, int Wm, int Hs, int Ws,
                                 double sigma, unsigned flags, double *result, float *iwe_out, float *diwe_out,
                                 void *workspace, size_t workspace_bytes, void *stream)
{
    return evk_cmax_linvel_objective_f64(x, y, t, p, n, p_scale, vx, vy, t_ref, Hm, Wm, Hs, Ws, sigma, flags, 0, 0.0, result,
                                         iwe_out, diwe_out, workspace, workspace_bytes, stream);
}

int evk_cmax_linvel_variance_f32(const float *x, const float *y, const float *t_rel, const float *p, int64_t n,
                                 float p_scale, float vx, float vy, int Hm, int Wm, int Hs, int Ws, double sigma,
                                 unsigned flags, double *result, float *iwe_out, float *diwe_out, void *workspace,
                                 size_t workspace_bytes, void *stream)
{
    return evk_cmax_linvel_objective_f32(x, y, t_rel, p, n, p_scale, vx, vy, Hm, Wm, Hs, Ws, sigma, flags, 0, 0.0, result,
                                         iwe_out, diwe_out, workspace, workspace_bytes, stream);
}

int evk_cmax_linvel_partial_f64(const double *x, const double *y, const double *t, const double *p, int64_t n, double p_scale,
                                double vx, double vy, double t_ref, int Hm, int Wm, int Hs, int Ws, unsigned flags,
                                float *images_out, unsigned long long *oob_out, void *workspace, size_t workspace_bytes, void *stream)
{
    using namespace evk;
    if (!images_out || (n > 0 && (!x || !y || !t || !p))) { set_error("evk_cmax_linvel_partial_f64: null array"); return EVK_E_ARG; }
    CmaxArgs A{};
    A.x = x; A.y = y; A.t = t; A.p = p; A.n = n;
    A.vx = vx; A.vy = vy; A.t_ref = t_ref; A.p_scale = p_scale;
    A.Hm = Hm; A.Wm = Wm; A.Hc = Hs + 1; A.Wc = Ws + 1;
    return run_cmax<WARP_LINVEL_F64>(A, 0.0, flags, 0, 0.0, nullptr, nullptr, nullptr, workspace, workspace_bytes,
                                     static_cast<cudaStream_t>(stream), images_out, oob_out);
}

int evk_cmax_linvel_partial_f32(const float *x, const float *y, const float *t_rel, const float *p, int64_t n, float p_scale,
                                float vx, float vy, int Hm, int Wm, int Hs, int Ws, unsigned flags, float *images_out,
                                unsigned long long *oob_out, void *workspace, size_t workspace_bytes, void *stream)
{
    using namespace evk;
    if (!images_out || (n > 0 && (!x || !y || !t_rel || !p))) { set_error("evk_cmax_linvel_partial_f32: null array"); return EVK_E_ARG; }
    CmaxArgs A{};
    A.x = x; A.y = y; A.t = t_rel; A.p = p; A.n = n;
    A.vx = vx; A.vy = vy; A.t_ref = 0.0; A.p_scale = p_scale;
    A.Hm = Hm; A.Wm = Wm; A.Hc = Hs + 1; A.Wc = Ws + 1;
    return run_cmax<WARP_LINVEL_F32>(A, 0.0, flags, 0, 0.0, nullptr, nullptr, nullptr, workspace, workspace_bytes,
                                     static_cast<cudaStream_t>(stream), images_out, oob_out);
}

int evk_cmax_peer_tail_f32(const float *const *peer_images, const unsigned long long *const *peer_oob, int world, int Hc, int Wc,
                           double sigma, unsigned flags, double *result, void *workspace, size_t workspace_bytes, void *stream)
{
    using namespace evk;
    if (!peer_images || !peer_oob || world < 1 || world > kMaxCmaxPeers || Hc < 2 || Wc < 2 || !result || !workspace) {
        set_error("evk_cmax_peer_tail_f32: bad arguments (1 <= world <= %d)", kMaxCmaxPeers);
        return EVK_E_ARG;
    }
    if (((uintptr_t)workspace & 255) != 0) { set_error("evk_cmax_peer_tail_f32: workspace must be 256-byte aligned"); return EVK_E_ARG; }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CmaxWorkspace ws;
    const size_t need = carve(workspace, Hc - 1, Wc - 1, &ws);
    if (workspace_bytes < need) { set_error("evk_cmax_peer_tail_f32: workspace of %zu bytes required", need); return EVK_E_WORKSPACE; }
    BlurTaps taps{};
    double mix_a = 1.0, mix_b = 0.0;
    const int do_blur = sigma > 0.0;
    if (do_blur) {
        int rc = make_taps(sigma, &taps);
        if (rc) return rc;
        if (taps.r > kFusedMaxR) { set_error("evk_cmax_peer_tail_f32: blur radius %d > %d", taps.r, kFusedMaxR); return EVK_E_UNSUPPORTED; }
        if (!(flags & EVK_CMAX_NO_CHANNEL_MIX)) mix_coeffs(taps, &mix_a, &mix_b);
    }
    CmaxPeers P{};
    P.world = world;
    for (int r = 0; r < world; ++r) {
        if (!peer_images[r] || !peer_oob[r]) { set_error("evk_cmax_peer_tail_f32: peer %d: null pointer", r); return EVK_E_ARG; }
        P.img[r] = peer_images[r];
        P.oob[r] = peer_oob[r];
    }
    // the sums and the ticket of the tail (gsums .. oob are contiguous)
    EVK_CUDA(cudaMemsetAsync(ws.gsums, 0, (size_t)((char *)(ws.oob + 1) - (char *)ws.gsums), st));
    prof_count(1);
    dim3 tgrid((Wc + kTileX - 1) / kTileX, (Hc + kTileY - 1) / kTileY), tblock(kTileX, kTileY);
    cmax_fused_var_tail_kernel_t<true><<<tgrid, tblock, 0, st>>>(P, nullptr, nullptr, 1, Hc, Wc, taps, do_blur, (flags & EVK_CMAX_WANT_GRAD) ? 1 : 0,
                                                                  mix_a, mix_b, nullptr, nullptr, ws.sums, ws.gmax, ws.oob, result, ws.w);
    EVK_CUDA(cudaGetLastError());
    return EVK_OK;
}

int evk_cmax_flow_variance_f32(const float *x, const float *y, const float *t, const float *p, int64_t n,
                               const float *flow, float t0, int Hs, int Ws, double sigma, unsigned flags,
                               double *result, float *iwe_out, void *workspace, size_t workspace_bytes, void *stream)
{
    using namespace evk;
    if (!flow || (n > 0 && (!x || !y || !t || !p))) { set_error("evk_cmax_flow_variance_f32: null array"); return EVK_E_ARG; }
    CmaxArgs A{};
    A.x = x; A.y = y; A.t = t; A.p = p; A.n = n;
    A.flow = flow; A.flow_t0 = t0; A.p_scale = 1.0;
    A.Hm = Hs; A.Wm = Ws; A.Hc = Hs + 1; A.Wc = Ws + 1;
    return run_cmax<WARP_FLOW_F32>(A, sigma, flags, 0, 0.0, result, iwe_out, nullptr, workspace, workspace_bytes,
                                   static_cast<cudaStream_t>(stream));
}

int evk_iwe_objective_f32(const float *iwe, const float *diwe, int Hc, int Wc, double sigma, unsigned flags, int objective,
                          double obj_param, double *result, void *workspace, size_t workspace_bytes, void *stream)
{
    using namespace evk;
    if (!iwe || !result || !workspace || Hc < 2 || Wc < 2) { set_error("evk_iwe_objective_f32: bad arguments"); return EVK_E_ARG; }
    if (((uintptr_t)workspace & 255) != 0) { set_error("evk_iwe_objective_f32: workspace must be 256-byte aligned"); return EVK_E_ARG; }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CmaxWorkspace ws;
    const size_t need = carve(workspace, Hc - 1, Wc - 1, &ws);
    if (workspace_bytes < need) { set_error("evk_iwe_objective_f32: workspace of %zu bytes required", need); return EVK_E_WORKSPACE; }
    const int npix = Hc * Wc;
    const bool grad = (flags & EVK_CMAX_WANT_GRAD) != 0 && diwe != nullptr;
    EVK_CUDA(cudaMemsetAsync(ws.gsums, 0, (size_t)((char *)(ws.oob + 1) - (char *)ws.gsums), st));
    prof_count(1);
    cmax_planar_kernel<<<(npix + 255) / 256, 256, 0, st>>>(iwe, grad ? diwe : nullptr, npix, ws.I, ws.D0, ws.D1, ws.sums);
    return launch_tail(ws, Hc, Wc, sigma, flags, objective, obj_param, grad, result, st);
}

int evk_variance_objective_f32(const float *iwe, const float *diwe, int Hc, int Wc, double sigma, unsigned flags,
                               double *result, void *workspace, size_t workspace_bytes, void *stream)
{
    return evk_iwe_objective_f32(iwe, diwe, Hc, Wc, sigma, flags, 0, 0.0, result, workspace, workspace_bytes, stream);
}

int evk_gaussian_blur_f32(const float *img, int H, int W, double sigma, float *out, float *tmp, void *stream)
{
    using namespace evk;
    if (!img || !out || !tmp || H < 1 || W < 1) { set_error("evk_gaussian_blur_f32: bad arguments"); return EVK_E_ARG; }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    BlurTaps taps{};
    const int do_blur = sigma > 0.0;
    if (do_blur) {
        int rc = make_taps(sigma, &taps);
        if (rc) return rc;
    }
    const int g = (H * W + 255) / 256;
    prof_count(do_blur ? 2 : 1);
    if (do_blur) cmax_blur_axis0_kernel<<<g, 256, 0, st>>>(img, tmp, H, W, taps);
    cmax_blur_axis1_store_kernel<<<g, 256, 0, st>>>(tmp, img, H, W, taps, do_blur, out);
    EVK_CUDA(cudaGetLastError());
    return EVK_OK;
}

static int model_dims(int model) { return model == EVK_WARP_LINVEL ? 2 : model == EVK_WARP_ROTATION ? 3 : model == EVK_WARP_XYZTHETA ? 4 : -1; }

static int check_model(const char *fn, int model, const double *params, int dims)
{
    const int d = model_dims(model);
    if (d < 0 || !params || dims != d) {
        evk::set_error("%s: model %d takes %d parameters (params %p, dims %d)", fn, model, d, (const void *)params, dims);
        return EVK_E_ARG;
    }
    return EVK_OK;
}

int evk_cmax_model_objective_f64(int model, const double *params, int dims, const double *x, const double *y, const double *t,
                                 const double *p, int64_t n, double p_scale, double t_ref, int Hm, int Wm, int Hs, int Ws,
                                 double sigma, unsigned flags, int objective, double obj_param, double *result, double *grad,
                                 void *workspace, size_t workspace_bytes, void *stream)
{
    using namespace evk;
    int rc = check_model("evk_cmax_model_objective_f64", model, params, dims);
    if (rc) return rc;
    if (!grad) { set_error("evk_cmax_model_objective_f64: grad is NULL"); return EVK_E_ARG; }
    if (n > 0 && (!x || !y || !t || !p)) { set_error("evk_cmax_model_objective_f64: null event array"); return EVK_E_ARG; }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (model == EVK_WARP_LINVEL) {
        rc = evk_cmax_linvel_objective_f64(x, y, t, p, n, p_scale, params[0], params[1], t_ref, Hm, Wm, Hs, Ws, sigma, flags, objective,
                                           obj_param, result, nullptr, nullptr, workspace, workspace_bytes, stream);
        if (rc) return rc;
        EVK_CUDA(cudaMemcpyAsync(grad, result + 1, 2 * sizeof(double), cudaMemcpyDefault, st));
        return EVK_OK;
    }
    CmaxArgs A{};
    A.x = x; A.y = y; A.t = t; A.p = p; A.n = n;
    A.t_ref = t_ref; A.p_scale = p_scale;
    A.Hm = Hm; A.Wm = Wm; A.Hc = Hs + 1; A.Wc = Ws + 1;
    for (int k = 0; k < dims; ++k) A.params[k] = params[k];
    if (model == EVK_WARP_ROTATION)
        return run_cmax<WARP_ROT_F64>(A, sigma, flags, objective, obj_param, result, nullptr, nullptr, workspace, workspace_bytes, st,
                                      nullptr, nullptr, grad);
    return run_cmax<WARP_XYZT_F64>(A, sigma, flags, objective, obj_param, result, nullptr, nullptr, workspace, workspace_bytes, st,
                                   nullptr, nullptr, grad);
}

int evk_cmax_model_objective_f32(int model, const double *params, int dims, const float *x, const float *y, const float *t_rel,
                                 const float *p, int64_t n, float p_scale, int Hm, int Wm, int Hs, int Ws, double sigma,
                                 unsigned flags, int objective, double obj_param, double *result, double *grad, void *workspace,
                                 size_t workspace_bytes, void *stream)
{
    using namespace evk;
    int rc = check_model("evk_cmax_model_objective_f32", model, params, dims);
    if (rc) return rc;
    if (!grad) { set_error("evk_cmax_model_objective_f32: grad is NULL"); return EVK_E_ARG; }
    if (n > 0 && (!x || !y || !t_rel || !p)) { set_error("evk_cmax_model_objective_f32: null event array"); return EVK_E_ARG; }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (model == EVK_WARP_LINVEL) {
        rc = evk_cmax_linvel_objective_f32(x, y, t_rel, p, n, p_scale, (float)params[0], (float)params[1], Hm, Wm, Hs, Ws, sigma, flags,
                                           objective, obj_param, result, nullptr, nullptr, workspace, workspace_bytes, stream);
        if (rc) return rc;
        EVK_CUDA(cudaMemcpyAsync(grad, result + 1, 2 * sizeof(double), cudaMemcpyDefault, st));
        return EVK_OK;
    }
    CmaxArgs A{};
    A.x = x; A.y = y; A.t = t_rel; A.p = p; A.n = n;
    A.t_ref = 0.0; A.p_scale = p_scale;
    A.Hm = Hm; A.Wm = Wm; A.Hc = Hs + 1; A.Wc = Ws + 1;
    for (int k = 0; k < dims; ++k) A.params[k] = params[k];
    if (model == EVK_WARP_ROTATION)
        return run_cmax<WARP_ROT_F32>(A, sigma, flags, objective, obj_param, result, nullptr, nullptr, workspace, workspace_bytes, st,
                                      nullptr, nullptr, grad);
    return run_cmax<WARP_XYZT_F32>(A, sigma, flags, objective, obj_param, result, nullptr, nullptr, workspace, workspace_bytes, st,
                                   nullptr, nullptr, grad);
}

int evk_cmax_model_warp_f64(int model, const double *params, int dims, const double *x, const double *y, const double *t,
                            const double *p, int64_t n, double t_ref, int Hm, int Wm, unsigned flags, float *xw, float *yw, float *pw,
                            float *jx, float *jy, void *stream)
{
    using namespace evk;
    int rc = check_model("evk_cmax_model_warp_f64", model, params, dims);
    if (rc) return rc;
    if (model == EVK_WARP_LINVEL) { set_error("evk_cmax_model_warp_f64: linvel images come from evk_cmax_linvel_objective_f64"); return EVK_E_ARG; }
    if (n < 0 || (n > 0 && (!x || !y || !t || !p || !xw || !yw || !pw)) || (!jx != !jy)) {
        set_error("evk_cmax_model_warp_f64: bad arguments");
        return EVK_E_ARG;
    }
    if (n == 0) return EVK_OK;
    CmaxArgs A{};
    A.x = x; A.y = y; A.t = t; A.p = p; A.n = n;
    A.t_ref = t_ref; A.p_scale = 1.0; A.abs_polarity = (flags & EVK_CMAX_ABS_POLARITY) ? 1 : 0;
    A.Hm = Hm; A.Wm = Wm;
    for (int k = 0; k < dims; ++k) A.params[k] = params[k];
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    prof_count(1);
    if (model == EVK_WARP_ROTATION)
        cmax_model_warp_kernel<WARP_ROT_F64><<<grid_simple(n, 256 * 4), 256, 0, st>>>(A, xw, yw, pw, jx, jy);
    else
        cmax_model_warp_kernel<WARP_XYZT_F64><<<grid_simple(n, 256 * 4), 256, 0, st>>>(A, xw, yw, pw, jx, jy);
    EVK_CUDA(cudaGetLastError());
    return EVK_OK;
}

int evk_iwe_objective_k_f32(const float *iwe, const float *diwe, int K, int Hc, int Wc, double sigma, unsigned flags, int objective,
                            double obj_param, double *result, double *grad, void *workspace, size_t workspace_bytes, void *stream)
{
    using namespace evk;
    if (!iwe || !result || !workspace || Hc < 2 || Wc < 2 || K < 0 || K > kMaxDims || (K > 0 && (!diwe || !grad))) {
        set_error("evk_iwe_objective_k_f32: bad arguments (0 <= K <= %d)", kMaxDims);
        return EVK_E_ARG;
    }
    if (((uintptr_t)workspace & 255) != 0) { set_error("evk_iwe_objective_k_f32: workspace must be 256-byte aligned"); return EVK_E_ARG; }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CmaxWorkspace ws;
    const size_t need = carve(workspace, Hc - 1, Wc - 1, &ws);
    if (workspace_bytes < need) { set_error("evk_iwe_objective_k_f32: workspace of %zu bytes required", need); return EVK_E_WORKSPACE; }
    const int npix = Hc * Wc;
    EVK_CUDA(cudaMemsetAsync(ws.gsums, 0, (size_t)((char *)(ws.oob + 1) - (char *)ws.gsums), st));
    prof_count(1);
    cmax_planar_kernel<<<(npix + 255) / 256, 256, 0, st>>>(iwe, nullptr, npix, ws.I, ws.D0, ws.D1, ws.sums);
    auto pass2 = [&](const float *W) -> int {
        prof_count(1);
        cmax_dot_k_kernel<<<(npix + 255) / 256, 256, 0, st>>>(W, diwe, K, npix, ws.gk);
        EVK_CUDA(cudaGetLastError());
        return EVK_OK;
    };
    return model_tail(ws, Hc, Wc, sigma, flags, objective, obj_param, (flags & EVK_CMAX_WANT_GRAD) != 0 && K > 0, K, pass2, result,
                      grad, st);
}

int evk_cmax_linvel_objective_batch_f64(const double *x, const double *y, const double *t, const double *p, int64_t n,
                                        double p_scale, const double *params_host, int n_params, double t_ref, int Hm, int Wm,
                                        int Hs, int Ws, double sigma, unsigned flags, int objective, double obj_param,
                                        double *results, void *workspace, size_t workspace_bytes, void *stream)
{
    using namespace evk;
    if (n < 0 || (n > 0 && (!x || !y || !t || !p)) || !params_host || n_params < 1 || n_params > kMaxCandidates || !results || !workspace) {
        set_error("evk_cmax_linvel_objective_batch_f64: bad arguments (1 <= n_params <= %d)", kMaxCandidates);
        return EVK_E_ARG;
    }
    if (((uintptr_t)workspace & 255) != 0) { set_error("evk_cmax batch: workspace must be 256-byte aligned"); return EVK_E_ARG; }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CmaxWorkspace ws;
    const size_t need = carve(workspace, Hs, Ws, &ws);
    if (workspace_bytes < need) { set_error("evk_cmax batch: workspace of %zu bytes required", need); return EVK_E_WORKSPACE; }
    CmaxArgs A{};
    A.x = x; A.y = y; A.t = t; A.p = p; A.n = n;
    A.t_ref = t_ref; A.p_scale = p_scale;
    A.Hm = Hm; A.Wm = Wm; A.Hc = Hs + 1; A.Wc = Ws + 1;
    A.abs_polarity = (flags & EVK_CMAX_ABS_POLARITY) ? 1 : 0;
    A.replicas = 1; A.acc = ws.acc; A.oob = ws.oob;
    const int npix = A.Hc * A.Wc;
    const bool grad = (flags & EVK_CMAX_WANT_GRAD) != 0;
    Candidates C{};
    C.n = n_params;
    for (int k = 0; k < n_params; ++k) { C.vx[k] = params_host[2 * k]; C.vy[k] = params_host[2 * k + 1]; }
    // bsums, btickets, gsums, gmax, sums, oob and the accumulators are contiguous: one memset
    EVK_CUDA(cudaMemsetAsync(ws.bsums, 0, (size_t)((char *)ws.acc - (char *)ws.bsums) + (size_t)n_params * npix * kBlockFloats * sizeof(float), st));
    if (n > 0) {
        ProfScope prof(st);
        prof_count(1);
        if (grad) cmax_scatter_batch_kernel<WARP_LINVEL_F64, true><<<grid_for(cmax_scatter_batch_kernel<WARP_LINVEL_F64, true>, 256, n, 256 * 2), 256, 0, st>>>(A, C);
        else cmax_scatter_batch_kernel<WARP_LINVEL_F64, false><<<grid_for(cmax_scatter_batch_kernel<WARP_LINVEL_F64, false>, 256, n, 256 * 2), 256, 0, st>>>(A, C);
        EVK_CUDA(cudaGetLastError());
    }
    if (objective == OBJ_VARIANCE && (sigma <= 0.0 || (int)(4.0 * sigma + 0.5) <= kFusedMaxR)) {
        // all candidates' tails in ONE launch (blockIdx.z = candidate)
        BlurTaps taps{};
        double mix_a = 1.0, mix_b = 0.0;
        const int do_blur = sigma > 0.0;
        if (do_blur) {
            int rc = make_taps(sigma, &taps);
            if (rc) return rc;
            if (!(flags & EVK_CMAX_NO_CHANNEL_MIX)) mix_coeffs(taps, &mix_a, &mix_b);
        }
        prof_count(1);
        dim3 tgrid((A.Wc + kTileX - 1) / kTileX, (A.Hc + kTileY - 1) / kTileY, n_params), tblock(kTileX, kTileY);
        cmax_fused_var_tail_kernel_t<false><<<tgrid, tblock, 0, st>>>(CmaxPeers{}, ws.acc, nullptr, 1, A.Hc, A.Wc, taps, do_blur, grad ? 1 : 0, mix_a, mix_b, nullptr,
                                                               nullptr, ws.bsums, ws.btickets, ws.oob, results);
        EVK_CUDA(cudaGetLastError());
        return EVK_OK;
    }
    for (int k = 0; k < n_params; ++k) {
        // per-candidate image-space tail on the shared scratch images (stream-ordered)
        EVK_CUDA(cudaMemsetAsync(ws.gsums, 0, (size_t)((char *)ws.oob - (char *)ws.gsums), st));   // keep the oob counter
        prof_count(1);
        cmax_gather_kernel<<<(npix + 255) / 256, 256, 0, st>>>(ws.acc + (size_t)k * npix * kBlockFloats, nullptr, 1, A.Hc, A.Wc, ws.I, ws.D0,
                                                                ws.D1, nullptr, nullptr, ws.sums);
        int rc = launch_tail(ws, A.Hc, A.Wc, sigma, flags, objective, obj_param, grad, results + 12 * k, st);
        if (rc) return rc;
    }
    return EVK_OK;
}

}  // extern "C"
