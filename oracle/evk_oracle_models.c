/*
 * evk_oracle_models.c -- CPU restatement of get_iwe for the rotation and xyztheta motion models.
 * TEST INFRASTRUCTURE ONLY (same rules and rounding points as evk_oracle.c; build with -ffp-contract=off).
 *
 * The reference leaves both models empty (lib/contrast_max/warps.py:63-83); their formulas are those of
 * event_utils_b200/contrast_max/warps.py and include/evk.h.  Everything after the warp is the reference's:
 *   get_iwe                 lib/contrast_max/objectives.py:184-192  (f64 warp and bounds mask, then f32)
 *   bounds mask             lib/util/event_util.py:26-27
 *   events_to_image_drv     lib/representations/image.py:179-217, with `dims` derivative channels instead of
 *                           the 2 that image.py:210 allocates
 *   derivative taps         lib/representations/image.py:131-135
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

#define EVO_API __attribute__((visibility("default")))

static inline int64_t trunc_to_long(float v)
{
    if (!(v == v) || v >= 9.2e18f || v <= -9.2e18f) return INT64_MIN;
    return (int64_t)v;
}

static inline int wrap_index(int64_t i, int64_t size, int64_t *out)
{
    if (i < 0) i += size;
    if (i < 0 || i >= size) return 0;
    *out = i;
    return 1;
}

/* model 1: rotation (cx, cy, omega), dims 3;  model 2: xyztheta (vx, vy, vz, omega), dims 4.  Returns dims. */
static int model_warp(int model, const double *q, double x, double y, double d, double *xw, double *yw, double *jx, double *jy)
{
    if (model == 1) {
        double th = -(q[2] * d), c = cos(th), s = sin(th);
        double X = x - q[0], Y = y - q[1];
        *xw = q[0] + c * X - s * Y;
        *yw = q[1] + s * X + c * Y;
        jx[0] = 1 - c; jx[1] = s; jx[2] = d * (*yw - q[1]);
        jy[0] = -s; jy[1] = 1 - c; jy[2] = -(d * (*xw - q[0]));
        return 3;
    }
    *xw = x - d * (q[0] + q[2] * x - q[3] * y);
    *yw = y - d * (q[1] + q[2] * y + q[3] * x);
    jx[0] = -d; jx[1] = 0.0; jx[2] = -(d * x); jx[3] = d * y;
    jy[0] = 0.0; jy[1] = -d; jy[2] = -(d * y); jy[3] = -(d * x);
    return 4;
}

/* iwe: (Hs+1)*(Ws+1) f32 zero-filled; diwe: dims*(Hs+1)*(Ws+1) f32 zero-filled or NULL.  Returns the number of
 * events whose footprint indexes outside the canvas (the reference's IndexError). */
EVO_API int64_t evo_iwe_model(int model, const double *params, const double *x, const double *y, const double *t, const double *p,
                              int64_t n, double t_ref, int Hm, int Wm, int Hs, int Ws, int use_polarity, float *iwe, float *diwe)
{
    const int Hc = Hs + 1, Wc = Ws + 1;
    const float clipx = (float)(Wc - 1), clipy = (float)(Hc - 1);
    const int64_t plane = (int64_t)Hc * Wc;
    int64_t oob = 0;
    for (int64_t i = 0; i < n; ++i) {
        double pp = use_polarity ? p[i] : fabs(p[i]);
        double d = t[i] - t_ref, xw, yw, jx[4], jy[4];
        int dims = model_warp(model, params, x[i], y[i], d, &xw, &yw, jx, jy);
        double mk = ((xw <= 0.0 || xw > (double)Wm) ? 0.0 : 1.0);
        mk *= ((yw <= 0.0 || yw > (double)Hm) ? 0.0 : 1.0);
        float xf = (float)(xw * mk), yf = (float)(yw * mk), pf = (float)(pp * mk);
        float m2 = (xf >= clipx ? 0.0f : 1.0f) * (yf >= clipy ? 0.0f : 1.0f);
        float pxf = floorf(xf), pyf = floorf(yf);
        float dx = xf - pxf, dy = yf - pyf;
        int64_t px = trunc_to_long(pxf * m2), py = trunc_to_long(pyf * m2);
        float w = pf * m2;
        int64_t x0, x1, y0, y1;
        if (!wrap_index(px, Wc, &x0) || !wrap_index(px + 1, Wc, &x1) ||
            !wrap_index(py, Hc, &y0) || !wrap_index(py + 1, Hc, &y1)) { ++oob; continue; }
        float ox = 1.0f - dx, oy = 1.0f - dy;
        iwe[y0 * Wc + x0] += (w * ox) * oy;
        iwe[y0 * Wc + x1] += (w * dx) * oy;
        iwe[y1 * Wc + x0] += (w * ox) * dy;
        iwe[y1 * Wc + x1] += (w * dx) * dy;
        if (!diwe) continue;
        for (int k = 0; k < dims; ++k) {
            /* image.py:211-213: w1 = jacobian_x * masked_ps, w2 = jacobian_y * masked_ps (f32) */
            float a1 = (float)(jx[k] * mk) * w, a2 = (float)(jy[k] * mk) * w;
            float *dk = diwe + k * plane;
            dk[y0 * Wc + x0] += a1 * (-oy) + a2 * (-ox);
            dk[y0 * Wc + x1] += a1 * oy + a2 * (-dx);
            dk[y1 * Wc + x0] += a1 * (-dy) + a2 * ox;
            dk[y1 * Wc + x1] += a1 * dy + a2 * dx;
        }
    }
    return oob;
}
