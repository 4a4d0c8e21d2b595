/*
 * evk.h -- C ABI of libevk.so: B200 (sm_100a) kernels for the event_utils hot path.
 *
 * The reference (TimoStoff/event_utils) is pure Python and has NO FFI of its own; its
 * "operator API" is a set of module-level Python functions (SURVEY.md section 8b).  Each entry
 * point below is what a ctypes/cffi binding for one of those functions binds to; the reference
 * call site it replaces is cited as file:line (paths relative to the reference tree).
 * INTEGRATION.md shows the ctypes stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 on success, a negative EVK_E_* code on failure; it never throws
 *     across the ABI.  evk_last_error() returns a thread-local human-readable message.
 *   - unless the name says `_host`, all data pointers are caller-owned DEVICE pointers and all
 *     work is enqueued on the caller's stream (a cudaStream_t passed as void*); nothing
 *     synchronises.  No torch types anywhere.
 *   - `oob` (may be NULL) is a device counter the kernels increment once per event whose index
 *     falls outside the output (the reference raises IndexError for those, image.py:96-99);
 *     such events are never written.  The caller zeroes and reads it.
 *   - outputs are fully overwritten unless EVK_ACCUMULATE is set.
 */
#ifndef EVK_H_
#define EVK_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

#define EVK_VERSION 100 /* 0.1.0 */

/* error codes */
#define EVK_OK 0
#define EVK_E_ARG (-1)       /* bad argument (null pointer, negative size, ...) */
#define EVK_E_CUDA (-2)      /* a CUDA runtime call failed, see evk_last_error() */
#define EVK_E_WORKSPACE (-3) /* workspace too small */
#define EVK_E_DEVICE (-4)    /* not an sm_100 device */
#define EVK_E_UNSUPPORTED (-5)

/* flags shared by the scatter entry points */
#define EVK_ACCUMULATE 0x1u   /* add into `out` instead of overwriting it */
#define EVK_BILINEAR 0x2u     /* spatial 4-tap bilinear splat instead of nearest (truncate) */
#define EVK_CLIP 0x4u         /* events_to_image_torch(clip_out_of_range=True) semantics */
#define EVK_AUTO_SPAN 0x200000u    /* voxel: ignore the t0/dt arguments, take t[0] and t[n-1]-t[0] on the device */
#define EVK_WINDOW_PAIRS 0x100000u /* evk_voxel_windows_f32: offsets are (start,end) pairs, 2*n_windows entries */
#define EVK_NO_FOLD 0x800000u /* evk_voxel_f32: leave the sums in the quad workspace (out may be NULL); evk_voxel_fold_allreduce_f32 finishes */
#define EVK_PEER_MULTICAST 0x1000000u /* evk_voxel_fold_allreduce_f32: entry 0 of both pointer arrays is an NVLS multicast address */
#define EVK_WINDOW_NEGPOS 0x400000u /* evk_voxel_windows_f32: out is [n_windows][2][B][H][W], the [p>0] / [p<=0] split per window */
#define EVK_NEGPOS_TRUTHY 0x8u /* neg/pos split on numpy truthiness (p != 0) instead of p > 0 */
/* kernel variant selection, bits 8..11 (0 = pick automatically) */
#define EVK_VARIANT_SHIFT 8
#define EVK_VARIANT_MASK (0xFu << EVK_VARIANT_SHIFT)
#define EVK_VARIANT_AUTO (0u << EVK_VARIANT_SHIFT)
#define EVK_VARIANT_GLOBAL_RED (1u << EVK_VARIANT_SHIFT) /* one scalar red.global.add.f32 per tap */
#define EVK_VARIANT_VECTOR_RED (2u << EVK_VARIANT_SHIFT) /* one red.global.add.v4.f32 per tap pair, quad-layout workspace */
#define EVK_VARIANT_SMEM_TILE (3u << EVK_VARIANT_SHIFT)  /* the shared-memory form of the entry point: voxel / image = vector or scalar reductions behind a per-CTA
                                                          * fixed-point write-combining table (forced on; AUTO probes for contention); cmax = the whole image of
                                                          * warped events in the CTA's shared memory, flushed by TMA bulk reductions (cmax_onchip_kernel) */
#define EVK_VARIANT_WARP_AGG (4u << EVK_VARIANT_SHIFT)   /* warp-aggregated (match.any) global reds, for hot-spot streams */
#define EVK_VARIANT_ROUTED (5u << EVK_VARIANT_SHIFT)     /* voxel: output tiles in shared memory, events routed to the owning SM through L2-resident rings; tiles leave by TMA bulk reduction (correct, 2x SLOWER than AUTO: opt-in, DESIGN.md section 4) */
/* The routed kernel is a cooperative web of spin waits; a watchdog inside it gives up after 0.5 s without progress
 * (the kernel takes < 1 ms per 50 M events), lets the launch end with an INCOMPLETE grid and adds this mark to the
 * caller's `oob` counter -- the device never hangs.  Counter values >= the mark mean "result invalid", not index errors. */
#define EVK_ROUTED_ABORT_MARK (1ull << 62)

#define EVK_TS_REVERSE 0x80u  /* timestamp images: timestamp_reverse=True (image.py:318-319) */
#define EVK_TS_RAW 0x1000u    /* timestamp images: normalize_timestamps=False (image.py:261): weights = t as given */

/* cmax flags */
#define EVK_CMAX_WANT_GRAD 0x10u    /* also produce the analytic gradient */
#define EVK_CMAX_ABS_POLARITY 0x20u /* use_polarity=False: p <- |p| (objectives.py:184-185) */
#define EVK_CMAX_NO_CHANNEL_MIX 0x40u /* do NOT reproduce the 3-D blur channel mixing (objectives.py:253) */

int evk_version(void);
const char *evk_last_error(void);
/* 0 if the current device is compute capability 10.x, EVK_E_DEVICE otherwise */
int evk_device_check(void);

/* ---------------------------------------------------------------------------------------------
 * Measurement hooks (bench.py).  With profiling enabled every DOMINANT kernel launch of the
 * scatter entry points (voxel / image scatter, cmax scatter) is bracketed by a CUDA event pair
 * recorded on the launching stream, and every kernel launch of the library is counted.
 * evk_prof_collect() synchronises those events, returns the summed device time of the bracketed
 * launches in *ms, their number in *timed and the total number of kernel launches in *launches,
 * and resets the counters.
 * --------------------------------------------------------------------------------------------- */
int evk_prof_enable(int on);
int evk_prof_collect(double *ms, long long *timed, long long *launches);

/* ---------------------------------------------------------------------------------------------
 * Voxel grid.  Replaces events_to_voxel_torch, lib/representations/voxel_grid.py:114-153
 * (per-bin loop :136-151 -> events_to_image_torch image.py:88-95 -> index_put_).
 *   tau = ((t - t0) / dt) * (B-1)   (f32, this order);  V[b, trunc(y), trunc(x)] += p*max(0,1-|tau-b|)
 * t0, dt are explicit so that a sharded caller can pass the GLOBAL values (voxel_grid.py:133-134
 * derives them from ts[0], ts[-1]).  x,y,t,p: n floats each (SoA), any 4-byte alignment.
 * out: B*H*W floats, layout [B][H][W].
 * With EVK_BILINEAR the spatial part is a 4-tap bilinear splat on the same (H,W) grid
 * (trilinear voxel; an extension, not a reference function).
 * workspace: evk_voxel_workspace_bytes() bytes (may be 0/NULL for the GLOBAL_RED variant).
 * --------------------------------------------------------------------------------------------- */
size_t evk_voxel_workspace_bytes(int B, int H, int W, unsigned flags);
int evk_voxel_f32(const float *x, const float *y, const float *t, const float *p, int64_t n,
                  float t0, float dt, int B, int H, int W, unsigned flags, float *out,
                  void *workspace, size_t workspace_bytes, unsigned long long *oob, void *stream);

/* Positive and negative events into separate grids in ONE pass.  Replaces
 * events_to_neg_pos_voxel_torch, lib/representations/voxel_grid.py:155-182 (two full
 * events_to_voxel_torch calls with weights [p>0] and [p<=0], :172-175); with EVK_NEGPOS_TRUTHY the
 * numpy flavour's split np.where(ps,1,0) / np.where(ps,0,1) (:234-235).
 * out_pos_neg: 2*B*H*W floats, [0] = positive grid, [1] = negative grid.
 * workspace: 2 * evk_voxel_workspace_bytes(B,H,W,flags) bytes. */
int evk_voxel_negpos_f32(const float *x, const float *y, const float *t, const float *p, int64_t n,
                         float t0, float dt, int B, int H, int W, unsigned flags, float *out_pos_neg,
                         void *workspace, size_t workspace_bytes, unsigned long long *oob,
                         void *stream);

/* Same, events given as one interleaved (N,4) [x,y,t,p] f32 array (the data-loader layout,
 * lib/data_loaders/base_dataset.py:306,510); ev must be 16-byte aligned. */
int evk_voxel_aos_f32(const float *ev, int64_t n, float t0, float dt, int B, int H, int W,
                      unsigned flags, float *out, void *workspace, size_t workspace_bytes,
                      unsigned long long *oob, void *stream);

/* Same, events in the reference's STORAGE layout (row f4): int16 x, int16 y, float64 t, bool/uint8 p as
 * the HDF5 and memmap formats hold them (lib/data_formats/event_packagers.py:90-93,
 * h5_to_memmap.py:115-117), polarity mapped p*2-1 like the loaders do (hdf5_dataset.py:22,
 * memmap_dataset.py:24).  Timestamps are made relative to t_first in float64, then cast to float32;
 * dt = (float)(t_last - t_first).  13 B/event instead of 16 and no host-side casts. */
int evk_voxel_packed_f32(const int16_t *x, const int16_t *y, const double *t, const uint8_t *p, int64_t n,
                         double t_first, double t_last, int B, int H, int W, unsigned flags, float *out,
                         void *workspace, size_t workspace_bytes, unsigned long long *oob, void *stream);

/* Multi-GPU finish of a sharded voxel build (no reference counterpart: the reference is single-process;
 * SURVEY 8e): after every rank has run evk_voxel_f32(..., EVK_NO_FOLD) on its shard into a workspace that
 * its peers can address (CUDA IPC / symmetric memory over NVLink), and a cross-GPU barrier, each rank calls
 * this once: it reduces ITS slice of the pixels over all ranks' workspaces, folds the temporal quads into
 * the B bins and writes the result into every rank's [B][H][W] grid -- fold and all-reduce in one kernel
 * over peer memory.  A second cross-GPU barrier must follow before the grids are read or the workspaces
 * reused.  peer_workspaces / peer_outs: HOST arrays of `world` device pointers, index = rank.
 * With EVK_PEER_MULTICAST entry 0 of each array is the buffer's NVLS multicast address instead (the
 * other entries are ignored): the NVSwitch sums the quads (multimem.ld_reduce) and fans the result out
 * (multimem.st), so the per-GPU link traffic no longer grows with the number of ranks. */
int evk_voxel_fold_allreduce_f32(const void *const *peer_workspaces, float *const *peer_outs, int world,
                                 int rank, int B, int H, int W, unsigned flags, void *stream);

/* Batched windows (voxel_grids_fixed_n_torch, voxel_grid.py:37-57; BaseVoxelDataset windows,
 * base_dataset.py:322-367): window w covers events [offsets[w], offsets[w+1]) and writes
 * out[w] ([n_windows][B][H][W]); t0/dt per window are taken from the window's first / last
 * timestamp exactly as voxel_grid.py:133-134 does.  offsets: n_windows+1 int64 on the device.
 * With EVK_WINDOW_PAIRS offsets holds 2*n_windows entries, (start,end) per window (windows may then
 * overlap or leave gaps, as events_to_voxel_timesync_torch's do, voxel_grid.py:105-106).
 * With EVK_WINDOW_NEGPOS out is [n_windows][2][B][H][W]: per window the two grids of
 * events_to_neg_pos_voxel_torch (voxel_grid.py:155-182), what BaseVoxelDataset.get_voxel_grid builds
 * with combined_voxel_channels=False (base_dataset.py:449-453).
 * n_events_hint: total number of events covered (0 = unknown), used only to size the launch. */
int evk_voxel_windows_f32(const float *x, const float *y, const float *t, const float *p,
                          const int64_t *offsets, int n_windows, int64_t n_events_hint, int B, int H,
                          int W, unsigned flags, float *out, unsigned long long *oob, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Event image.  Replaces events_to_image_torch, lib/representations/image.py:46-100 and
 * interpolate_to_image, image.py:102-115.
 *   nearest : img[trunc(y)*m, trunc(x)*m] += p           (m = [x<clipx][y<clipy] with EVK_CLIP;
 *             NOTE the weight is not masked, image.py:94-95)
 *   bilinear: 4-tap splat of p*m at floor(x)*m, floor(y)*m with the unmasked fractions
 * Himg, Wimg are the CANVAS sizes (sensor+1 when bilinear and padding, image.py:64-67); the
 * caller derives clipx/clipy as image.py:73-74 does.  `fill` is the background (`default`).
 * --------------------------------------------------------------------------------------------- */
size_t evk_image_workspace_bytes(int Himg, int Wimg, unsigned flags);
int evk_image_f32(const float *x, const float *y, const float *p, int64_t n, int Himg, int Wimg,
                  float clipx, float clipy, unsigned flags, float fill, float *out,
                  void *workspace, size_t workspace_bytes, unsigned long long *oob, void *stream);

/* Average-timestamp images of the positive / negative events.  Replaces
 * events_to_timestamp_image_torch, lib/representations/image.py:286-353 (and the numpy flavour
 * :219-284 after its casts).  t_first / t_last are ts[0] / ts[-1]; Himg, Wimg the canvas
 * (sensor+1 with padding); clipx/clipy as image.py:311-312.  out_pos / out_neg: Himg*Wimg floats.
 * workspace: evk_timestamp_image_workspace_bytes() bytes, 16-byte aligned. */
size_t evk_timestamp_image_workspace_bytes(int Himg, int Wimg);
int evk_timestamp_image_f32(const float *x, const float *y, const float *t, const float *p, int64_t n,
                            float t_first, float t_last, int Himg, int Wimg, float clipx, float clipy,
                            unsigned flags, float *out_pos, float *out_neg, void *workspace,
                            size_t workspace_bytes, unsigned long long *oob, void *stream);

/* Integer-exact event-count image (nearest, weight +1 per event): out is u32 [Himg][Wimg].
 * The bit-exact form of events_to_image(_torch) for ps == 1 (image.py:37-38, :95). */
int evk_count_u32(const float *x, const float *y, int64_t n, int Himg, int Wimg, float clipx,
                  float clipy, unsigned flags, unsigned int *out, unsigned long long *oob,
                  void *stream);

/* ---------------------------------------------------------------------------------------------
 * The reference's lower-level splat / gather helpers, for callers that use them directly.
 *   evk_splat_idx_f32       interpolate_to_image, lib/representations/image.py:102-115
 *                           (in place on img [H][W]; px,py int64; dx,dy,w f32)
 *   evk_splat_drv_idx_f32   interpolate_to_derivative_img, image.py:117-136
 *                           (in place on dimg [K][H][W]; w1,w2 are [K][n])
 *   evk_image_drv_f32       events_to_image_drv, image.py:162-217 after its f64->f32 casts
 *                           (:179-183): x,y,p f32, Jacobians jx,jy [K][n] f32 (K may be 0),
 *                           writes img [Himg][Wimg] and dimg [K][Himg][Wimg]
 *   evk_gather_bilinear_f64 image_to_event_weights, image.py:138-160 (f64, img [H][W] f64)
 * --------------------------------------------------------------------------------------------- */
int evk_splat_idx_f32(const int64_t *px, const int64_t *py, const float *dx, const float *dy,
                      const float *w, int64_t n, int H, int W, float *img, unsigned long long *oob,
                      void *stream);
int evk_splat_drv_idx_f32(const int64_t *px, const int64_t *py, const float *dx, const float *dy,
                          const float *w1, const float *w2, int K, int64_t n, int H, int W,
                          float *dimg, unsigned long long *oob, void *stream);
int evk_image_drv_f32(const float *x, const float *y, const float *p, const float *jx, const float *jy,
                      int K, int64_t n, int Himg, int Wimg, float clipx, float clipy, unsigned flags,
                      float *img, float *dimg, unsigned long long *oob, void *stream);
int evk_gather_bilinear_f64(const double *x, const double *y, int64_t n, const double *img, int H,
                            int W, double *out, unsigned long long *oob, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Dense-flow warp.  Replaces warp_events_flow_torch, lib/transforms/optic_flow.py:5-46
 * (F.grid_sample bilinear, align_corners=True, zero padding, :37-44).
 * flow: [2][H][W] f32.  xw/yw: n floats.  x' = x + u(x,y)*(t-t0), y' = y + v(x,y)*(t-t0).
 * workspace (optional, evk_warp_flow_workspace_bytes(), 16-byte aligned): lets the kernel re-lay the
 * flow out as {u,v} pairs so that the two taps of an image row are one 16-byte load.
 * --------------------------------------------------------------------------------------------- */
size_t evk_warp_flow_workspace_bytes(int H, int W);
int evk_warp_flow_f32(const float *x, const float *y, const float *t, int64_t n, const float *flow,
                      int H, int W, float t0, float *xw, float *yw, void *workspace,
                      size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Contrast maximisation, fused: linvel warp -> bounds mask -> bilinear IWE (+ derivative
 * images) -> Gaussian blur -> variance objective (+ analytic gradient).
 * Replaces variance_objective.evaluate_function / evaluate_gradient,
 * lib/contrast_max/objectives.py:211-264, i.e. get_iwe :165-199, linvel_warp.warp warps.py:51-61,
 * events_bounds_mask event_util.py:15-28, events_to_image_drv image.py:162-217,
 * scipy gaussian_filter + np.var / np.mean objectives.py:233-234,253-262.
 *   x,y,t,p : n doubles each (the reference API hands f64 numpy arrays) -- `_f64`, parity mode
 *             n floats each, t already relative to t_ref  -- `_f32`, fast mode
 *   (Hm,Wm) : img_size of the bounds mask;  (Hs,Ws): sensor size of the IWE canvas, which is
 *             (Hs+1)x(Ws+1); the reference always uses (180,240) (objectives.py:191-192).
 *   result  : 8 doubles on the device: f, g[0], g[1], sum(IWE), #events indexing outside the
 *             canvas (the reference's IndexError), var, and the un-mixed 2-D gradient (2)
 *             (g = 0 without EVK_CMAX_WANT_GRAD)
 *   iwe_out : optional (Hs+1)*(Ws+1) floats (the un-blurred IWE), diwe_out optional 2x that.
 *   p_scale : polarity multiplier (1, or 100 for the adaptive-lifespan branch objectives.py:225)
 *   workspace: evk_cmax_workspace_bytes(Hs,Ws) bytes of device scratch, 256-byte aligned.
 * --------------------------------------------------------------------------------------------- */
size_t evk_cmax_workspace_bytes(int Hs, int Ws);
int evk_cmax_linvel_variance_f64(const double *x, const double *y, const double *t, const double *p,
                                 int64_t n, double p_scale, double vx, double vy, double t_ref,
                                 int Hm, int Wm, int Hs, int Ws, double sigma, unsigned flags,
                                 double *result,
                                 float *iwe_out, float *diwe_out, void *workspace,
                                 size_t workspace_bytes, void *stream);
int evk_cmax_linvel_variance_f32(const float *x, const float *y, const float *t_rel, const float *p,
                                 int64_t n, float p_scale, float vx, float vy, int Hm, int Wm, int Hs,
                                 int Ws,
                                 double sigma, unsigned flags, double *result, float *iwe_out,
                                 float *diwe_out, void *workspace, size_t workspace_bytes,
                                 void *stream);

/* The reference's other objective functions on the same fused event pass (row f3).  `objective` is
 * one of EVK_OBJ_*; `obj_param` is the ISOA threshold / the SOSA exponent p.  result: 12 doubles --
 * [0] f, [1..2] g, [3] sum(IWE), [4] events outside the canvas, [5] mean(G), [6..7] un-mixed gradient,
 * [8] mean(G^2), [9] sum(exp(-p G)), [10] max(G), [11] #(G > thresh)   (G = blurred IWE).
 *   EVK_OBJ_VARIANCE  variance_objective  objectives.py:202-264   (result as documented above)
 *   EVK_OBJ_SOS       sos_ / rms_objective objectives.py:266-357   f = -mean(G^2), g = -mean(2 IWE * G3(dIWE))
 *   EVK_OBJ_SOE       soe_objective       objectives.py:358-400   f = -mean(exp G), g = -mean(exp(G) G3(dIWE))
 *   EVK_OBJ_MOA       moa_objective       objectives.py:401-430   f = -max(G), no gradient
 *   EVK_OBJ_ISOA      isoa_objective      objectives.py:431-477   f = +#(G > thresh), g = -sum([G>thresh] G3(dIWE))
 *   EVK_OBJ_SOSA      sosa_objective      objectives.py:478-523   f = -sum(exp(-p G)), g = -sum(-p exp(-p G) G3(dIWE)) */
#define EVK_OBJ_VARIANCE 0
#define EVK_OBJ_SOS 1
#define EVK_OBJ_SOE 2
#define EVK_OBJ_MOA 3
#define EVK_OBJ_ISOA 4
#define EVK_OBJ_SOSA 5
int evk_cmax_linvel_objective_f64(const double *x, const double *y, const double *t, const double *p,
                                  int64_t n, double p_scale, double vx, double vy, double t_ref,
                                  int Hm, int Wm, int Hs, int Ws, double sigma, unsigned flags,
                                  int objective, double obj_param, double *result, float *iwe_out,
                                  float *diwe_out, void *workspace, size_t workspace_bytes,
                                  void *stream);
int evk_cmax_linvel_objective_f32(const float *x, const float *y, const float *t_rel, const float *p,
                                  int64_t n, float p_scale, float vx, float vy, int Hm, int Wm,
                                  int Hs, int Ws, double sigma, unsigned flags, int objective,
                                  double obj_param, double *result, float *iwe_out, float *diwe_out,
                                  void *workspace, size_t workspace_bytes, void *stream);
/* K parameter candidates in ONE pass over the events (grid_search_initial, events_cmax.py:241-311,
 * evaluates num_samples^dims = 25 points per level): every event is read once and splatted into K
 * accumulators; results: 12 doubles per candidate (layout above).  params_host: K (vx,vy) pairs in
 * HOST memory, 1 <= K <= 32. */
int evk_cmax_linvel_objective_batch_f64(const double *x, const double *y, const double *t, const double *p,
                                        int64_t n, double p_scale, const double *params_host, int n_params,
                                        double t_ref, int Hm, int Wm, int Hs, int Ws, double sigma,
                                        unsigned flags, int objective, double obj_param, double *results,
                                        void *workspace, size_t workspace_bytes, void *stream);
int evk_iwe_objective_f32(const float *iwe, const float *diwe, int Hc, int Wc, double sigma,
                          unsigned flags, int objective, double obj_param, double *result,
                          void *workspace, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Contrast maximisation for every motion model of lib/contrast_max/warps.py (README: linvel_warp,
 * xyztheta_warp, pure_rotation_warp).  The reference leaves the last two empty (warps.py:63-83); this
 * library defines them (contrast_max/warps.py).  d = t - t_ref, events transported back to t_ref:
 *   EVK_WARP_LINVEL     (vx, vy)            warps.py:51-61; dispatches to evk_cmax_linvel_objective_* (same bits)
 *   EVK_WARP_ROTATION   (cx, cy, omega)     th = -omega d:  x' = cx + cos th (x-cx) - sin th (y-cy),
 *                                                           y' = cy + sin th (x-cx) + cos th (y-cy)
 *                       dx'/dp = (1 - cos th, sin th, d (y'-cy)),  dy'/dp = (-sin th, 1 - cos th, -d (x'-cx))
 *   EVK_WARP_XYZTHETA   (vx, vy, vz, omega) x' = x - d (vx + vz x - omega y),  y' = y - d (vy + vz y + omega x)
 *                       dx'/dp = (-d, 0, -d x, d y),  dy'/dp = (0, -d, -d y, -d x)
 * Everything after the warp is get_iwe + the objective as for linvel (objectives.py:184-192, image.py:179-217,
 * objectives.py:231-264 and :266-523): f64 warp and bounds mask, f32 cast, the fixed (Hs+1)x(Ws+1) canvas.
 * The derivative images have `dims` channels (image.py:210 allocates 2; interpolate_to_derivative_img,
 * image.py:131-135, already loops over all of them), and scipy's 3-D blur of the (dims,H,W) stack mixes the
 * gradient entries by M[k][j] = sum_m w[|m|] [reflect(k+m, dims) == j] (objectives.py:253;
 * EVK_CMAX_NO_CHANNEL_MIX: identity).
 * Rotation and xyztheta run two passes over the events: pass 1 forms the IWE (the linvel event-pass kernels);
 * pass 2 is the gradient in GATHER form, g_k = -c sum_j M[k][j] sum_events p (jx_j Sx + jy_j Sy), with W the
 * blurred weight image of the objective held in shared memory and Sx, Sy the x / y differences of W over the
 * event's 2x2 footprint -- the same cost for any number of parameters.
 *   params : `dims` doubles in HOST memory; dims must be the model's (2, 3, 4)
 *   result : the 12 doubles of evk_cmax_linvel_objective_* ([1],[2] = grad[0], grad[1]); grad: `dims` doubles,
 *            device-addressable (device or pinned host memory)
 *   _f32   : fast mode, t_rel = t - t_ref already subtracted, as evk_cmax_linvel_objective_f32
 * workspace: evk_cmax_workspace_bytes(Hs,Ws) bytes, 256-byte aligned.
 * --------------------------------------------------------------------------------------------- */
#define EVK_WARP_LINVEL 0
#define EVK_WARP_ROTATION 1
#define EVK_WARP_XYZTHETA 2
int evk_cmax_model_objective_f64(int model, const double *params, int dims, const double *x,
                                 const double *y, const double *t, const double *p, int64_t n,
                                 double p_scale, double t_ref, int Hm, int Wm, int Hs, int Ws,
                                 double sigma, unsigned flags, int objective, double obj_param,
                                 double *result, double *grad, void *workspace,
                                 size_t workspace_bytes, void *stream);
int evk_cmax_model_objective_f32(int model, const double *params, int dims, const float *x,
                                 const float *y, const float *t_rel, const float *p, int64_t n,
                                 float p_scale, int Hm, int Wm, int Hs, int Ws, double sigma,
                                 unsigned flags, int objective, double obj_param, double *result,
                                 double *grad, void *workspace, size_t workspace_bytes, void *stream);
/* get_iwe's warp and mask for a model on the device (objectives.py:184-190): xw, yw, pw = x', y', p times the
 * bounds mask, jx, jy = [dims][n] Jacobians times the mask (may both be NULL), all cast to f32 as
 * events_to_image_drv does (image.py:179-183) -- the inputs of evk_image_drv_f32.  Rotation / xyztheta only;
 * EVK_CMAX_ABS_POLARITY: p <- |p|. */
int evk_cmax_model_warp_f64(int model, const double *params, int dims, const double *x, const double *y,
                            const double *t, const double *p, int64_t n, double t_ref, int Hm, int Wm,
                            unsigned flags, float *xw, float *yw, float *pw, float *jx, float *jy,
                            void *stream);
/* The precomputed-image form with K <= 8 derivative channels (diwe: [K][Hc][Wc]) and K gradient entries
 * (grad, device-addressable); result as above.  For any warp, including user-defined ones. */
int evk_iwe_objective_k_f32(const float *iwe, const float *diwe, int K, int Hc, int Wc, double sigma,
                            unsigned flags, int objective, double obj_param, double *result,
                            double *grad, void *workspace, size_t workspace_bytes, void *stream);

/* scipy.ndimage.gaussian_filter(img, sigma) for a 2-D f32 image (truncate=4, mode='reflect', f64 line
 * accumulation, f32 store after each axis) -- the blur every objective applies (objectives.py:233 ...).
 * tmp: H*W floats of scratch; out may not alias img. */
int evk_gaussian_blur_f32(const float *img, int H, int W, double sigma, float *out, float *tmp, void *stream);

/* The objective (and gradient) of a PRECOMPUTED image of warped events, i.e. the iwe= / d_iwe=
 * form of evaluate_function / evaluate_gradient (objectives.py:211-264 with iwe given; used by
 * grid_cmax, events_cmax.py:68-70).  iwe: [Hc][Wc] f32, diwe: [2][Hc][Wc] f32 or NULL. */
int evk_variance_objective_f32(const float *iwe, const float *diwe, int Hc, int Wc, double sigma,
                               unsigned flags, double *result, void *workspace,
                               size_t workspace_bytes, void *stream);

/* Cross-GPU barrier on a stream, for the fused peer kernels.  peer_slots[r] = rank r's array of `world` 32-bit slots, mapped
 * on every rank (symmetric memory), zero before the first barrier; `epoch` = 1, 2, 3, ... (the caller counts).  Rank `rank`
 * stores `epoch` into slot [rank] of every rank and waits until all its own slots have reached it. */
int evk_peer_barrier(unsigned *const *peer_slots, int world, int rank, unsigned epoch, void *stream);

/* Sharded contrast maximisation, one process per GPU (SURVEY 8e): the all-reduce of the partial images is FUSED into the
 * objective kernel over NVLink peer memory -- no NCCL call, no host synchronisation between the two halves.
 *   evk_cmax_linvel_partial_*  event pass of THIS rank's shard; leaves its planar partial images images_out[3][Hs+1][Ws+1]
 *                              (IWE, dIWE/dvx, dIWE/dvy; objectives.py:184-192) and its out-of-canvas event count.
 *                              images_out / oob_out live in memory every rank has mapped (symmetric memory).
 *   (a cross-GPU barrier)
 *   evk_cmax_peer_tail_f32     every rank reads ALL ranks' partial images through peer pointers, sums them in rank order
 *                              while it gathers its tiles, blurs, reduces and writes f, g (objectives.py:231-264) --
 *                              bit-identical on all ranks.  result[4] = total out-of-canvas events. */
int evk_cmax_linvel_partial_f64(const double *x, const double *y, const double *t, const double *p, int64_t n,
                                double p_scale, double vx, double vy, double t_ref, int Hm, int Wm, int Hs, int Ws,
                                unsigned flags, float *images_out, unsigned long long *oob_out, void *workspace,
                                size_t workspace_bytes, void *stream);
int evk_cmax_linvel_partial_f32(const float *x, const float *y, const float *t_rel, const float *p, int64_t n,
                                float p_scale, float vx, float vy, int Hm, int Wm, int Hs, int Ws, unsigned flags,
                                float *images_out, unsigned long long *oob_out, void *workspace,
                                size_t workspace_bytes, void *stream);
int evk_cmax_peer_tail_f32(const float *const *peer_images, const unsigned long long *const *peer_oob, int world,
                           int Hc, int Wc, double sigma, unsigned flags, double *result, void *workspace,
                           size_t workspace_bytes, void *stream);

/* Objective only (f) for a dense-flow warp: warp_events_flow_torch + bilinear IWE
 * (lib/visualization/draw_flow.py:18-21) + the variance objective.  flow: [2][Hs][Ws]. */
int evk_cmax_flow_variance_f32(const float *x, const float *y, const float *t, const float *p,
                               int64_t n, const float *flow, float t0, int Hs, int Ws, double sigma,
                               unsigned flags, double *result, float *iwe_out, void *workspace,
                               size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------
 * RobustNorm (row f4): clamp a tensor between two of its order statistics and rescale it.  Replaces
 * RobustNorm.__call__ / .percentile, lib/data_loaders/data_augmentation.py:82-130 (two kthvalue sorts),
 * the step after the voxel grid in the loaders (base_dataset.py:471).
 *   k_low / k_top: 1-based ranks, k = 1 + round(.01 q (n-1)) computed by the caller (:100)
 *   out = x if both statistics are 0, else (clamp(x, t_min, t_max) - t_min) / (t_max + 1e-6)
 *   t_min_max: optional 2 floats on the device receiving the two statistics.
 * --------------------------------------------------------------------------------------------- */
size_t evk_robust_norm_workspace_bytes(void);
int evk_robust_norm_f32(const float *x, int64_t n, int64_t k_low, int64_t k_top, float *out,
                        float *t_min_max, void *workspace, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Host-buffer pipeline: the same voxel build for events living in HOST memory (pinned memory
 * gives full PCIe bandwidth).  Events are streamed in chunks through a double-buffered device
 * staging area so the H2D copy of chunk k+1 overlaps the scatter of chunk k; the finished grid
 * is copied back to `out_host`.  Synchronous (returns when out_host is complete).
 * *oob_host receives the out-of-range event count.
 * --------------------------------------------------------------------------------------------- */
typedef struct evk_pipeline evk_pipeline_t;
int evk_pipeline_create(evk_pipeline_t **pipe, int64_t chunk_events);
void evk_pipeline_destroy(evk_pipeline_t *pipe);
int evk_voxel_host_f32(evk_pipeline_t *pipe, const float *x, const float *y, const float *t,
                       const float *p, int64_t n, float t0, float dt, int B, int H, int W,
                       unsigned flags, float *out_host, unsigned long long *oob_host);
/* the same for host arrays in the storage layout (see evk_voxel_packed_f32): 13 B/event over PCIe */
int evk_voxel_host_packed_f32(evk_pipeline_t *pipe, const int16_t *x, const int16_t *y, const double *t,
                              const uint8_t *p, int64_t n, double t_first, double t_last, int B, int H,
                              int W, unsigned flags, float *out_host, unsigned long long *oob_host);

/* ---------------------------------------------------------------------------------------------
 * 64-bit content hash of a HOST buffer (every byte enters; multi-threaded above 2 MiB, result independent
 * of the thread count).  The identity of an event set in the host-side cache of uploaded events: the
 * reference's objective is a pure function of the arrays it is handed at every call
 * (lib/contrast_max/objectives.py:211-236), so a cached device copy may only be reused when the host
 * arrays are byte-identical to the ones that were uploaded.  No device work.
 * --------------------------------------------------------------------------------------------- */
uint64_t evk_host_hash64(const void *data, size_t nbytes, uint64_t seed);
/* k buffers in one call (one pool of threads for all of them); out[a] = hash of buffer a under a seed derived from
 * `seed` and a, so equal contents at different positions hash differently. */
void evk_host_hash64_multi(const void *const *ptrs, const size_t *nbytes, int k, uint64_t seed, uint64_t *out);

/* The staging copy of the host pipeline, for callers that fill their own pinned buffers: k host arrays of `nbytes`
 * each, dst[a] <- src[a], in 1 MiB blocks on 8 threads (EVK_HOST_COPY_THREADS) of the library's persistent worker
 * pool (half of the CPUs the process may run on, at most 32; EVK_HOST_THREADS) with non-temporal stores (the destination
 * is read next by the DMA engine, not by the CPU; EVK_HOST_COPY_STREAM=0 -> memcpy).  evk_voxel_host_f32 uses it for ordinary pageable sources -- what the
 * reference's loaders produce (lib/data_loaders/base_dataset.py:446-453).  No device work. */
void evk_host_copy(void *const *dst, const void *const *src, int k, size_t nbytes);
/* Upload k host arrays (nbytes[a] each) into device buffers the caller allocated -- the event set of a
 * contrast-maximisation run (the reference hands numpy arrays to every objective call, lib/contrast_max/objectives.py:211),
 * numpy inputs of the image functions.  Pageable sources go through the pipeline's pinned bounce slots, filled by the
 * worker pool while the previous pieces are on the wire; pinned sources are copied directly.  Synchronous: the data is on
 * the device when it returns.  A pipeline serves one call at a time. */
int evk_host_upload(evk_pipeline_t *pipe, void *const *dst_dev, const void *const *src_host, int k, const size_t *nbytes);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* EVK_H_ */
