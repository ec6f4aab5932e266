/* rpsf_b200.h — C ABI of the B200-native regularizepsf correction path.
 *
 * The reference (punch-mission/regularizepsf) is pure Python and has no FFI; its boundary for
 * this path is the public Python API.  Each entry point below names the reference interface it
 * replaces (paths relative to the reference repository root).  The Python mirror of that API
 * (regularizepsf_b200/transform.py, psf.py) is the only in-tree caller and binds these symbols
 * with ctypes; INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions: every function returns 0 on success or a negative RPSF_E_* code;
 * rpsf_last_error() gives the message for the calling thread.  No C++ exceptions cross the
 * ABI.  Device pointers are caller-owned; `stream` is a cudaStream_t passed as void* (NULL =
 * legacy default stream).  Stream-taking calls enqueue work and return without
 * synchronising.  Calls that touch a transform's device state (its laid-out kernel, its plans'
 * workspaces and scratch) are ordered by one event per transform: a call on a stream other than
 * the last one's waits for the last one, so it sees the kernel laid out before it was issued and
 * never shares a plan's workspace with a call still in flight.  Calls sharing a plan therefore
 * do not overlap; use one plan per concurrent stream or thread to run them side by side.
 */
#ifndef RPSF_B200_H
#define RPSF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RPSF_ABI_VERSION 3

/* status codes */
#define RPSF_OK 0
#define RPSF_E_INVALID_ARGUMENT (-1)
#define RPSF_E_INVALID_COORDINATE (-2) /* maps to regularizepsf.exceptions.InvalidCoordinateError */
#define RPSF_E_INCORRECT_SHAPE (-3)    /* maps to regularizepsf.exceptions.IncorrectShapeError   */
#define RPSF_E_UNSUPPORTED (-4)        /* patch size / dtype / pad mode without a device path    */
#define RPSF_E_CUDA (-5)
#define RPSF_E_NO_KERNEL (-6)          /* apply before rpsf_transform_set_kernel                 */

/* element types */
#define RPSF_F32 0
#define RPSF_F64 1
#define RPSF_U8 2
#define RPSF_I16 3
#define RPSF_U16 4
#define RPSF_I32 5
#define RPSF_I64 6
#define RPSF_U32 7

/* np.pad modes with an on-device index map (transform.py:119-123, `pad_mode`) */
#define RPSF_PAD_SYMMETRIC 0
#define RPSF_PAD_REFLECT 1
#define RPSF_PAD_EDGE 2
#define RPSF_PAD_WRAP 3
#define RPSF_PAD_CONSTANT 4
/* every other np.pad mode (mean, median, maximum, minimum, linear_ramp, ...): the caller materialises the padded frame
 * (np.pad of 2P per side, as transform.py:119-123 does) and passes a pointer to the UNPADDED pixel (0, 0) inside it;
 * rows / columns in [-2P, dim + 2P) must then be addressable through the pitch.  Device-pointer entry points only. */
#define RPSF_PAD_MATERIALIZED 5

typedef struct rpsf_transform rpsf_transform;
typedef struct rpsf_plan rpsf_plan;

/* CUDA graphs.  A stream capture may contain, once their plans exist and each has run once outside the capture:
 * rpsf_apply (forward and adjoint plans), rpsf_apply_source, rpsf_apply_masked, rpsf_kernel_gradient(_masked), rpsf_transform_set_kernel,
 * rpsf_construct_kernel(_dev), rpsf_construct_kernel_backward(_dev), rpsf_psf_fft2 and rpsf_psf_fft2_adjoint (native
 * patch sizes), rpsf_apply_stack, rpsf_stack_set_kernel and rpsf_construct_kernels(_dev).  These neither cudaMalloc nor synchronise then; their scratch is cudaMallocAsync on the stream, which
 * the capture turns into allocation nodes.  On a capturing stream a call that touches a transform's device state makes
 * the transform's order event an external dependency of the graph (cudaEventWaitExternal at its start,
 * cudaEventRecordExternal at its end), so each replay is ordered after the calls issued before its launch and before
 * those issued after it; from then on every eager call on that transform waits for the event.  What would allocate
 * or synchronise (a plan's first call, the first saturation branch, plan creation, the host path, upload / free, IPC,
 * the builder) returns RPSF_E_UNSUPPORTED while a capture is open, before any CUDA call that would invalidate it.
 * Entry points without a stream argument see a capture once a call of this library has run on the capturing stream:
 * the library remembers such streams, on every thread, until it finds their capture ended (at a stream-less call, or
 * at an eager call on the same stream).  While any of them captures, plan creation, upload / free, IPC and the host
 * path are refused on every thread, which is stricter than a relaxed capture mode needs.  A stream the library has
 * seen capturing must not be destroyed before its capture has ended and a later call of the library has run.
 * The caller keeps the transforms and plans a graph uses alive as long as the graph. */

int rpsf_abi_version(void);
const char* rpsf_last_error(void);
/* 1: patch size P runs natively (powers of two 16..512); 2: it runs embedded in the next power of two M >= 2 P - 1
 * (2 <= P <= 256: the transfer kernel is re-sampled on the M-grid so that the M-point circular convolution of the
 * zero-padded windowed patch reproduces the reference's P-point one, transform.py:151-165 — same results, (M / P)^2
 * the work, the generic gather and colour-phase overlap-add kernels); 0: no device path */
int rpsf_patch_size_supported(int patch_size);

/* ---- transform: replaces ArrayPSFTransform.__init__ (transform.py:28-37) -------------------
 * coords: n x 2 host int32 (row, col) upper-left patch corners in unpadded frame coordinates,
 * in IndexedCube order (util.py:56-82).  compute_dtype: RPSF_F32 or RPSF_F64 (validation mode). */
int rpsf_transform_create(rpsf_transform** out, const int32_t* coords, int n_patches, int patch_size,
                          int compute_dtype, int device);
/* The same for one rank of a patch-row slab split (SURVEY.md section 8e: "holds only those patches' kernels"): `keep`
 * (n_patches bytes, may be NULL = all) marks the patches whose transfer kernel this device will hold.  The whole
 * coordinate list is still given, so colour classes — and with them the per-pixel summation order — are those of the
 * complete transform and sharded results stay bit-identical.  rpsf_transform_set_kernel then takes the kept patches
 * only, in list order; a plan whose row band needs a patch that was not kept fails with RPSF_E_INVALID_ARGUMENT. */
int rpsf_transform_create_subset(rpsf_transform** out, const int32_t* coords, int n_patches, int patch_size,
                                 int compute_dtype, int device, const uint8_t* keep);
int rpsf_transform_destroy(rpsf_transform* t);

/* Load the transfer kernel: `kernel_full` is the (N,P,P) complex cube in the reference layout
 * (IndexedCube.values of ArrayPSFTransform._transfer_kernel, transform.py:37,82; full unshifted
 * spectrum) on the device, complex64 (RPSF_F32) or complex128 (RPSF_F64).  Builds the private
 * Hermitian-half, 1/P^2-scaled, register-ordered copy that rpsf_apply reads. */
int rpsf_transform_set_kernel(rpsf_transform* t, const void* kernel_full, int kernel_dtype, void* stream);

/* number of colour classes of the overlap graph (4 for calculate_covering inputs, util.py:10-53) */
int rpsf_transform_num_colours(const rpsf_transform* t);

/* A fence in the transform's stream order, with no launches: `stream` waits for the transform's previous calls (eager
 * calls and graph replays) and the calls issued after this one wait for what `stream` has queued up to here.  For a
 * caller that writes, on `stream`, a buffer that captured calls of the transform read. */
int rpsf_transform_order(rpsf_transform* t, void* stream);

/* ---- construct: replaces the arithmetic of ArrayPSFTransform.construct (transform.py:78-82) -
 * source_fft / target_fft / kernel_out: `count` complex elements on the device, all complex64
 * (dtype RPSF_F32) or all complex128 (RPSF_F64).  The coordinate check (transform.py:74-76)
 * stays on the host. */
int rpsf_construct_kernel(const void* source_fft, const void* target_fft, void* kernel_out, int64_t count,
                          int dtype, double alpha, double epsilon, int device, void* stream);
/* The same with alpha and epsilon read on the device from alpha_epsilon (2 doubles, [alpha, epsilon]), so that a caller
 * holding them in device memory need not synchronise; bit-identical to rpsf_construct_kernel given the same values. */
int rpsf_construct_kernel_dev(const void* source_fft, const void* target_fft, void* kernel_out, int64_t count,
                              int dtype, const double* alpha_epsilon, int device, void* stream);

/* Vector-Jacobian product of rpsf_construct_kernel (transform.py:78-82), for a gradient that reaches the PSFs, alpha and
 * epsilon.  kernel_grad is G, the gradient of the loss with respect to K in PyTorch's convention (dL/dRe + i dL/dIm);
 * with a = |S|, b = |T|, c = epsilon b, D = a^(alpha+1) + c^(alpha+1), f = a^(alpha-1) / D, w = Re(G S conj(T)):
 *   source_grad = f conj(G) T + w a^(alpha-3) ((alpha-1) c^(alpha+1) - 2 a^(alpha+1)) / D^2 S
 *   target_grad = f G S - w (alpha+1) epsilon^(alpha+1) a^(alpha-1) b^(alpha-1) / D^2 T
 *   alpha_epsilon_grad[0] = sum w a^(alpha-1) c^(alpha+1) ln(a/c) / D^2
 *   alpha_epsilon_grad[1] = -sum w (alpha+1) epsilon^alpha a^(alpha-1) b^(alpha+1) / D^2
 * A bin with G = 0 contributes exact zeros to all four outputs; where K is finite the 0 * inf products of these forms (at
 * a = 0, b = 0 or c = 0) take their limit 0; where K is not finite and G != 0 the bin's cube outputs are NaN and so are
 * both sums.  The four cubes are `count` complex elements on the device, all complex64 (RPSF_F32) or all complex128
 * (RPSF_F64); source_grad and target_grad may be NULL (not computed).  alpha_epsilon_grad (device, 2 doubles, may be
 * NULL) is accumulated in double for both dtypes over a fixed partition in a fixed order: bit-stable from run to run.
 * Stream-ordered (scratch is cudaMallocAsync / cudaFreeAsync on `stream`), no host synchronisation. */
int rpsf_construct_kernel_backward(const void* source_fft, const void* target_fft, const void* kernel_grad,
                                   int64_t count, int dtype, double alpha, double epsilon, void* source_grad,
                                   void* target_grad, double* alpha_epsilon_grad, int device, void* stream);
/* The same with alpha and epsilon read on the device from alpha_epsilon (2 doubles; not the output alpha_epsilon_grad);
 * bit-identical to rpsf_construct_kernel_backward given the same values. */
int rpsf_construct_kernel_backward_dev(const void* source_fft, const void* target_fft, const void* kernel_grad,
                                       int64_t count, int dtype, const double* alpha_epsilon, void* source_grad,
                                       void* target_grad, double* alpha_epsilon_grad, int device, void* stream);

/* ---- PSF cube FFT: replaces scipy.fft.fft2 in ArrayPSF.__init__ (psf.py:216-219) -----------
 * values: (n, P, P) real on the device; out: (n, P, P) complex, full spectrum, same precision. */
int rpsf_psf_fft2(const void* values, void* out, int64_t n_patches, int patch_size, int dtype, int device,
                  void* stream);
/* Vector-Jacobian product of rpsf_psf_fft2 (psf.py:216-219): values_grad = Re(fft2(conj(spectrum_grad))) = P^2
 * Re(ifft2(spectrum_grad)), the gradient with respect to the real values of a loss whose gradient with respect to the
 * spectrum is spectrum_grad (PyTorch's convention).  spectrum_grad: (n, P, P) complex on the device; values_grad: (n, P,
 * P) real, same precision.  Patch sizes 16, 32, ..., 512 only; the others are RPSF_E_UNSUPPORTED.  Stream-ordered
 * (an (n, P, P) complex scratch cube is cudaMallocAsync / cudaFreeAsync on `stream`). */
int rpsf_psf_fft2_adjoint(const void* spectrum_grad, void* values_grad, int64_t n_patches, int patch_size, int dtype,
                          int device, void* stream);

/* ---- builder: per-cell averaging of star cutouts (SURVEY.md section 8f-4) -------------------
 * Replaces regularizepsf/builder.py:45-125 (_average_patches and its mean / percentile helpers):
 * every cutout is divided by its centre pixel [P/2][P/2] (builder.py:63,90); cell c stacks the
 * cutouts cell_items[cell_offsets[c] .. cell_offsets[c+1]) in that order (the reference's dict
 * insertion order; the matching of builder.py:45-51 stays on the host) and reduces the stack per
 * pixel: NaN-aware mean (np.nansum / count of finite values), np.nanmedian, or np.nanpercentile
 * (linear).  NaN results (empty or all-NaN stacks, 0/0) become 0 (builder.py:118-122).  float64,
 * bit-identical to numpy.  cutouts: device (n_cutouts, P, P) float64; out: device (n_cells, P, P)
 * float64; the index arrays are HOST pointers.  percentile in [0, 100] (RPSF_AVG_PERCENTILE only;
 * 50 is computed as the median, as builder.py:79-82 does).  Stream-ordered: the index arrays are
 * copied before the call returns, temporaries are cudaMallocAsync / cudaFreeAsync on `stream`. */
#define RPSF_AVG_MEAN 0
#define RPSF_AVG_MEDIAN 1
#define RPSF_AVG_PERCENTILE 2
int rpsf_average_patches(const double* cutouts, int64_t n_cutouts, int patch_size, const int64_t* cell_offsets,
                         const int32_t* cell_items, int64_t n_cells, int method, double percentile, double* out,
                         int device, void* stream);

/* The per-patch stages that follow the averaging in ArrayPSFBuilder.build (builder.py:236-258), one CTA per patch,
 * float64, device pointers, stream-ordered (scratch is cudaMallocAsync / cudaFreeAsync on `stream`):
 *   rpsf_plane_background  image_processing.py:13-46 (calculate_background): the least-squares plane
 *                          c0 * col + c1 * row + c2 through the ring of pixels just inside the patch border that are
 *                          fainter than the centre; NaN where the patch is exactly 0.  out: (n, P, P).
 *   rpsf_isolate_cores     builder.py:239-258 in place on (n, P, P): subtract that plane, zeros -> NaN, drop the pixels
 *                          below 0.5 % of the centre (eroded, outside counted as faint), non-finite -> 0, keep the
 *                          4-connected island of the centre pixel dilated by one pixel, divide by the sum.
 * Every mask is an integer decision and follows the reference; the plane is solved from the 3 x 3 normal equations
 * (minimum-norm when the ring is degenerate, like LAPACK gelsd) and the sum is a tree, so values agree with the
 * reference to ~1e-13 of the patch maximum rather than bit for bit (tests/test_gpu_builder.py states 1e-11). */
int rpsf_plane_background(const double* patches, int64_t n_patches, int patch_size, double* out, int device, void* stream);
/* The per-star body of _find_patches (image_processing.py:78-121), one CTA per detected star: the width x width window
 * of the frame at the rounded corner through np.pad(mode="reflect"), scipy.ndimage.shift(order=3, mode="mirror") by
 * (-corner + round(corner) - 0.5) (cubic B-spline prefilter + 4 x 4 interpolation, rounded to the frame's dtype as
 * scipy does), minus its plane background (NaN where the shifted patch is 0); accepted[i] = every pixel below
 * saturation_threshold (a NaN fails) and star_minimum < centre < star_maximum.  frame: device (H, W) float32 / float64,
 * contiguous; corners: HOST (n, 2) float64 = the reference's dict keys (row - width/2, col - width/2); out: device
 * (n, width, width) float64; accepted: device n bytes.  Values agree with scipy to ~1e-15 of the patch maximum (float64
 * frames).  The pixel-mask patch (:102-106, :119) is left to the caller: the reference casts its spline-shifted values
 * to bool by truncation, which only scipy's own instruction order reproduces.  Synchronises `stream` before returning
 * (the corner list is read from pageable memory). */
int rpsf_star_cutouts(const void* frame, int frame_dtype, int height, int width, const double* corners, int64_t n_stars,
                      int cutout_size, double saturation_threshold, double star_minimum, double star_maximum, double* out,
                      unsigned char* accepted, int device, void* stream);
int rpsf_isolate_cores(double* patches, int64_t n_patches, int patch_size, int device, void* stream);

/* ---- plan: geometry of apply() for one frame shape ------------------------------------------
 * Replaces the padding / slicing bookkeeping of ArrayPSFTransform.apply (transform.py:119-123,
 * 141-149, 167-177).  [row_begin,row_end) is the band of output rows this plan owns (0,H for
 * the whole frame; a sub-range for patch-row slabs across GPUs).  max_batch frames share the
 * workspace. */
int rpsf_plan_create(rpsf_plan** out, rpsf_transform* t, int height, int width, int pad_mode, int row_begin,
                     int row_end, int max_batch);
/* A plan whose rpsf_apply computes the transpose of the plan rpsf_plan_create(t, H, W, pad_mode, 0, H, .) would run
 * (no saturation): input = `batch` (H, W) frames of output gradients, output = (H, W) frames of input gradients.
 * It runs the three default kernels on the bounding box of the patch footprints (zero-bordered copy of the input,
 * conj of the transfer kernel, built at the first adjoint plan of `t`) and folds the box onto the frame along the
 * np.pad index map (pad_mode 0..4; RPSF_PAD_MATERIALIZED is RPSF_E_UNSUPPORTED).  rpsf_apply takes whole frames
 * (img_row0 = out_row0 = 0, img_rows = H); rpsf_apply_stages and rpsf_apply_host, a finite saturation threshold and
 * output mirrors are RPSF_E_UNSUPPORTED on it. */
int rpsf_plan_create_adjoint(rpsf_plan** out, rpsf_transform* t, int height, int width, int pad_mode, int max_batch);
/* Gradient of <apply(image), grad> with respect to the transfer kernel, summed over `batch` frames (no saturation):
 * kernel_grad[n] = sum_b conj(X_n) G_n / P^2 with X_n = FFT2(w * patch n of the padded image) and G_n = FFT2(w * patch n of
 * the zero-extended grad), in PyTorch's convention (dL/dRe + i dL/dIm).  `kernel_grad` is a device (n, P, P) complex cube
 * of the compute dtype in the layout rpsf_transform_set_kernel reads; patches that do not touch the frame get 0.
 * `adjoint_plan` comes from rpsf_plan_create_adjoint(t, H, W, pad_mode, .), `forward_plan` from rpsf_plan_create(t, H, W,
 * pad_mode, 0, H, .) with an infinite saturation threshold; both workspaces are reused, nothing is allocated.  Embedded
 * patch sizes, sharded transforms, a finite saturation threshold, the materialised pad and a partial row band are
 * RPSF_E_UNSUPPORTED; plans of different transforms, shapes or pad modes and a batch above either plan's capacity are
 * RPSF_E_INVALID_ARGUMENT.  With rpsf_plan_enable_timing on the forward plan, rpsf_plan_read_timing of that plan
 * reports K1 of the image, the copy of grad plus K1 of the box, and the zeroing plus the gradient kernel. */
int rpsf_kernel_gradient(rpsf_plan* adjoint_plan, rpsf_plan* forward_plan, const void* image, int64_t img_pitch,
                         int64_t img_frame_stride, const void* grad, int64_t grad_pitch, int64_t grad_frame_stride, int batch,
                         void* kernel_grad, void* stream);
/* rpsf_kernel_gradient of apply with a caller-given bad-pixel mask (rpsf_apply_masked): X is K1 of the padded frame
 * filled under the mask (the forward plan's rpsf_plan_set_saturation gives the neighbourhood width; its threshold must be
 * infinite), G that of (1 - M) grad.  mask: uint8, nonzero = masked, pixel (y, x) of frame b at mask +
 * b*mask_frame_stride + y*mask_pitch + x; mask_frame_stride 0 shares one mask across the frames.  The first call of a
 * forward plan allocates its fill scratch (as the saturation branch does) and cannot be captured. */
int rpsf_kernel_gradient_masked(rpsf_plan* adjoint_plan, rpsf_plan* forward_plan, const void* image, int64_t img_pitch,
                                int64_t img_frame_stride, const void* grad, int64_t grad_pitch, int64_t grad_frame_stride,
                                int batch, void* kernel_grad, const void* mask, int64_t mask_pitch,
                                int64_t mask_frame_stride, void* stream);
int rpsf_plan_destroy(rpsf_plan* p);
/* info[0]=active patches, [1]=colours, [2]=workspace bytes (patch spectra and row bands, see rpsf_plan_workspace),
 * [3]=first frame row read,
 * [4]=one past the last frame row read, [5]=1 if colour 0 tiles the band exactly,
 * [6]=overlap-add kernel: 2 = streaming chains (registers only), 1 = single-launch row-pair gather
 *      through a shared-memory plane, 0 = one launch per colour class,
 * [7]=teams per CTA of the row-pair gather,
 * [8]=chunks per chain of the streaming chains (from a cost model of max_batch and the SM count), 0 when [6] != 2 */
int rpsf_plan_info(const rpsf_plan* p, int64_t info[9]);
/* overlap-add kernel choice: 0 = automatic (streaming chains when every owned row pair is a chain of
 * half-overlapping patch columns — any calculate_covering grid —, else the row-pair gather when patch
 * corner rows share one parity, else colour phases); 1 = force the colour-phase kernel, 2 = force the
 * row-pair gather (test hooks) */
int rpsf_plan_set_overlap_mode(rpsf_plan* p, int mode);
/* gather + row-FFT kernel choice: 0 = automatic (the persistent bulk-copy kernel), 1 = force the
 * one-row-pair-per-team kernel with direct loads (test hook; same arithmetic up to rounding) */
int rpsf_plan_set_gather_mode(rpsf_plan* p, int mode);

/* column pass: info[0] = 0 (the column pass from the row bands into the spectrum workspace, the only one there is) and
 * info[1] = 0 (bytes per frame of a column-pass workspace of its own: none).  Kept so that callers that report
 * the column pass keep working. */
int rpsf_plan_column_info(const rpsf_plan* p, int64_t info[2]);

/* ---- saturation arguments of apply (transform.py:88-90,125-138,171-172) ---------------------
 * threshold = +inf (the default) disables the branch.  Otherwise every apply on this plan pads
 * the frame 2P per side, masks padded > threshold, dilates the mask `dilation` times with the
 * 3x3 cross (dilation < 1: until stable, as scipy.ndimage.binary_dilation), replaces masked
 * pixels IN RASTER ORDER by the nanmean of padded[i-w//2:i+w//2, j-w//2:j+w//2], corrects the
 * filled frame and writes the raw pixel back into every masked output pixel.  Needs the whole
 * frame resident (img_row0 = 0, img_rows = height). */
int rpsf_plan_set_saturation(rpsf_plan* p, double threshold, int dilation, int neighborhood_width);

/* ---- apply, device-resident: replaces ArrayPSFTransform.apply (transform.py:85-177) ---------
 * image: `batch` frames of compute-dtype pixels; row `img_row0 + i` of frame b is at
 *        image + b*img_frame_stride + i*img_pitch (elements); rows [info[3], info[4]) must be
 *        resident.  out: rows [row_begin,row_end) are written; row r of frame b is at
 *        out + b*out_frame_stride + (r - out_row0)*out_pitch. */
int rpsf_apply(rpsf_plan* p, const void* image, int64_t img_pitch, int64_t img_frame_stride, int img_row0,
               int img_rows, void* out, int64_t out_pitch, int64_t out_frame_stride, int out_row0, int batch,
               void* stream);

/* rpsf_apply with the saturation mask decided on `src`: the same `batch` frames before their conversion to the
 * compute dtype, of src_dtype, row `img_row0 + i` of frame b at src + b*src_frame_stride + i*src_pitch (elements).
 * The reference compares float64 values with the threshold; a float64 or 32/64-bit integer pixel just above it can
 * round to it in float32.  Everything but the initial mask (the fill, the correction, the restored pixels) uses
 * `image`.  Without saturation `src` is not read. */
int rpsf_apply_source(rpsf_plan* p, const void* image, int64_t img_pitch, int64_t img_frame_stride, int img_row0,
                      int img_rows, void* out, int64_t out_pitch, int64_t out_frame_stride, int out_row0, int batch,
                      const void* src, int src_dtype, int64_t src_pitch, int64_t src_frame_stride, void* stream);

/* rpsf_apply with a caller-given bad-pixel mask M (uint8, nonzero = masked, laid out as for
 * rpsf_kernel_gradient_masked; mask_frame_stride 0 shares one mask across the frames).  On a forward plan: the pixels of
 * pad(M) (padded with the plan's index map; the margin of constant mode is unmasked), ORed into the dilated saturation
 * mask (only pad(M) with an infinite threshold), are filled in raster order with the nanmean of their neighbourhood as
 * saturated pixels are, and get their raw values back after the correction.  `src` (may be null) is rpsf_apply_source's.
 * On an adjoint plan (src null, infinite threshold, rpsf_plan_set_saturation giving the neighbourhood width): the
 * transpose of that map, which with an infinite threshold is linear in the image, with the fill's contributors decided
 * by the mask alone (finite-input semantics; a structural NaN, a masked pixel whose window holds no contributor,
 * passes nothing back).  Needs a pad mode with an index map and whole frames resident.  The first call of a plan
 * allocates its padded-size scratch and cannot be captured in a CUDA graph; later ones can. */
int rpsf_apply_masked(rpsf_plan* p, const void* image, int64_t img_pitch, int64_t img_frame_stride, int img_row0,
                      int img_rows, void* out, int64_t out_pitch, int64_t out_frame_stride, int out_row0, int batch,
                      const void* src, int src_dtype, int64_t src_pitch, int64_t src_frame_stride, const void* mask,
                      int64_t mask_pitch, int64_t mask_frame_stride, void* stream);

/* ---- apply, host buffers (the call a reference user makes): H2D + convert + apply + D2H ------
 * image: `batch` contiguous (H, W) frames of image_dtype on the host (pinned or pageable);
 * out: `batch` contiguous (row_end-row_begin, W) frames of out_dtype (RPSF_F32 / RPSF_F64).
 * Synchronous on return. */
int rpsf_apply_host(rpsf_plan* p, const void* image, int image_dtype, void* out, int out_dtype, int batch);

/* ---- transform stacks: M transfer kernels on one set of patch corners and one patch size ------
 * For a sweep of (alpha, epsilon): one call applies every kernel to the same frames, and the work that does not depend
 * on the kernel (the saturation / mask fill, the row pass) runs once per frame instead of once per kernel. */
typedef struct rpsf_stack rpsf_stack;

/* rpsf_construct_kernel for n_kernels (alpha, epsilon) pairs in one pass over S and T: kernel m, bit-identical to
 * rpsf_construct_kernel(..., alpha_epsilon[2m], alpha_epsilon[2m + 1], ...), is written to kernel_out + m * count
 * (complex elements).  alpha_epsilon: HOST array of 2 * n_kernels doubles.  Launches only (one per 64 kernels). */
int rpsf_construct_kernels(const void* source_fft, const void* target_fft, void* kernel_out, int64_t count, int dtype,
                           const double* alpha_epsilon, int n_kernels, int device, void* stream);
/* The same with alpha_epsilon in device memory (2 * n_kernels doubles); bit-identical to rpsf_construct_kernel_dev. */
int rpsf_construct_kernels_dev(const void* source_fft, const void* target_fft, void* kernel_out, int64_t count,
                               int dtype, const double* alpha_epsilon, int n_kernels, int device, void* stream);

/* A stack of n_kernels >= 1 transfer kernels on the coordinates of rpsf_transform_create (same arguments, same errors).
 * Each kernel is loaded with rpsf_stack_set_kernel(index, ...), which takes what rpsf_transform_set_kernel takes.
 * rpsf_stack_destroy frees the stack; destroy its plans first. */
int rpsf_stack_create(rpsf_stack** out, const int32_t* coords, int n_patches, int patch_size, int compute_dtype,
                      int device, int n_kernels);
int rpsf_stack_set_kernel(rpsf_stack* stack, int index, const void* kernel_full, int kernel_dtype, void* stream);
int rpsf_stack_destroy(rpsf_stack* stack);
/* A whole-frame plan (rows [0, height)) of a stack for up to max_batch frames per call; n_kernels * max_batch <= 65535.
 * Its workspace holds the patch spectra of n_kernels * max_batch frames and the row bands of max_batch frames (the
 * spectra are 75.8 MB per frame and kernel at 2048^2 / 256 px, float32).  It runs through rpsf_apply_stack only (the
 * other apply entry points return RPSF_E_INVALID_ARGUMENT); free it with rpsf_plan_destroy, and set its saturation
 * with rpsf_plan_set_saturation.  RPSF_PAD_MATERIALIZED is RPSF_E_UNSUPPORTED. */
int rpsf_plan_create_stack(rpsf_plan** out, rpsf_stack* stack, int height, int width, int pad_mode, int max_batch);
/* Every kernel of the stack applied to `batch` whole frames: output frame m * batch + b (at out + (m * batch + b) *
 * out_frame_stride) is bit-identical to rpsf_apply_masked (mask non-null), rpsf_apply_source (src non-null) or rpsf_apply
 * with kernel m alone on frame b.  n_kernels must be the stack's.  The saturation / mask fill and the row pass run once
 * per frame; the column pass runs once per kernel from the shared row spectra; one overlap-add covers every output
 * frame.  The first call of a plan allocates its workspace (and, with saturation or a mask, its fill scratch) and
 * cannot be captured in a CUDA graph; later ones can. */
/* Column pass of a stack plan: mode 0 (the default) runs k2_stack, which transforms each tile of the row spectra once
 * per frame and then multiplies and inverse-transforms it per kernel, for stacks of two kernels or more where it exists (native patch sizes whose
 * column-pass stage ring fits a 36 KB stage: float32 up to 256 px, float64 up to 64 px); mode 1 forces the per-kernel column pass (the existing
 * one, once per kernel on the shared row spectra), which embedded patch sizes always run.  Both give the same bits
 * (test and benchmark hook).  rpsf_plan_stack_info sets *fused to 1 when the plan runs k2_stack. */
int rpsf_plan_set_stack_mode(rpsf_plan* p, int mode);
int rpsf_plan_stack_info(const rpsf_plan* p, int* fused);
int rpsf_apply_stack(rpsf_plan* p, const void* image, int64_t img_pitch, int64_t img_frame_stride, void* out,
                     int64_t out_pitch, int64_t out_frame_stride, int n_kernels, int batch, const void* src, int src_dtype,
                     int64_t src_pitch, int64_t src_frame_stride, const void* mask, int64_t mask_pitch,
                     int64_t mask_frame_stride, void* stream);

/* ---- helpers -------------------------------------------------------------------------------- */
/* 2-D dtype conversion on the device (the `.astype(float)` of transform.py:117) */
int rpsf_convert(const void* src, int src_dtype, int64_t src_pitch, void* dst, int dst_dtype, int64_t dst_pitch,
                 int rows, int cols, int device, void* stream);
/* stage outputs for tests: the plan's workspace pointer / size.  It holds the patch spectra
 * [max_batch][active patch][P][P/2] complex at offset 0, then the row bands: the row pass transforms each frame row
 * once per corner column (and corner-row parity) and stores it there without the row window, and the column pass
 * applies the window as it reads a patch's rows.  After rpsf_apply_stages(..., 2) the first bytes are the patch
 * spectra exactly as with a spectrum of its own per patch; after stages = 1 the patch part holds nothing defined. */
int rpsf_plan_workspace(const rpsf_plan* p, void** ptr, int64_t* bytes);
/* run only the first `stages` kernels of apply (1 = K1, 2 = K1+K2, 3 = all); test hook */
int rpsf_apply_stages(rpsf_plan* p, const void* image, int64_t img_pitch, int64_t img_frame_stride, int img_row0,
                      int img_rows, void* out, int64_t out_pitch, int64_t out_frame_stride, int out_row0,
                      int batch, int stages, void* stream);
/* ---- fused output gather for patch-row slabs across GPUs (SURVEY.md sections 5 and 8e) ----------
 * The reference has no counterpart (it is single-process).  With mirrors set, the overlap-add kernel of
 * rpsf_apply stores every owned pixel to `out` AND to the same position of each mirror buffer — the other
 * ranks' full frames, mapped into this process with the IPC calls below, written over NVLink while the
 * kernel runs — so no all-gather follows.  Mirrors must have the layout of `out` (pitch, frame stride,
 * first row); n = 0 clears them.  Only for coverings (the streaming overlap-add), without saturation.
 * The caller orders the ranks (e.g. a barrier after the call, before anyone reads its frame). */
int rpsf_plan_set_output_mirrors(rpsf_plan* p, int n, void* const* mirrors);
/* cudaMalloc + cudaIpcGetMemHandle / cudaIpcOpenMemHandle (lazy peer access) / cudaIpcCloseMemHandle;
 * free an rpsf_ipc_alloc buffer with rpsf_device_free once every peer has closed it */
int rpsf_ipc_alloc(void** ptr, int64_t bytes, int device, unsigned char handle[64]);
int rpsf_ipc_open(void** ptr, const unsigned char handle[64], int device);
int rpsf_ipc_close(void* ptr, int device);

/* Per-stage device timing for bench.py's roofline: when enabled, rpsf_apply records CUDA events
 * on the caller's stream around K1, K2 and the K3 colour phases.  rpsf_plan_read_timing
 * synchronises those events, adds the elapsed milliseconds of every apply call since the last
 * read into ms[0..2] (K1 incl. the zero-fill when colour 0 does not tile the band, K2, K3),
 * stores the call count and resets. */
int rpsf_plan_enable_timing(rpsf_plan* p, int enabled);
int rpsf_plan_read_timing(rpsf_plan* p, double ms[3], int* calls);
/* the np.pad index map the gather kernel uses (host evaluation): source index for padded
 * position i of an axis of length n, or -1 for the zero fill of RPSF_PAD_CONSTANT */
int rpsf_pad_index(int i, int n, int pad_mode);
/* for host-only bindings (INTEGRATION.md): cudaMalloc + synchronous copy of a host buffer (e.g.
 * the kernel cube for rpsf_transform_set_kernel), and the matching free (synchronises first) */
int rpsf_upload(void** device_ptr, const void* src_host, int64_t bytes, int device);
int rpsf_device_free(void* device_ptr, int device);
/* test hook: synchronous device -> host copy of raw bytes (cudaMemcpy) */
int rpsf_copy_to_host(void* dst_host, const void* src_device, int64_t bytes, int device);
/* number of kernel launches issued by the library since load (bench.py's gpu_launches) */
int64_t rpsf_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* RPSF_B200_H */
