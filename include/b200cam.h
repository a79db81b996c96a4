/* b200cam.h - C ABI of libb200cam.so: the B200 (sm_100a) optical-encoder hot path.
 *
 * The reference (carlosh93/privacy-preserving-vision) has no FFI layer on this path: its
 * boundary is the PyTorch nn.Module `Camera` (Face-DeId/Camera/Optics.py:9).  This library sits
 * directly under that module: `Camera.forward` -> torch.autograd.Function -> ctypes -> here.
 * Each entry point names the reference lines whose arithmetic it replaces.
 *
 * Conventions
 *  - every pointer except `kappa` is a DEVICE pointer to fp32 data owned by the caller
 *    (PyTorch allocates; the library never allocates in a compute call, never synchronises,
 *    never throws).  Complex arrays are interleaved (re,im) fp32 pairs.
 *  - image tensors are NCHW contiguous, 16-byte aligned: img[b][c][y][x], c = 3 wavelengths.
 *  - `stream` is a cudaStream_t; all work is enqueued on it and is CUDA-graph capturable
 *    (b200cam_init must have been called for that N on that device before capture).
 *  - return value: 0 on success, a positive cudaError_t value, or a negative B200CAM_E_* code.
 *  - N must be one of 64, 128, 256, 512, 1024.
 *  - bf16 tensors (the _bf16 entry points: sensor image out, its gradient in) cross this ABI as `unsigned short*`: the
 *    bfloat16 bit patterns (C has no bf16 type), i.e. a torch.bfloat16 tensor's data pointer as it is.
 */
#ifndef B200CAM_H_
#define B200CAM_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200CAM_VERSION 100            /* major*10000 + minor*100 + patch */
#define B200CAM_MAX_TIES 8             /* recorded arg-max positions per image */

#define B200CAM_E_BAD_SIZE   (-1)      /* unsupported N or B < 1 */
#define B200CAM_E_NULL       (-2)      /* required pointer is NULL */
#define B200CAM_E_WORKSPACE  (-3)      /* workspace too small */
#define B200CAM_E_NOT_INIT   (-4)      /* b200cam_init(N) not called on this device */
#define B200CAM_E_ALIGN      (-5)      /* pointer not 16-byte aligned */
#define B200CAM_E_DEVICE     (-6)      /* a kernel reported a device-side error (see b200cam_device_error) */

/* Device-side error word.  Three kernels wait for other CTAs / ranks (the per-image maximum exchanged between the clusters
 * of an image, the grid barrier of the cooperative PSF kernels, the peer all-reduce of dL/dh).  A wait that outlives its
 * deadline is never turned into a result: the kernel stores one of these codes in a per-device word (mapped host memory)
 * and the next call of b200cam_device_error on that device returns it (0 = none; `clear` != 0 resets it).  The Python
 * wrappers check it after the backward of a step and raise. */
#define B200CAM_DEVERR_IMAGE_MAX_WAIT 1
#define B200CAM_DEVERR_ALLREDUCE_WAIT 2
#define B200CAM_DEVERR_GRID_BARRIER   3
int b200cam_device_error(int clear);

int b200cam_version(void);
const char* b200cam_error_string(int code);
int b200cam_supported(int N);
/* number of kernels this library has enqueued so far in this process (bench.py's gpu_launches) */
unsigned long long b200cam_launch_count(void);
/* diagnostic, no device needed: the number of batch chunks the column kernels of an N x N step split B images into when
 * `slots` CTAs are resident at once (SMs x occupancy) - the wave model of col_chunks() in csrc/b200cam.cu; 0 for an
 * unsupported N or B < 1 */
int b200cam_col_chunks(int N, int B, int slots);

/* Build the per-device twiddle table for N and opt the kernels into large dynamic shared
 * memory.  Allocates (once per device and N) - call outside stream capture. */
int b200cam_init(int N);

size_t b200cam_otf_bytes(int N);                                   /* 3*(N/2+1)*N complex */
/* The PSF workspace must be ZERO-FILLED once before its first use (it holds the grid-barrier words of the cooperative PSF
 * kernels, which the library leaves at zero); use one workspace per stream - calls that share one must not overlap. */
size_t b200cam_psf_workspace_bytes(int N);
size_t b200cam_sensor_workspace_bytes(int N, int B, int want_img_grad);
/* size of the optional saved forward spectrum (row-transformed rfft of every image plane) */
size_t b200cam_spectrum_bytes(int N, int B);

/* Image_Caption sensor epilogue (img_psf_conv, Image_Caption/Camera/Utils.py:289-295): out = nearest-resize(crop(|conv|))
 *   out[pl][i][j] = | conv[pl][off + max(i-1,0)][off + max(j-1,0)] |,  i, j < P;   conv is [planes][n][n]
 * and its adjoint (grad_conv is written everywhere: zero outside the window; d|v|/dv = 0 at v == 0 as torch.abs). */
int b200cam_crop_abs_resize_fwd(const float* conv, float* out, int planes, int n, int P, int off, void* stream);
int b200cam_crop_abs_resize_bwd(const float* grad_out, const float* conv, float* grad_conv, int planes, int n, int P, int off,
                                void* stream);

/* Zernike projection (SURVEY 8 f1; the step in front of the PSF synthesis in a training loop).
 *   h[p] = sum_j coef[j] * Z[j][p]      replaces `get_Heith_Map`, Face-DeId/Camera/Optics.py:79-83 and
 *                                        Image_Caption/Camera/Lens.py:176 (torch.sum(coef * volume, 0))
 *   grad_coef[j] = sum_p Z[j][p] * grad_h[p]   its adjoint (what autograd computes for the line above)
 * Z is [T][NN] fp32 (NN = N*N, a multiple of 4), one pass over it each way.  The forward's workspace
 * (b200cam_zernike_workspace_bytes) must be ZERO-FILLED once before the first call; the library leaves it reusable. */
size_t b200cam_zernike_workspace_bytes(int T, long long NN);
int b200cam_zernike_fwd(const float* coef, const float* Z, float* h, void* workspace, size_t workspace_bytes, int T,
                        long long NN, void* stream);
int b200cam_zernike_bwd(const float* grad_h, const float* Z, float* grad_coef, int T, long long NN, void* stream);
/* The same with the support of the basis: `active` (device, nactive ints, ascending) lists the float4 positions - index into
 * [NN/4] - at which at least one Z_j is non-zero.  The Zernike basis is zero outside the unit disc (21 % of the square): only
 * the listed positions are read, h is zero elsewhere.  NULL = every position (the calls above). */
int b200cam_zernike_fwd_ex(const float* coef, const float* Z, float* h, void* workspace, size_t workspace_bytes, int T,
                           long long NN, void* stream, const int* active, int nactive);
int b200cam_zernike_bwd_ex(const float* grad_h, const float* Z, float* grad_coef, int T, long long NN, void* stream,
                           const int* active, int nactive);

/* PSF synthesis, forward.  Replaces Camera.get_psf + the regularisers
 * (Face-DeId/Camera/Optics.py:89-120 and :124-125):
 *   V_l = A_l * exp(i*kappa_l*h);  U = ifftn(fftn(V) * H) over (lambda,y,x);  psf = |U|^2 / sum.
 *   h      [N][N]        lens height map in metres (Optics.py:79-83 output)
 *   A      [3][N][N] cplx constant pupil table  rad * t * focus * pre-phase (Optics.py:95-100)
 *   Ht     [3][N][N] cplx transfer function of Optics.py:103, TRANSPOSED to [m][u][v]
 *   rho    [N][N]        0/1 mask of Optics.py:55
 *   kappa  HOST [3]      k_l * flmb_l (Optics.py:89-90)
 *   psf    [3][N][N]     out: `psfs[0]` (centred frame, as Camera.get_psf returns it)
 *   field  [3][N][N] cplx out: propagated field U, kept for the backward pass
 *   stats  [4]           out: { sum|U|^2, loss_rad (:113), centering_loss (:124-125), scratch } */
int b200cam_psf_fwd(const float* h, const float* A, const float* Ht, const float* rho,
                    const float* kappa, float* psf, float* field, float* stats,
                    void* workspace, size_t workspace_bytes, int N, void* stream);

/* The same PSF synthesis in two calls, so that a caller can put work between them: after b200cam_psf_field the
 * workspace holds |U|^2 and the partial sums of it, which is all the OTF needs (b200cam_psf_otf_early, on the same
 * stream) - the sensor pipeline can then start while b200cam_psf_finish still writes psf and the two regularisers
 * (Optics.py:110,113,124-125).  b200cam_psf_fwd == b200cam_psf_field + b200cam_psf_finish. */
/* has_dependent != 0: `dependent_stream` (a cudaStream_t, 0 = the legacy default stream) is made to wait until the
 * FIRST kernel of the chain has finished, so that a large batch kernel enqueued there afterwards does not occupy every SM
 * before the chain's next (higher-priority) kernel is resident. */
int b200cam_psf_field(const float* h, const float* A, const float* Ht, const float* kappa, float* field,
                      void* workspace, size_t workspace_bytes, int N, void* stream, void* dependent_stream,
                      int has_dependent);
int b200cam_psf_otf_early(float* otf, void* workspace, size_t workspace_bytes, int N, void* stream);
int b200cam_psf_finish(const float* rho, float* psf, float* stats, void* workspace, size_t workspace_bytes, int N,
                       void* stream);

/* PSF synthesis, backward (autograd through Optics.py:89-125 in closed form).
 *   grad_psf     [3][N][N] or NULL   dL/dpsf
 *   grad_rad     [1] or NULL         dL/dloss_rad        (device scalars: the two regularisers are separate autograd
 *   grad_cen     [1] or NULL         dL/dcentering_loss   outputs, so their gradients arrive as two 0-dim tensors)
 *   grad_h       [N][N]              out: dL/dh */
int b200cam_psf_bwd(const float* grad_psf, const float* grad_rad, const float* grad_cen, const float* h,
                    const float* A, const float* Ht, const float* rho, const float* kappa,
                    const float* psf, const float* field, float* stats, float* grad_h,
                    void* workspace, size_t workspace_bytes, int N, void* stream);

/* Data parallel (one process per GPU, batch sharded, SURVEY 8e): b200cam_psf_bwd whose last kernel also all-reduces
 * dL/dh over NVLink peer memory - every rank pushes its rows into all peers' buffers as (value, epoch) 8-byte words (data
 * and flag in one store: no fence, no remote atomic), polls its own buffer for the peers' words, rank-ordered sum,
 * result * scale (1/world for the mean) in grad_h on every rank, bit-identical.  Replaces the framework-level gradient
 * all-reduce a DDP wrapper would issue for the reference's Camera parameters.
 *   peer_bufs  HOST array [world] of device pointers: rank r's symmetric buffer of b200cam_comm_bytes(N, world) bytes as
 *              mapped in THIS process (e.g. torch.distributed._symmetric_memory buffer_ptrs); zero-filled once before
 *              the first call, then owned by the library (per-tile epochs and the double-buffered slots live in it).
 * All ranks must call it the same number of times (it is a collective).  A rank whose peers do not arrive within
 * B200CAM_COMM_TIMEOUT_S seconds (environment, default 30) does NOT return a partial sum: its dL/dh is filled with NaN and
 * the device error word is set to B200CAM_DEVERR_ALLREDUCE_WAIT (b200cam_device_error). */
size_t b200cam_comm_bytes(int N, int world);
int b200cam_psf_bwd_allreduce(const float* grad_psf, const float* grad_rad, const float* grad_cen, const float* h, const float* A,
                              const float* Ht, const float* rho, const float* kappa, const float* psf, const float* field,
                              float* stats, float* grad_h, void* workspace, size_t workspace_bytes, int N, void* stream,
                              void* const* peer_bufs, int rank, int world, float scale);

/* Sensor image, forward.  Replaces Optics.py:126-128 + conv2D (Face-DeId/Camera/Utils.py:7-12):
 *   sensor_b = circconv(img_b, roll(psf, -N/2)) / max over (c,y,x).
 *   img      [B][3][N][N]
 *   psf      [3][N][N]                 centred PSF
 *   sensor   [B][3][N][N]              out
 *   img_max  [B]                       out: the per-image maximum before division
 *   tie_count[B], tie_pos[B][MAX_TIES] out: how many positions attain the maximum, and the first
 *                                      MAX_TIES of them as flat indices into (3,N,N)
 *   otf      b200cam_otf_bytes(N)      out: rfft2(roll(psf))/N^2 in the library's transposed layout
 *   spectrum b200cam_spectrum_bytes(N,B) or NULL  out: the row-transformed spectra of img (library layout),
 *                                      kept for b200cam_sensor_bwd (autograd would save rfftn(img), Utils.py:8);
 *                                      NULL (inference): nothing is kept, the backward recomputes them */
int b200cam_sensor_fwd(const float* img, const float* psf, float* sensor, float* img_max,
                       int* tie_count, int* tie_pos, float* otf, float* spectrum,
                       void* workspace, size_t workspace_bytes, int B, int N, void* stream);

/* The forward in two halves, for callers that overlap the PSF synthesis with the PSF-independent part of the
 * sensor path (same reference lines as b200cam_sensor_fwd; sensor_fwd == sensor_rows + sensor_finish on one stream):
 *   b200cam_sensor_rows    row transforms of the images (first half of rfftn, Utils.py:8) into `spectrum`; resets
 *                          img_max / tie_count.  Needs no PSF: may run on another stream beside b200cam_psf_fwd.
 *   b200cam_psf_otf        OTF of the PSF in the library's layout: rfft2(roll(psf, -N/2)) / N^2 (Optics.py:126 +
 *                          second operand of Utils.py:9-10).  Batch independent: may follow b200cam_psf_fwd on its stream.
 *   b200cam_sensor_finish  [OTF of the PSF unless otf_ready != 0], spectral product, inverse transform, per-image
 *                          max, normalise.
 * b200cam_sensor_split_supported(N, B) tells whether the split entry points apply (not with B200CAM_FUSED=1 at N=256). */
int b200cam_sensor_split_supported(int N, int B);
int b200cam_sensor_rows(const float* img, float* spectrum, float* img_max, int* tie_count, int B, int N, void* stream);
int b200cam_psf_otf(const float* psf, float* otf, int N, void* stream);
int b200cam_sensor_finish(const float* psf, float* sensor, float* img_max, int* tie_count, int* tie_pos, float* otf,
                          const float* spectrum, int otf_ready, void* workspace, size_t workspace_bytes, int B, int N,
                          void* stream);

/* Opt-in sensor read-out epilogue (north_star step 5 "sensor noise plus quantisation"; SURVEY trap T6).  The reference has
 * no live sensor noise and no quantiser (its gaussian_noise call is commented out: Image_Caption/Camera/Lens.py:295-301,
 * Utils.py:300-302; Face-DeId has none), so flags = 0 reproduces it.  With flags:
 *     y = conv / max;   NOISE: y += noise_scale * noise[b][c][y][x];   QUANT: y = round(clamp(y, 0, 1) * L) / L,  L = 2^quant_bits - 1
 * With NOISE, `noise` is a caller-supplied standard-normal tensor shaped like the images (drawn with the framework's seeded
 * generator, e.g. torch.randn: no kernel reproduces that stream).  b200cam_sensor_bwd treats the epilogue as the identity
 * (straight through).  Same arguments / reference lines as the calls without _ex.  The Image_Caption camera applies the same
 * epilogue through b200cam_lens_normalise_ex (below).
 *
 * NOISE_PHILOX (instead of NOISE, not with it): the kernels draw the standard normals themselves, so no noise tensor is
 * written and read back.  `noise` is then the DEVICE address (8-byte aligned) of a struct b200cam_noise_seed, read by the
 * kernels when they run (a CUDA graph replay sees whatever key the block holds by then); noise_scale must be > 0.  The value
 * added to element e of the call's [B][3][N][N] batch (flat index) is n(e) below, bit for bit what b200cam_sensor_noise writes
 * for that e, added with the arithmetic of NOISE: the output equals the NOISE call on the materialised tensor.
 *   Philox4x32-10 (Random123 / cuRAND constants), key = (lo32(key), hi32(key)), counter = (lo32(j), hi32(j), 0, 0) with
 *   j = first4 + e / 4; its four words x_0..x_3 serve e % 4 = 0..3:
 *     u_k = (2 (x_k >> 9) + 1) 2^-24        (exact in fp32, in [2^-24, 1 - 2^-24])
 *     n_0 = r cospi(2 u_1), n_1 = r sinpi(2 u_1), r = sqrt(-2 log u_0);  n_2, n_3 the same from (u_2, u_3)   (Box-Muller)
 *   so |n| <= sqrt(48 ln 2) = 5.77: the normal tail beyond that (probability ~1e-8) is cut off.  A value depends only on (key,
 *   first4 + e / 4): a batch split into shards, each with first4 advanced by the float4s before it, gives the whole batch's
 *   noise.  Not torch.randn's stream. */
#define B200CAM_SENSOR_NOISE 1
#define B200CAM_SENSOR_QUANT 2
#define B200CAM_SENSOR_NOISE_PHILOX 4
struct b200cam_noise_seed {
    unsigned long long key;      /* Philox key */
    unsigned long long first4;   /* counter of the call's first four elements */
};
/* The noise of NOISE_PHILOX materialised: out[e] = n(e) for e in [0, count), count % 4 == 0, out 16-byte aligned, seed_block
 * as above (for tests, and for callers whose read-out does not run in these kernels). */
int b200cam_sensor_noise(const void* seed_block, float* out, long long count, void* stream);
int b200cam_sensor_fwd_ex(const float* img, const float* psf, float* sensor, float* img_max, int* tie_count, int* tie_pos,
                          float* otf, float* spectrum, void* workspace, size_t workspace_bytes, int B, int N, void* stream,
                          int flags, const float* noise, float noise_scale, int quant_bits);
int b200cam_sensor_finish_ex(const float* psf, float* sensor, float* img_max, int* tie_count, int* tie_pos, float* otf,
                             const float* spectrum, int otf_ready, void* workspace, size_t workspace_bytes, int B, int N,
                             void* stream, int flags, const float* noise, float noise_scale, int quant_bits);

/* Sensor image, backward (autograd through Optics.py:126-128 in closed form, incl. the amax term).
 *   grad_sensor [B][3][N][N]   dL/dsensor
 *   sensor, img_max, tie_count, tie_pos, otf, spectrum (or NULL): outputs of b200cam_sensor_fwd on the same img/psf
 *   grad_psf    [3][N][N]      out: dL/dpsf (centred frame), summed over the batch
 *   grad_img    [B][3][N][N]   out or NULL (no reference caller needs it) */
int b200cam_sensor_bwd(const float* grad_sensor, const float* img, const float* sensor,
                       const float* img_max, const int* tie_count, const int* tie_pos,
                       const float* psf, const float* otf, const float* spectrum,
                       float* grad_psf, float* grad_img,
                       void* workspace, size_t workspace_bytes, int B, int N, void* stream);

/* bf16 hand-over to a downstream network that runs in bf16 (torch.autocast): the same forward and backward, with the sensor
 * image written and its gradient read in bf16.  Saves the cast kernels at the boundary: the fp32 image written and re-read
 * by the cast, the bf16 gradient widened into an fp32 copy.
 *   b200cam_sensor_fwd_bf16 / _finish_bf16   the arguments of the _ex calls, with the sensor output split in two:
 *       conv    [B][3][N][N] fp32 scratch: the un-normalised image (caller-owned; dead once the call's kernels have run)
 *       sensor  [B][3][N][N] bf16 out: the fp32 sensor image after the read-out epilogue, rounded to nearest-even - bit for bit
 *               the fp32 call's output cast with torch's .to(torch.bfloat16)
 *   b200cam_sensor_bwd_bf16   b200cam_sensor_bwd with grad_sensor [B][3][N][N] bf16, widened exactly in the row kernels; it
 *       takes no sensor image (the backward never reads it).  dL/dpsf and dL/dimg are those of b200cam_sensor_bwd on the
 *       widened gradient, bit for bit.
 * These always run the default two-pass pipeline: the opt-in B200CAM_PLANE=1 and B200CAM_ONE_PASS=1 kernels are fp32 only
 * and are not used.  With B200CAM_PLANE=1 at N = 256 b200cam_sensor_rows writes the plane layout, which
 * b200cam_sensor_finish_bf16 cannot read: it returns B200CAM_E_BAD_SIZE there (use b200cam_sensor_fwd_bf16). */
int b200cam_sensor_fwd_bf16(const float* img, const float* psf, float* conv, unsigned short* sensor, float* img_max, int* tie_count,
                            int* tie_pos, float* otf, float* spectrum, void* workspace, size_t workspace_bytes, int B, int N,
                            void* stream, int flags, const float* noise, float noise_scale, int quant_bits);
int b200cam_sensor_finish_bf16(const float* psf, float* conv, unsigned short* sensor, float* img_max, int* tie_count, int* tie_pos,
                               float* otf, const float* spectrum, int otf_ready, void* workspace, size_t workspace_bytes, int B,
                               int N, void* stream, int flags, const float* noise, float noise_scale, int quant_bits);
int b200cam_sensor_bwd_bf16(const unsigned short* grad_sensor, const float* img, const float* img_max, const int* tie_count,
                            const int* tie_pos, const float* psf, const float* otf, const float* spectrum, float* grad_psf,
                            float* grad_img, void* workspace, size_t workspace_bytes, int B, int N, void* stream);

/* uint8 images (what a decoder yields, a quarter of the bytes of fp32): the same calls with img [B][3][N][N] as uint8, 16-byte
 * aligned.  Each value is read as x * fp32(1/255) wherever the kernels read the image (the row transforms, the arg-max term of
 * the backward), bit-identical to torch's img.float() / 255.0 on the GPU: every output - sensor image (fp32 or bf16), spectra,
 * dL/dpsf, dL/dimg - is that of the fp32 call on the converted batch, bit for bit.  No fp32 copy of the batch is made.
 *   b200cam_sensor_rows_u8       b200cam_sensor_rows; finish with b200cam_sensor_finish / _finish_ex / _finish_bf16 unchanged
 *   b200cam_sensor_fwd_u8        b200cam_sensor_fwd_ex (epilogue arguments included)
 *   b200cam_sensor_fwd_u8_bf16   b200cam_sensor_fwd_bf16
 *   b200cam_sensor_bwd_u8        b200cam_sensor_bwd (the same img as the forward; spectrum NULL re-runs the row pass on it)
 *   b200cam_sensor_bwd_u8_bf16   b200cam_sensor_bwd_bf16
 * Workspace sizes are those of the fp32 calls.  These always run the default two-pass pipeline (the opt-in B200CAM_PLANE=1
 * kernels read fp32 images only; B200CAM_ONE_PASS=1 still applies).  With B200CAM_PLANE=1 at N = 256 b200cam_sensor_finish
 * expects the plane layout, so b200cam_sensor_rows_u8 returns B200CAM_E_BAD_SIZE there (use b200cam_sensor_fwd_u8). */
int b200cam_sensor_rows_u8(const unsigned char* img, float* spectrum, float* img_max, int* tie_count, int B, int N, void* stream);
int b200cam_sensor_fwd_u8(const unsigned char* img, const float* psf, float* sensor, float* img_max, int* tie_count, int* tie_pos,
                          float* otf, float* spectrum, void* workspace, size_t workspace_bytes, int B, int N, void* stream, int flags,
                          const float* noise, float noise_scale, int quant_bits);
int b200cam_sensor_fwd_u8_bf16(const unsigned char* img, const float* psf, float* conv, unsigned short* sensor, float* img_max,
                               int* tie_count, int* tie_pos, float* otf, float* spectrum, void* workspace, size_t workspace_bytes,
                               int B, int N, void* stream, int flags, const float* noise, float noise_scale, int quant_bits);
int b200cam_sensor_bwd_u8(const float* grad_sensor, const unsigned char* img, const float* sensor, const float* img_max,
                          const int* tie_count, const int* tie_pos, const float* psf, const float* otf, const float* spectrum,
                          float* grad_psf, float* grad_img, void* workspace, size_t workspace_bytes, int B, int N, void* stream);
int b200cam_sensor_bwd_u8_bf16(const unsigned short* grad_sensor, const unsigned char* img, const float* img_max, const int* tie_count,
                               const int* tie_pos, const float* psf, const float* otf, const float* spectrum, float* grad_psf,
                               float* grad_img, void* workspace, size_t workspace_bytes, int B, int N, void* stream);

/* Plain circular convolution of a batch with one centred kernel per channel, and its adjoints.  Replaces the FFT
 * part of img_psf_conv (Image_Caption/Camera/Utils.py:251-297): the caller zero-pads image and PSF to N (a power of
 * two, Utils.py:266-277 and psf2otf :127-158), then
 *     out_b = irfft2( rfft2(img_b) * rfft2(roll(kernel, -N/2)) )               (Utils.py:279-288)
 * (the reference's abs / crop / nearest resize and the batch-global max of Lens.py:312 stay in the wrapper).
 *   img, out    [B][3][N][N]      kernel [3][N][N] (centre at N/2, N/2)
 *   otf         b200cam_otf_bytes(N)   out (fwd) / in (bwd)
 *   spectrum    b200cam_spectrum_bytes(N,B) or NULL: row spectra of img kept for the backward
 *   grad_kernel [3][N][N] out: sum over the batch;  grad_img [B][3][N][N] out or NULL */
int b200cam_conv_fwd(const float* img, const float* kernel, float* out, float* otf, float* spectrum, void* workspace,
                     size_t workspace_bytes, int B, int N, void* stream);
int b200cam_conv_bwd(const float* grad_out, const float* img, const float* otf, const float* spectrum, float* grad_kernel,
                     float* grad_img, void* workspace, size_t workspace_bytes, int B, int N, void* stream);

/* PSF synthesis of the Image_Caption camera (OpticsZernike.forward, Image_Caption/Camera/Lens.py:176-274), batch
 * independent, and its adjoint into the height map.  R = wave resolution (R x R height map, R % 4 == 0), P = patch size.
 *   phase plate        field = A * exp(i delta_l (h + noise))        Utils.py:192-205 (fp64 phase -> complex64), 396-410
 *   Fresnel propagation zero-pad R -> n = R + 2 (R/4), FFT2, x H, IFFT2, crop     Utils.py:329-378.  n = 1344 = 2^6 3 7 for the
 *                      shipped R = 896: mixed-radix transforms (2/3/4/5/7/8 and any prime <= 31), zero rows / columns pruned
 *   intensity, area down-sampling to P x P (nearest x up, up x up mean)           Utils.py:208, 216-248
 *   per-channel normalisation, disc masks and energy loss                         Lens.py:239, 269-274
 * Inputs (device unless noted):
 *   h [R][R] fp32; noise [R][R] fp32 or NULL - the U(-tol,tol) field of PhasePlate._build drawn by the caller with the
 *   reference's own torch.rand call; A [3][R][R] complex64 = aperture * spherical wavefront (Lens.py:191-213, Utils.py:88-97);
 *   delta HOST double[3] = 2 pi / lambda_l * (n_l - 1); Hx [3][n] complex128 = exp(-i pi lambda_l z f_k^2), f in FFT order
 *   (the transfer function is separable: H(fx, fy) = Hx(fx) Hx(fy), multiplied in fp64); tw [n] complex64 = exp(-2 pi i k / n);
 *   mask1 / mask2 [P][P][3] fp64 (flags & 1 / flags & 2), else NULL.
 * Outputs: field, U [3][R][R] complex64 (saved for the backward); psf [P][P][3] fp32 (normalised, unmasked); chan_sum [3];
 *   psf_out [P][P][3] fp64 = psf (* mask2 with flag 2); loss: device double = || psf * mask1 - psf ||_2 (flag 1).
 * flags: 1 = energy loss (prueba "1"/"3"), 2 = mask the PSF (prueba "2"/"3"). */
int b200cam_lens_psf_supported(int R, int P);
int b200cam_lens_psf_padded(int R);                                  /* n */
size_t b200cam_lens_psf_workspace_bytes(int R, int P);
int b200cam_lens_psf_fwd(const float* h, const float* noise, const float* A, const double* delta, const double* Hx, const float* tw,
                         float* field, float* U, float* psf, float* chan_sum, const double* mask1, const double* mask2, int flags,
                         double* psf_out, double* loss, void* workspace, size_t workspace_bytes, int R, int P, void* stream);
/* grad_psf_out [P][P][3] fp64 (dL/dpsf_out) or NULL, grad_loss device double or NULL; the rest as produced by the forward.
 * grad_h [R][R] fp32 out. */
int b200cam_lens_psf_bwd(const double* grad_psf_out, const double* grad_loss, const double* loss, const float* psf,
                         const float* chan_sum, const float* field, const float* U, const double* delta, const double* Hx,
                         const float* tw, const double* mask1, const double* mask2, int flags, float* grad_h, void* workspace,
                         size_t workspace_bytes, int R, int P, void* stream);

/* Sensor image of the Image_Caption camera: img_psf_conv (Image_Caption/Camera/Utils.py:251-297) + the batch-global
 * normalisation (Lens.py:312) with the padding, |.|, crop and nearest resize inside the transform kernels.  P = patch size
 * (64, 128, 256 or 512), transform size n = 2P (b200cam_init(n) first).  The 4x zero-padded image and the 4x convolution
 * output of the reference never exist: zero rows / columns are pruned from every pass.
 *   b200cam_lens_sensor_fwd   raw[b][c][i][j] = conv[pt + max(i,1)][pt + max(j,1)], conv = ifft2(fft2(pad(img)) * OTF), pt = P/2
 *                             (signed: the sensor value is |raw|; = Utils.py:279-295), gmax = max(gmax, max |raw|) by integer
 *                             atomics (zero it first; all-reduce it across ranks for a sharded batch)
 *       img [B][3][P][P]; kernel [3][n][n] = the PSF zero-padded with its centre at (n/2, n/2) (psf2otf, Utils.py:127-158);
 *       otf  b200cam_otf_bytes(n) out; spectrum b200cam_spectrum_bytes(n, B) out (row spectra of the images, for the backward)
 *   b200cam_lens_normalise    y = |raw| / gmax                                                         (Lens.py:312)
 *   b200cam_lens_sensor_dot   dot_ties[0] = sum(grad_y * y), dot_ties[1] = #{ |raw| == gmax } over this rank's batch
 *   b200cam_lens_sensor_bwd   adjoint: dL/dconv = sign(raw) (grad_y / gmax - [|raw| == gmax] coef), coef = s / (gmax n) a device
 *                             scalar from the (all-reduced) dot_ties; grad_kernel [3][n][n] summed over the batch (crop it to
 *                             the PSF window), grad_img [B][3][P][P] or NULL
 * workspace: b200cam_lens_sensor_workspace_bytes(P, B), shared by the four calls of a step.
 * Read-out variants (same reference lines, same checks):
 *   b200cam_lens_sensor_fwd_u8  the forward from uint8 images img [B][3][P][P] (what a decoder or the caption HDF5 store
 *                               yields, a quarter of the bytes): each value is read as x * fp32(1/255), bit-identical to
 *                               torch's img.float() / 255.0 on the GPU; the padded image still never exists.  The backward is
 *                               the same (it reads the saved spectrum and raw, never the image).
 *   b200cam_lens_normalise_ex   y = |raw| / gmax followed by the opt-in read-out epilogue of b200cam_sensor_fwd_ex
 *                               (flags B200CAM_SENSOR_NOISE / _QUANT, noise [B][3][P][P] indexed like y, or _NOISE_PHILOX with
 *                               e the flat index into y; flags = 0 is b200cam_lens_normalise).  b200cam_lens_sensor_dot / _bwd read raw, not y: straight through.
 * bf16 variants (a downstream network in bf16): same arguments and checks, y / grad_y as bf16 bit patterns.
 *   b200cam_lens_normalise_bf16   b200cam_lens_normalise_ex rounded to nearest-even as the last step (= its output cast with
 *                                 torch); b200cam_lens_sensor_dot_bf16 / _bwd_bf16 read grad_y in bf16, widened exactly, and
 *                                 equal the fp32 calls on the widened gradient, bit for bit. */
size_t b200cam_lens_sensor_workspace_bytes(int P, int B);
int b200cam_lens_sensor_fwd(const float* img, const float* kernel, float* raw, float* gmax, float* otf, float* spectrum, void* workspace,
                            size_t workspace_bytes, int B, int P, void* stream);
int b200cam_lens_sensor_fwd_u8(const unsigned char* img, const float* kernel, float* raw, float* gmax, float* otf, float* spectrum,
                               void* workspace, size_t workspace_bytes, int B, int P, void* stream);
int b200cam_lens_normalise(const float* raw, const float* gmax, float* y, long long count, void* stream);
int b200cam_lens_normalise_ex(const float* raw, const float* gmax, float* y, long long count, void* stream, int flags, const float* noise,
                              float noise_scale, int quant_bits);
int b200cam_lens_sensor_dot(const float* grad_y, const float* raw, const float* gmax, float* dot_ties, void* workspace, size_t workspace_bytes,
                            int B, int P, void* stream);
int b200cam_lens_sensor_bwd(const float* grad_y, const float* raw, const float* gmax, const float* coef, const float* otf, const float* spectrum,
                            float* grad_kernel, float* grad_img, void* workspace, size_t workspace_bytes, int B, int P, void* stream);
int b200cam_lens_normalise_bf16(const float* raw, const float* gmax, unsigned short* y, long long count, void* stream, int flags,
                                const float* noise, float noise_scale, int quant_bits);
int b200cam_lens_sensor_dot_bf16(const unsigned short* grad_y, const float* raw, const float* gmax, float* dot_ties, void* workspace,
                                 size_t workspace_bytes, int B, int P, void* stream);
int b200cam_lens_sensor_bwd_bf16(const unsigned short* grad_y, const float* raw, const float* gmax, const float* coef, const float* otf,
                                 const float* spectrum, float* grad_kernel, float* grad_img, void* workspace, size_t workspace_bytes, int B,
                                 int P, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200CAM_H_ */
