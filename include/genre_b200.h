/*
 * genre_b200.h — C ABI of libgenre_b200.so (sm_100a).
 *
 * This is the drop-in boundary for the GenRe/ShapeHD geometric-projection hot path.  Every entry
 * point takes plain device pointers, sizes, element strides and a cudaStream_t (passed as void*);
 * there are no torch types.  The caller (the Python mirror of the reference's toolbox packages, or
 * any other host) owns every buffer, including scratch ("workspace"): the library never allocates
 * device memory and never synchronises the device.  All launches go to the given stream and are
 * CUDA-graph capturable.
 *
 * Each function states the reference interface it replaces (paths relative to the reference root).
 * Reference convention: cffi functions on THCudaTensor*, returning int 1, failing through
 * THError("aborting") (toolbox/cam_bp/cam_bp/src/back_projection.c:9-57).  Here: return 0 on success,
 * a positive cudaError_t if a launch failed, or a negative GENRE_B200_E* code for an argument error;
 * genre_b200_last_error() gives the message (thread-local).  The Python mirror turns non-zero into
 * RuntimeError, which is what THError became on the Python side.
 *
 * All tensors are fp32 unless stated otherwise.  "strides" are in ELEMENTS, not bytes, and may be 0
 * (broadcast) where noted.
 */
#ifndef GENRE_B200_H
#define GENRE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GENRE_B200_OK 0
#define GENRE_B200_EINVAL (-1)      /* bad shape / null pointer / unsupported size        */
#define GENRE_B200_EWORKSPACE (-2)  /* workspace too small (see *_workspace_bytes)         */
#define GENRE_B200_EALIGN (-3)      /* a dense buffer is not 16-byte aligned               */

/* flags for the projection entry points */
#define GENRE_B200_FLAG_SHIFT_TDF 1u /* fuse Camera_back_projection_layer.shift_tdf: 1 - R*tdf */

const char *genre_b200_last_error(void);
/* library/ABI version: major*1000 + minor */
int genre_b200_version(void);

/* ---------------------------------------------------------------------------------------------
 * Camera back-projection, depth -> voxel TDF.
 * Replaces back_projection_forward (toolbox/cam_bp/cam_bp/src/back_projection.h:1,
 * back_projection.c:9-17, back_projection_kernel.cu:199-306,760-838) together with the dense
 * initialisation the Python caller performs (functions/cam_back_projection.py:22-24) and, when
 * GENRE_B200_FLAG_SHIFT_TDF is set, modules/camera_backprojection_module.py:26-28.
 *
 *   depth   [N, C, H, W]  any strides (sN,sC,sH,sW); ray depth, pixels with depth < 0 are skipped
 *   fl      [N, C]        strides (fN, fC)     focal length in pixels
 *   camdist [N, C]        strides (dN, dC)     camera distance from the origin along -x
 *   tdf     [N, C, R, R, R] dense, 16-byte aligned, written completely (no pre-initialisation needed)
 *             without SHIFT: mean point-to-centre distance on hit voxels, 1/R elsewhere
 *             with    SHIFT: 1 - R*mean on hit voxels, 1 - R*(1/R) elsewhere
 *   cnt     [N, C, R, R, R] dense or NULL; if given, the per-voxel point count as fp32 (what the
 *             reference keeps on ctx for backward, cam_back_projection.py:28)
 *   flags   0 or GENRE_B200_FLAG_SHIFT_TDF; any other bit is rejected with GENRE_B200_EINVAL
 *   workspace: genre_b200_voxelize_workspace_bytes(N*C, H*W, R) bytes, 16-byte aligned
 * ------------------------------------------------------------------------------------------- */
size_t genre_b200_voxelize_workspace_bytes(int64_t n_maps, int64_t pixels_per_map, int res);

int genre_b200_cam_bp_forward(const float *depth, int64_t N, int64_t C, int64_t H, int64_t W,
                              int64_t sN, int64_t sC, int64_t sH, int64_t sW,
                              const float *fl, int64_t fN, int64_t fC,
                              const float *camdist, int64_t dN, int64_t dC,
                              float *tdf, float *cnt, int res, unsigned flags,
                              void *workspace, size_t workspace_bytes, void *stream);

/* Replaces back_projection_backward (back_projection.h:2, back_projection_kernel.cu:365-471,897-963)
 * with the intended cam_dist indexing (the reference reads cam_dist with cnt's strides at :401).
 *   cnt, grad_tdf [N,C,R,R,R] dense;  grad_depth [N,C,H,W] dense (fully written);
 *   grad_fl, grad_camdist [N,C] dense (fully written). */
int genre_b200_cam_bp_backward(const float *depth, int64_t N, int64_t C, int64_t H, int64_t W,
                               int64_t sN, int64_t sC, int64_t sH, int64_t sW,
                               const float *fl, int64_t fN, int64_t fC,
                               const float *camdist, int64_t dN, int64_t dC,
                               const float *cnt, const float *grad_tdf, int res,
                               float *grad_depth, float *grad_fl, float *grad_camdist, void *stream);

/* Replaces get_surface_mask (back_projection.h:3, back_projection_kernel.cu:309-358,840-891).
 *   cnt  [N,C,R,R,R] dense (from genre_b200_cam_bp_forward);  mask [N,C,R,R,R] dense, fully written:
 *   1 everywhere except empty voxels that lie behind the observed depth surface. */
int genre_b200_surface_mask(const float *depth, int64_t N, int64_t C, int64_t H, int64_t W,
                            int64_t sN, int64_t sC, int64_t sH, int64_t sW,
                            const float *fl, int64_t fN, int64_t fC,
                            const float *camdist, int64_t dN, int64_t dC,
                            const float *cnt, float *mask, int res, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Spherical back-projection, spherical depth map -> voxel TDF + count.
 * Replaces spherical_back_proj_forward / _backward (back_projection.h:4-5,
 * back_projection_kernel.cu:474-757; functions/sperical_to_tdf.py:13-47).
 *   sph  [N, C, H, W]    any strides; radius along the ray, < 0 skipped
 *   grid [N, C, H, W, 3] any strides (gN may be 0: one direction table shared by the batch)
 *   tdf, cnt [N,C,R,R,R] dense, fully written: mean distance / count on hit voxels, 0 elsewhere
 * ------------------------------------------------------------------------------------------- */
int genre_b200_sph_bp_forward(const float *sph, int64_t N, int64_t C, int64_t H, int64_t W,
                              int64_t sN, int64_t sC, int64_t sH, int64_t sW,
                              const float *grid, int64_t gN, int64_t gC, int64_t gH, int64_t gW, int64_t gD,
                              float *tdf, float *cnt, int res,
                              void *workspace, size_t workspace_bytes, void *stream);

int genre_b200_sph_bp_backward(const float *sph, int64_t N, int64_t C, int64_t H, int64_t W,
                               int64_t sN, int64_t sC, int64_t sH, int64_t sW,
                               const float *grid, int64_t gN, int64_t gC, int64_t gH, int64_t gW, int64_t gD,
                               const float *cnt, const float *grad_tdf, int res,
                               float *grad_sph, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Stop probability along rays.  Replaces calc_prob_forward / calc_prob_backward
 * (toolbox/calc_prob/calc_prob/src/calc_prob.h:1-2, calc_prob_kernel.cu:112-266).
 *   prob_in, stop_prob, grad_in...: [n_rays, Z] dense (the reference's [N,C,X,Y,Z] flattened)
 *   forward : stop[z] = p[z] * prod_{k<z} (1 - p[k])        (p must lie in (0,1), as the reference)
 *   backward: grad_prob from stop_prob_weighted = stop * grad_stop (calc_prob.py:27)
 * ------------------------------------------------------------------------------------------- */
int genre_b200_calc_prob_forward(const float *prob_in, float *stop_prob, int64_t n_rays, int64_t Z, void *stream);
int genre_b200_calc_prob_backward(const float *prob_in, const float *stop_prob_weighted, float *grad_prob,
                                  int64_t n_rays, int64_t Z, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Fused spherical renderer: voxel occupancy -> spherical depth map.
 * Replaces render_spherical.forward (toolbox/spherical_proj.py:62-72): trilinear grid_sample
 * (align_corners=True semantics of torch 0.4.1, zero padding) of vox.permute(0,1,4,3,2) along
 * rays dir[h,w]*2*(1 - k/(Z-1)), clamp to [1e-5, 1-1e-5], stop-probability scan, expected depth
 * sum_k s_k*k/(Z-1) + prod_k(1 - p_k), without materialising any [N,1,S,S,Z] tensor.
 *   vox  [N, R, R, R] dense (C must be 1 as in the reference)
 *   dirs [S, S, 3]    dense fp64 unit directions (the numpy table of spherical_proj.py:43-51 BEFORE its
 *                     float cast; sample positions are formed in fp64 and rounded once, like :52-57)
 *   depth_weight [Z]  the module's registered buffer linspace(0,1,Z) (spherical_proj.py:58)
 *   out  [N, S, S]    dense
 * ------------------------------------------------------------------------------------------- */
int genre_b200_render_spherical_forward(const float *vox, int64_t N, int res,
                                        const double *dirs, int sph_res, int z_res,
                                        const float *depth_weight, float *out, void *stream);
/* gradient of the above w.r.t. vox; grad_vox [N,R,R,R] must be zeroed by the caller (accumulated with
 * atomics, like grid_sampler_3d_backward); z_res <= 256 */
int genre_b200_render_spherical_backward(const float *vox, int64_t N, int res,
                                         const double *dirs, int sph_res, int z_res,
                                         const float *depth_weight,
                                         const float *grad_out, float *grad_vox, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Chamfer nearest-neighbour distance.  Replaces nnd_forward_cuda / nnd_backward_cuda
 * (toolbox/nndistance/src/my_lib_cuda.h:1-4, nnd_cuda.cu:6-177; functions/nnd.py:8-63).
 *   xyz1 [B,N,3], xyz2 [B,M,3] dense;  dist1 [B,N], dist2 [B,M] squared distances;
 *   idx1 [B,N], idx2 [B,M] int32 argmin, lowest index on ties.
 *   backward fully writes grad_xyz1 [B,N,3], grad_xyz2 [B,M,3] (zeroing included).
 * Unlike the reference (nnd_cuda.cu:130-131 launches on the legacy default stream) the given
 * stream is honoured.
 * ------------------------------------------------------------------------------------------- */
int genre_b200_nnd_forward(const float *xyz1, const float *xyz2, int64_t B, int64_t N, int64_t M,
                           float *dist1, float *dist2, int32_t *idx1, int32_t *idx2, void *stream);
int genre_b200_nnd_backward(const float *xyz1, const float *xyz2, int64_t B, int64_t N, int64_t M,
                            const float *grad_dist1, const float *grad_dist2,
                            const int32_t *idx1, const int32_t *idx2,
                            float *grad_xyz1, float *grad_xyz2, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Stage-level entry points of the voxelisation pipeline (used by bench.py to time the dominant
 * kernel on its own, and by tests).  genre_b200_cam_bp_forward == stage_project + stage_splat.
 * ------------------------------------------------------------------------------------------- */
int genre_b200_cam_bp_stage_project(const float *depth, int64_t N, int64_t C, int64_t H, int64_t W,
                                    int64_t sN, int64_t sC, int64_t sH, int64_t sW,
                                    const float *fl, int64_t fN, int64_t fC,
                                    const float *camdist, int64_t dN, int64_t dC, int res,
                                    void *workspace, size_t workspace_bytes, void *stream);
int genre_b200_voxelize_stage_splat(int64_t n_maps, int64_t pixels_per_map, int res,
                                    float *tdf, float *cnt, float hit_alpha, float hit_beta, float background,
                                    void *workspace, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------
 * ConvTranspose3d(kernel K in {4, 8}, stride 2, padding K/2 - 1) forward as a tcgen05 implicit GEMM (TF32 operands,
 * FP32 accumulation in TMEM).  Replaces the cuDNN call behind nn.ConvTranspose3d in networks/networks.py:211-222
 * (Unet_3D Deconv3d_skip: the channel concatenation of :221 is walked as two K ranges, never materialised) and
 * :253-256 (deconv3d_2x of VoxelDecoder / VoxelGenerator).
 *   src0 [B*D][cg0][H][W][16 B], src1 [...] or NULL   channel-blocked activations; a channel group is 16 bytes per
 *           position: 4 fp32 read as TF32 (f16 = 0) or 8 fp16 (f16 = 1; same 10-bit mantissa, half the operand bytes:
 *           the kernels are bound by shared-memory operand bandwidth, so this path is ~2x faster)
 *   wpack   weights packed per (parity, z-tap, 8-channel chunk) stage: see genre_shapehd_b200/ops_conv.py
 *   scale, shift [npad]   y = act(acc * scale + shift): bias and folded eval-mode BatchNorm3d
 *   slope   LeakyReLU slope (1 = none);   out [B*2D][cgo][2H][2W][4]
 * Supported: W in {16,32}, H % 16 == 0, cg0 + cg1 even, 4*cgo <= npad, npad in {32,64}.
 * ------------------------------------------------------------------------------------------- */
int genre_b200_convt3d_s2_forward(const void *src0, int cg0, const void *src1, int cg1,
                                  int64_t B, int64_t D, int64_t H, int64_t W,
                                  const void *wpack, int ksize, int npad, int f16,
                                  const float *scale, const float *shift, float slope,
                                  float *out, int cgo, void *stream);

/* Stride-1 convolution with `taps` (3 or 5) taps per dimension on channel-blocked activations, same tcgen05 kernel:
 *   out[b,z,y,x,n] = act(scale[n] * sum_{t,c} in[b, z+base-tz, y+base-ty, x+base-tx, c] * W[t][c][n] + shift[n])
 * Replaces the cuDNN call behind nn.Conv3d of Unet_3D.enc1 (networks/networks.py:151,197: Conv3d(2->20, k=8, s=2, p=3))
 * after a space-to-depth of the input (k=8/s=2 over C channels == 5 taps/s=1 over 8C channels).
 *   wpack [taps][C/8][taps*taps][2][npad/8][8][4];  out [B*D][cgo][H][W][4];  W in {16,32,64}, H % 16 == 0, npad = 32
 *   (npad = 64 with 3 taps: Conv3d(1 -> 64, k4, s2, p1) over the 2x space-to-depth input, VoxelDiscriminator main.0;
 *    npad = 96 with 5 taps: Conv3d(20 -> 80, k8, s2, p3) = the input gradient of Unet_3D.dec5) */
int genre_b200_conv3d_taps_forward(const void *src0, int cg0, const void *src1, int cg1,
                                   int64_t B, int64_t D, int64_t H, int64_t W,
                                   const void *wpack, int taps, int base, int npad, int f16,
                                   const float *scale, const float *shift, float slope,
                                   float *out, int cgo, void *stream);

/* Conv3d(kernel 4, stride 2, padding 1) forward on the same tcgen05 kernel.  Replaces the cuDNN call behind conv3d_half
 * (VoxelDiscriminator, networks/networks.py:247-250) and Unet_3D.enc2..enc5 (:152-155).  The input arrives as its 8 parity
 * sub-volumes in one channel-blocked tensor src [B*D'][8*cgs][H'][W'][16 B] (D' = D/2 ...; group index = s*cgs + c,
 * s = (pz*2+py)*2+px); sub-volume s is a K range with 2 taps per dimension (kernel index 3 - 2t - p).
 *   wpack [2][kblocks*8*cgs/2][4][2][npad/8][8][g];  out [B*D'][cgo][H'][W'][4];  W' in {16,32}, H' % 16 == 0, cgs even,
 *   npad in {32,64,96,128}.  kblocks: 1, or 3 when src holds the lo|hi|hi blocks of genre_b200_blocked_split3. */
int genre_b200_conv3d_k4s2_forward(const void *src, int cgs, int kblocks, int64_t B, int64_t D, int64_t H, int64_t W,
                                   const void *wpack, int npad, int f16,
                                   const float *scale, const float *shift, float slope,
                                   float *out, int cgo, void *stream);

/* The k 4 / s 2 / p 1 convolutions of the SMALL volumes (coarse side <= 8^3: Unet_3D.enc4, enc5, dec2, dec3,
 * networks/networks.py:157-165; the 4^3 / 8^3 stages of VoxelDecoder / VoxelGenerator / VoxelDiscriminator :40-57,:79-97,:247-256)
 * as a tcgen05 implicit GEMM over the flattened, zero-separated volume (csrc/convflat.cu).  Replaces the cuDNN calls behind
 * those nn.Conv3d / nn.ConvTranspose3d modules in eval mode.
 *   genre_b200_convflat_positions: positions per channel-group array of the operand of a coarse (B, D, H, W) volume
 *       (*lead = index of position 0);
 *   genre_b200_convflat_pack: NCDHW fp32 -> operand [parts][cgs][P][8 fp16] (parts 2 = fp16 hi | lo' = (a - hi) * 2^11), groups
 *       [cg_off, ...); subvol = 1: src is [B, C, 2D, 2H, 2W] and becomes 8 parity sub-volume blocks of C/8 groups (C % 8 == 0);
 *       src NULL: zero `zero_groups` groups (padding to an even group count);
 *   genre_b200_convflat_forward: out[B, Cout, Do, Ho, Wo] (NCDHW fp32) = lrelu(scale * conv + shift); transposed 1:
 *       ConvTranspose3d, output 2x the coarse volume; 0: Conv3d of the 2x volume given as sub-volume blocks (cgs % 16 == 0),
 *       output the coarse volume.  wpack [classes 8|1][ceil(Cout/npad)][cgs/2][8 taps][2][parts*npad/8][8][8] fp16, npad 64 | 80,
 *       op 1 (fp16 operands) | 2 (hi/lo split, fp32-accurate). */
int64_t genre_b200_convflat_positions(int64_t B, int D, int H, int W, int *lead);
int genre_b200_convflat_pack(const float *src, int C, int64_t B, int D, int H, int W, int subvol, void *operand, int cg_off,
                             int cgs, int parts, int zero_groups, void *stream);
int genre_b200_convflat_forward(const void *operand, int cgs, int64_t B, int D, int H, int W, int transposed,
                                const void *wpack, int npad, int op, const float *scale, const float *shift, float slope,
                                float *out, int Cout, void *stream);

/* The two degenerate convolutions at the bottom of the U-Net as weight-streaming FP32 products (csrc/skinny_gemm.cu):
 * Conv3d whose kernel covers its whole input (Unet_3D.enc6, networks/networks.py:157: W is [N = Cout][K = Cin*k^3], w_is_nk = 1)
 * and ConvTranspose3d on a 1^3 input (Unet_3D.dec1 :162, VoxelDecoder / VoxelGenerator main.0 :40,:79: W is [K = Cin][N = Cout*k^3],
 * w_is_nk = 0, chan_div = k^3).  Replaces the cuDNN / cuBLAS calls behind those modules in eval mode.
 *   out[M][N] = lrelu(scale[n / chan_div] * (x[M][K] @ W) + shift[n / chan_div]); fp32 throughout (FP32 FMAs, fixed summation order);
 *   the contiguous extent of W a multiple of 4; workspace = genre_b200_skinny_gemm_workspace_bytes(M, N, K, w_is_nk). */
size_t genre_b200_skinny_gemm_workspace_bytes(int64_t M, int64_t N, int64_t K, int w_is_nk);
int genre_b200_skinny_gemm(const float *x, const float *W, int64_t M, int64_t N, int64_t K, int w_is_nk, int chan_div,
                           const float *scale, const float *shift, float slope, float *out, void *workspace,
                           size_t workspace_bytes, void *stream);

/* ConvTranspose3d(Cin -> 1, kernel 4, stride 2, padding 1) on 64-wide volumes as a tcgen05 GEMM over the 64 kernel taps
 * (P[position, tap] = sum_c x[c, position] W[c, tap]) followed by a shared-memory col2im (csrc/convt_c1_col2im.cu).  Replaces the
 * cuDNN call behind the last layer of each decoder (Unet_3D.dec6 networks/networks.py:167-168, VoxelDecoder :57, VoxelGenerator :98).
 *   src0 [B*D][parts*cg0][H][64][8 fp16], src1 likewise (cg1 groups) or NULL; parts 1 (op 1: fp16) | 2 (op 2: hi | lo' split,
 *   fp32-accurate); cg0 + cg1 even; H % 8 == 0; W == 64; wpack [(cg0+cg1)/2][2][parts*8][8][8] fp16 with row n = t*8 + r = tap 2t + r
 *   per dimension; bias: one float on the device; out [B][2D][2H][128] fp32, fully overwritten (a strided memset node + one kernel). */
int genre_b200_convt_c1_col2im_forward(const void *src0, int cg0, const void *src1, int cg1, int64_t B, int64_t D, int64_t H,
                                       int64_t W, const void *wpack, int op, const float *bias, float *out, void *stream);

/* ConvTranspose3d(Cin -> 1, kernel 4, stride 2, padding 1) forward on channel-blocked fp32 inputs (FP32 pipe: with one
 * output channel there is no GEMM for the tensor cores).  Replaces the cuDNN call behind the last layer of each decoder:
 * Unet_3D.dec6 (networks/networks.py:167-168, two sources = the skip concatenation), VoxelDecoder main.17 (:57),
 * VoxelGenerator (:98).   weight [Cin][64] = the module's [Cin,1,4,4,4];  out [B][2D][2H][2W] (NCDHW, C = 1). */
int genre_b200_convt_c1_forward(const float *src0, int cg0, const float *src1, int cg1,
                                int64_t B, int64_t D, int64_t H, int64_t W,
                                const float *weight, float bias, int act_sigmoid, float *out, void *stream);

/* ConvTranspose3d(k 8, s 2, p 3), Cout <= 20, with the four (y,x) output parity classes merged along N (one N = 80 MMA
 * over the union of 5x5 taps instead of four N = 20 MMAs over 4x4): Unet_3D.dec5 = ConvT(80 -> 20) (networks/networks.py:166),
 * 53.7 of the refiner's 78 GFLOP.  Operands as genre_b200_convt3d_s2_forward except wpack
 * [2 z-parity][4][Cin chunk][25][2][npad/8][8][g] with npad = 80 columns n = (py*2+px)*20 + co; scale, shift [20]. */
int genre_b200_convt3d_s2_merged_forward(const void *src0, int cg0, const void *src1, int cg1,
                                         int64_t B, int64_t D, int64_t H, int64_t W,
                                         const void *wpack, int ksize, int npad, int f16,
                                         const float *scale, const float *shift, float slope,
                                         float *out, int cgo, void *stream);

/* Conv3d(k 8, s 2, p 3), Cout <= 20, as a 3-tap stride-1 convolution over the 4x space-to-depth input whose N = 160
 * columns are the 8 output classes of the 2x finer output grid: Unet_3D.enc1 = Conv3d(2 -> 20) on 128^3
 * (networks/networks.py:151).  src [B*D][cg][H][W][16 B] with D,H,W = input extent / 4 (genre_b200_ncdhw_to_blocked
 * mode 3); wpack [3][chunk][9][2][20][8][g]; scale, shift [20]; out [B*2D][cgo][2H][2W][4] fp32.  W,H % 16 == 0. */
int genre_b200_conv3d_k8s2_s4d_forward(const void *src, int cg, int64_t B, int64_t D, int64_t H, int64_t W,
                                       const void *wpack, int npad, int f16,
                                       const float *scale, const float *shift, float slope,
                                       float *out, int cgo, void *stream);

/* ConvTranspose3d(Cin -> 1, k 4, s 2, p 1) on the tensor cores: 3 union taps per dimension, the 8 output classes as
 * N columns, bias [1] (device) and optional sigmoid in the epilogue, NCDHW fp32 output [B][2D][2H][2W].  Same layers
 * as genre_b200_convt_c1_forward (the FP32-pipe variant); wpack [3][chunk][9][2][2][8][g].  W in {16,32,64}. */
int genre_b200_convt_c1_tc_forward(const void *src0, int cg0, const void *src1, int cg1,
                                   int64_t B, int64_t D, int64_t H, int64_t W,
                                   const void *wpack, int f16, const float *bias, int act_sigmoid,
                                   float *out, void *stream);

/* Backward of ConvTranspose3d(Cin -> 1, k 4, s 2, p 1) (Unet_3D.dec6 networks/networks.py:167-168 and the decoders' last
 * layers): cuDNN answers the weight gradient of this 1-channel layer with a grouped direct kernel that takes 40.7 ms of
 * a 60 ms Unet_3D training step at B=4 (profiles/r01_train_unet_launches.csv).
 *   wgrad: x [B][Cin][D][H][W], gy [B][1][2D][2H][2W] -> dW [Cin][1][4][4][4]; deterministic (fixed-order reduction of
 *          per-CTA partials in `workspace`, genre_b200_convt_c1_wgrad_workspace_bytes(Cin) bytes); Cin <= 64, H % 8 == 0.
 *   dgrad: gy, weight -> dx [B][Cin][D][H][W]; Cin <= 192, H % 8 == 0. */
size_t genre_b200_convt_c1_wgrad_workspace_bytes(int cin);
int genre_b200_convt_c1_wgrad(const float *x, const float *gy, int64_t B, int64_t Cin, int64_t D, int64_t H, int64_t W,
                              float *dW, void *workspace, size_t workspace_bytes, void *stream);
int genre_b200_convt_c1_dgrad(const float *gy, const float *weight, int64_t B, int64_t Cin, int64_t D, int64_t H, int64_t W,
                              float *dx, void *stream);

/* Weight gradient of Conv3d(Cin <= 2 -> Cout <= 20, k 8, s 2, p 3) = Unet_3D.enc1 (networks/networks.py:151): the
 * cuDNN kernel for it (wgrad2d_grouped_direct_kernel) is 40.7 ms of a 60 ms Unet_3D training step at B=4.
 * x [B][Cin][D][H][W], gy [B][Cout][D/2][H/2][W/2] -> dW [Cout][Cin][8][8][8]; deterministic; H % 16 == 0, W <= 128. */
size_t genre_b200_conv_k8s2_wgrad_workspace_bytes(void);
int genre_b200_conv_k8s2_wgrad(const float *x, const float *gy, int64_t B, int64_t Cin, int64_t Cout,
                               int64_t D, int64_t H, int64_t W, float *dW,
                               void *workspace, size_t workspace_bytes, void *stream);

/* BatchNorm3d with BATCH statistics (training) fused with its ReLU / LeakyReLU, forward and backward, NCDHW fp32:
 * nn.BatchNorm3d + nn.LeakyReLU of Conv3d_block / Deconv3d_skip (networks/networks.py:193-222) and the BatchNorm3d + ReLU of
 * the decoders' stacks (:40-57) while training (cuDNN: 5.3 ms of a 22 ms Unet_3D step for ~0.3 ms worth of HBM traffic).
 * x, y, dy, dx [B][C][S] contiguous and 16-byte aligned, S = D*H*W a multiple of 4; gamma / beta / running_* [C] or NULL;
 * slope: 1 = no activation, 0 = ReLU; two-pass variance, fixed-order reductions (bitwise reproducible).
 * OPT-IN (GENRE_B200_BN_TRAIN=1): written after round 1's GPU budget was spent, not yet run on a GPU. */
size_t genre_b200_bn_workspace_bytes(int64_t C);
int genre_b200_bn_act_train_forward(const float *x, int64_t B, int64_t C, int64_t S,
                                    const float *gamma, const float *beta, float *running_mean, float *running_var,
                                    float eps, float momentum, float slope,
                                    float *y, float *save_mean, float *save_invstd,
                                    void *workspace, size_t workspace_bytes, void *stream);
int genre_b200_bn_act_train_backward(const float *x, const float *dy, int64_t B, int64_t C, int64_t S,
                                     const float *gamma, const float *beta, const float *save_mean, const float *save_invstd,
                                     float slope, float *dx, float *dgamma, float *dbeta,
                                     void *workspace, size_t workspace_bytes, void *stream);

/* Layout boundary of the convolution kernels: contiguous NCDHW fp32 (what networks/networks.py's modules exchange,
 * e.g. Unet_3D.forward networks.py:170-190) <-> channel-blocked [B*D][C/g][H][W][g] (16 bytes per unit).
 *   mode 0: plain;  mode 1: space-to-depth, channel = ((c*2+pz)*2+py)*2+px (Conv3d k8 s2, Unet_3D.enc1; with cpad > 8C the
 *           channel axis is zero-padded to cpad channels: Conv3d(1 -> 64, k4 s2), VoxelDiscriminator's first layer);
 *   mode 2: the 8 parity sub-volumes one after the other, each padded to cpad channels (Conv3d k4 s2);
 *   mode 3: 4x space-to-depth, channel = ((c*4+rz)*4+ry)*4+rx (Conv3d k8 s2 as a 3-tap convolution, Unet_3D.enc1).
 *   group 4: fp32 units, group 8: fp16 units (cast on the way).  One pass, 16-byte stores. */
int genre_b200_ncdhw_to_blocked(const float *src, int64_t B, int64_t C, int64_t D, int64_t H, int64_t W,
                                int mode, int group, int cpad, void *dst, void *stream);

/* blocked fp32 [B*D][cg][H][W][4] -> contiguous NCDHW [B,C,D,H,W], 4*(cg-1) < C <= 4*cg (channel padding dropped) */
int genre_b200_blocked_to_ncdhw(const float *src, int cg, int64_t B, int64_t C, int64_t D, int64_t H, int64_t W,
                                float *dst, void *stream);

/* ---- fused GenRe glue (SURVEY 8f-1; opt-in, inference only; genre_shapehd_b200/fused.py) --------------------------
 * The frozen callers wrap the ops in ~19 dense elementwise passes over 128^3 volumes (depth_pred_with_sph_inpaint.py:
 * 120-126, genre_full_model.py:120-143).  These three entry points fold them into the kernels. */

/* render_spherical over clamp(vox * pre_scale, pre_lo, pre_hi) applied as each voxel is fetched
 * (`render_spherical(torch.clamp(proj * 50, 1e-5, 1 - 1e-5))`, depth_pred_with_sph_inpaint.py:124). */
int genre_b200_render_spherical_forward_pre(const float *vox, int64_t N, int res, const double *dirs,
                                            int sph_res, int z_res, const float *depth_weight,
                                            float pre_scale, float pre_lo, float pre_hi, float *out, void *stream);

/* The spherical renderer with EMPTY-SPACE SKIPPING (forward): same contract and results (within ~1e-6) as
 * genre_b200_render_spherical_forward / _forward_pre (use_pre != 0 renders clamp(vox * pre_scale, pre_lo, pre_hi)).
 * A pre-pass marks the 8^3 bricks that hold a voxel > 1e-5 (dilated by one voxel); along each ray, 32-sample chunks that
 * only touch unmarked bricks (every sample clamps to p = 1e-5, spherical_proj.py:66) are advanced in closed form instead
 * of 32 x 8 gathers.  GenRe's input is a thin shell: ~80 % of the chunks.  workspace: caller-owned,
 * genre_b200_render_spherical_workspace_bytes(N, res) bytes (zeroed by the call).  Falls back to the plain kernels when
 * res % 4 != 0 or z_res > 1024. */
size_t genre_b200_render_spherical_workspace_bytes(int64_t N, int res);
int genre_b200_render_spherical_forward_skip(const float *vox, int64_t N, int res, const double *dirs, int sph_res,
                                             int z_res, const float *depth_weight, int use_pre, float pre_scale,
                                             float pre_lo, float pre_hi, float *out, void *workspace,
                                             size_t workspace_bytes, void *stream);

/* Net.backproject_spherical (genre_full_model.py:134-143) in one call: radius = in_bias + in_scale * sph (the
 * `1 - crop_sph`; the crop is expressed through the strides), out = 1 - R * mean distance on hit voxels and 0
 * elsewhere (= (-tdf + 1/R) * R * clamp(cnt,0,1)), maps written out_map_stride floats apart (a channel of the
 * refiner's [B,2,R,R,R] input).  Workspace as genre_b200_sph_bp_forward. */
int genre_b200_sph_bp_forward_fused(const float *sph, int64_t N, int64_t C, int64_t H, int64_t W,
                                    int64_t sN, int64_t sC, int64_t sH, int64_t sW,
                                    const float *grid, int64_t gN, int64_t gC, int64_t gH, int64_t gW, int64_t gD,
                                    float in_scale, float in_bias, float *out, int64_t out_map_stride, int res,
                                    void *workspace, size_t workspace_bytes, void *stream);

/* dst[m][:] = clamp(src[m][:] * scale, lo, hi), dst maps dst_map_stride floats apart
 * (`torch.clamp(proj_depth / 50, 1e-5, 1 - 1e-5)` + torch.cat, genre_full_model.py:126-127). */
int genre_b200_scale_clamp_strided(const float *src, int64_t maps, int64_t n, float scale, float lo, float hi,
                                   float *dst, int64_t dst_map_stride, void *stream);

/* blocked fp32 [BD][cg4][H][W][4] -> blocked fp16 [BD][(cg4+1)/2][H][W][8], channel padding zero-filled: turns the
 * fp32 output of one tensor-core layer into the fp16 operand of the next without going through NCDHW */
int genre_b200_blocked_f32_to_f16(const float *src, int cg4, int64_t BD, int64_t H, int64_t W, void *dst, void *stream);

/* blocked fp32 [BD][cg4][H][W][4] -> fp16 [BD][2 parts][(cg4+1)/2][H][W][8]: part 0 = hi = fp16(a), part 1 = lo' =
 * fp16((a - hi) * 2^11).  The activation operand of the conv kernels' op = 2 ("f16x2") mode: the fp32-accurate replacement of
 * the reference's fp32 cuDNN convolutions (networks/networks.py:197-218) at 2 tensor-core MMAs per K step
 * (A_hi x [W_hi | W_lo'] and A_lo' x W_hi; weights packed [W_hi | W_lo'] along N by ops_conv._pack).  In that mode every
 * conv entry point above takes per-part channel-group counts and `f16` = 2. */
int genre_b200_blocked_split2_f16(const float *src, int cg4, int64_t BD, int64_t H, int64_t W, void *dst, void *stream);

/* blocked fp32 [BD][cg][H][W][4] -> [BD][3*cg][H][W][4] = (lo | hi | hi): hi = value rounded to TF32, lo = value - hi.
 * With weights packed as (W_hi | W_lo | W_hi) along K, the TF32 tensor-core kernels above compute
 * A_lo*W_hi + A_hi*W_lo + A_hi*W_hi = the fp32 product to ~2^-21 relative (small terms first: the tensor core's
 * fp32 accumulator truncates, ~2^-26 of the partial sum per MMA step) ("3xTF32"): the mode the 3D nets run in when
 * torch.backends.cudnn.allow_tf32 is off, so that occupancies match the fp32 reference within 1e-4. */
int genre_b200_blocked_split3(const float *src, int cg, int64_t BD, int64_t H, int64_t W, float *dst, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Ground-truth surface voxels (SURVEY 8f-3).  Replaces the per-sample CPU code of Model.preprocess
 * (models/genre_full_model.py:86-96, scipy.ndimage.binary_erosion inside DataLoader workers):
 *     val  = flip(transpose(voxel, (0,2,1)), 2)                      (transpose_flip != 0; :89-90)
 *     out  = clip(val - binary_erosion(val != 0, ones((3,3,3)), iterations), 0, 1)   (:91-93, border value 0)
 *   vox, out [N, R, R, R] dense fp32, distinct buffers; R a multiple of 32, at most 256; 1 <= iterations <= 15
 *   workspace: genre_b200_voxel_surface_workspace_bytes(N, R) bytes (one bit per voxel), caller-owned
 * Bit-exact against scipy (tests/test_gpu_toolbox.py).
 * ------------------------------------------------------------------------------------------- */
size_t genre_b200_voxel_surface_workspace_bytes(int64_t N, int res);
int genre_b200_voxel_surface(const float *vox, int64_t N, int res, int iterations, int transpose_flip, float *out,
                             void *workspace, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Batched marching cubes (the mesh export of the reference's visualiser).  Replaces the per-sample CPU
 * call of Visualizer._save_iso_obj (visualize/visualizer.py:153-166: skimage.measure.marching_cubes_lewiner
 * in a process pool) for a whole batch on the device.  The case table is genre_shapehd_b200/csrc/mc_table.h,
 * generated from a rule by gen_mc_table.py: ambiguous faces cut off each in-corner, cube-interior
 * ambiguities are not resolved (no MC33), so in ambiguous cells the triangles and the topology can differ
 * from Lewiner's; the vertices are the same iso-crossings of grid edges.
 *
 *   vol     [N, D, H, W] dense fp32; 1 <= N <= 65535, D, H >= 2, 2 <= W <= 256, 3*D*H*W and 5*(D-1)(H-1)(W-1)
 *           within int32.  A voxel is inside when value > level (NaN: outside).
 *   workspace: genre_b200_iso_surface_workspace_bytes(N, D, H, W) bytes, 16-byte aligned, caller-owned
 *           (1 bit per voxel + 16 bytes per z row); emit reads what count wrote there, so the two calls must
 *           share the workspace, the volume and the level, in stream order.
 *
 * _count: per-sample totals[N][2] int64 = (vertices, triangles), written on the device (the caller reads
 *           them back to size the mesh buffers).  3 kernels.
 * _emit:  bases[N][2] int64 = where each sample's vertices / triangles start in verts / faces (usually the
 *           exclusive prefix sum of totals); verts [sum V, 3] fp32, faces [sum F, 3] int32 with indices local
 *           to the sample, values [sum V] fp32 or NULL.  1 kernel.
 *   Order (a contract: the output is deterministic and equal bit for bit to the oracle): one vertex per
 *   crossed grid edge p -> p + e_a, sorted by the C-order index of p, then by a; faces sorted by cell
 *   (C order), then by triangle index in the table.  Each operation rounds once:
 *       t       = (level - f(p)) / (f(p + e_a) - f(p))
 *       coord_a = (p_a + t) * s_a + o_a,   coord_b = p_b * s_b + o_b   (b != a)
 *   with (s, o) = (sx, ox) for array axis 0 (D), (sy, oy) for axis 1 (H), (sz, oz) for axis 2 (W);
 *   values = max(f(p), f(p + e_a)).  Triangle normals (right hand) point from the > level side to the
 *   <= level side.
 * ------------------------------------------------------------------------------------------- */
size_t genre_b200_iso_surface_workspace_bytes(int64_t N, int D, int H, int W);
int genre_b200_iso_surface_count(const float *vol, int64_t N, int D, int H, int W, float level, void *workspace,
                                 size_t workspace_bytes, int64_t *totals, void *stream);
int genre_b200_iso_surface_emit(const float *vol, int64_t N, int D, int H, int W, float level, float sx, float sy,
                                float sz, float ox, float oy, float oz, const int64_t *bases, float *verts, int *faces,
                                float *values, void *workspace, size_t workspace_bytes, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* GENRE_B200_H */
