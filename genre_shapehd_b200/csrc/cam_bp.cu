// cam_bp.cu — camera back-projection (depth -> voxel TDF), its backward, and the surface mask.
//
// Reference: toolbox/cam_bp/cam_bp/src/back_projection_kernel.cu
//   forward  kernel :199-276 + inplace_safe_divide :281-306 + wrap :760-838
//   backward kernel :365-471 + wrap :897-963
//   surface mask    :309-358 + wrap :840-891
//
// Bit-exactness of the voxel index: every fp32 operation below is written with an explicit
// round-to-nearest intrinsic in the order nvcc 12.9 emits for the reference source when it is built
// with its own flags (default --fmad=true, IEEE div/sqrt; toolbox/cam_bp/setup.sh:25-29), read off
// the sm_100a SASS of oracle/_ref/libref_cam_bp.so:
//     imind   = fma(size-1, -0.5, idx)                      (exact for image sizes < 2^23)
//     norm^2  = fma(fl, fl, fma(imind_w, imind_w, imind_h*imind_h))
//     cos     = fl / sqrt(norm^2)                           (IEEE sqrt, IEEE div)
//     z       = depth * cos
//     gy, gz  = (imind_{w,h} * -z) / fl ;  gx = z - cam_dist
//     index   = FLOOR_I((g + 0.5) * R)                       (add, mul, trunc; no contraction possible)
//     centre  = ((float)index + 0.5) / R - 0.5
//     dist^2  = fma(dz, dz, fma(dx, dx, dy*dy))
// Intrinsics are never contracted by the compiler, so this file does not depend on -fmad.
#include "voxelize.cuh"

namespace gb {

struct CamPoint {
  float gx, gy, gz;      // point in the unit cube frame
  float imh, imw;        // centred pixel coordinates
  float norm;            // |(imh, imw, fl)|
  int ix, iy, iz;        // voxel index
  bool in_bounds;
};

// shared by forward and backward: pixel (h, w) with ray depth d -> point and voxel index
__device__ __forceinline__ CamPoint cam_unproject(float d, float fl, const ExactDivisor &dfl, float cam_dist, int h,
                                                  int w, float Hm1, float Wm1, int R, float Rf) {
  CamPoint p;
  p.imh = __fmaf_rn(Hm1, -0.5f, (float)h);
  p.imw = __fmaf_rn(Wm1, -0.5f, (float)w);
  const float n2 = __fmaf_rn(fl, fl, __fmaf_rn(p.imw, p.imw, __fmul_rn(p.imh, p.imh)));
  p.norm = __fsqrt_rn(n2);
  const float cos_theta = __fdiv_rn(fl, p.norm);
  const float z = __fmul_rn(d, cos_theta);
  p.gy = div_exact(__fmul_rn(p.imw, -z), dfl);
  p.gz = div_exact(__fmul_rn(p.imh, -z), dfl);
  p.gx = __fadd_rn(z, -cam_dist);
  p.ix = floor_i_ref(__fmul_rn(__fadd_rn(p.gx, 0.5f), Rf));
  p.iy = floor_i_ref(__fmul_rn(__fadd_rn(p.gy, 0.5f), Rf));
  p.iz = floor_i_ref(__fmul_rn(__fadd_rn(p.gz, 0.5f), Rf));
  p.in_bounds = (p.ix >= 0) & (p.ix < R) & (p.iy >= 0) & (p.iy < R) & (p.iz >= 0) & (p.iz < R);
  return p;
}

// ------------------------------------------------------------------------------------------------
// project: PROJ_PIX pixels per thread (independent loads and tickets in flight), 1024 pixels per CTA
// ------------------------------------------------------------------------------------------------
constexpr int PROJ_THREADS = 256;
constexpr int PROJ_PIX = 4;

// Offsets inside one depth map are 32-bit (checked on the host); only the per-map base is 64-bit.
struct CamProjArgs {
  const float *depth;
  int C, H, W;
  long long sN, sC;
  int sH, sW;
  const float *fl_in;
  long long fN, fC;
  const float *cd_in;
  long long dN, dC;
  int R;
  float qscale;
  VoxWorkspace ws;
  int fast_shift;
};

// the project stage of one CTA: pixels [bx * 1024, bx * 1024 + 1024) of map `map`
template <bool W_FAST>
__device__ __forceinline__ void cam_project_body(const CamProjArgs &a, int bx, int map, unsigned *s_hist) {
  const float *__restrict__ depth = a.depth;
  const float *__restrict__ fl_in = a.fl_in;
  const float *__restrict__ cd_in = a.cd_in;
  const int C = a.C, H = a.H, W = a.W, sH = a.sH, sW = a.sW, R = a.R, fast_shift = a.fast_shift;
  const long long sN = a.sN, sC = a.sC, fN = a.fN, fC = a.fC, dN = a.dN, dC = a.dC;
  const float qscale = a.qscale;
  const VoxWorkspace &ws = a.ws;
  int n = map, c = 0;
  if (C != 1) {
    n = map / C;
    c = map - n * C;
  }
  const int P = H * W;
  const float *dmap = depth + n * sN + c * sC;
  const float fl = fl_in[n * fN + c * fC];
  const float cam_dist = cd_in[n * dN + c * dC];
  const ExactDivisor dfl = make_divisor(fl);
  const VoxGrid grid = make_grid(R);
  const float Hm1 = __fadd_rn((float)H, -1.0f), Wm1 = __fadd_rn((float)W, -1.0f);
  const int fast = W_FAST ? W : H;  // extent of the axis consecutive threads walk along

  // A pixel with depth exactly 0 (GenRe's background, depth_pred_with_sph_inpaint.py:139) unprojects to
  // (-cam_dist, -+0, -+0) whatever its position: z = 0 * cos = 0, gy = (w~ * -0) / fl = -+0.  Whether that point is
  // inside the grid is therefore a property of the map, evaluated once with the same operations; when it is
  // outside (any camera further than 0.5 from the origin) such pixels skip the whole unprojection.
  bool zero_in_bounds;
  {
    const int ix0 = floor_i_ref(__fmul_rn(__fadd_rn(__fadd_rn(0.0f, -cam_dist), 0.5f), grid.Rf));
    const int iyz0 = floor_i_ref(__fmul_rn(0.5f, grid.Rf));
    zero_in_bounds = (ix0 >= 0) & (ix0 < R) & (iyz0 >= 0) & (iyz0 < R);
    const float afl = fabsf(fl);
    if (!(afl >= 0x1p-40f && afl <= 0x1p40f)) zero_in_bounds = true;  // degenerate focal length: no shortcut
  }

  const int p0 = bx * (PROJ_THREADS * PROJ_PIX) + threadIdx.x;
  auto coords = [&](int p, int &h, int &w) {
    const int slow = fast_shift >= 0 ? (p >> fast_shift) : (p / fast);
    const int fst = p - slow * fast;
    h = W_FAST ? slow : fst;
    w = W_FAST ? fst : slow;
  };
  float d[PROJ_PIX];
#pragma unroll
  for (int k = 0; k < PROJ_PIX; ++k) {
    const int p = p0 + k * PROJ_THREADS;
    int h, w;
    coords(p, h, w);
    d[k] = (p < P) ? __ldg(dmap + (h * sH + w * sW)) : -1.0f;
  }
  unsigned gv[PROJ_PIX], q[PROJ_PIX];
#pragma unroll
  for (int k = 0; k < PROJ_PIX; ++k) {
    gv[k] = VOX_INVALID;
    q[k] = 0;
    // reference skips only d < 0 (back_projection_kernel.cu:225)
    if (!(d[k] < 0.0f) && (zero_in_bounds || d[k] != 0.0f)) {
      int h, w;
      coords(p0 + k * PROJ_THREADS, h, w);
      const CamPoint pt = cam_unproject(d[k], fl, dfl, cam_dist, h, w, Hm1, Wm1, R, grid.Rf);
      if (pt.in_bounds) {
        const float dx = __fadd_rn(pt.gx, -vox_centre(pt.ix, grid));
        const float dy = __fadd_rn(pt.gy, -vox_centre(pt.iy, grid));
        const float dz = __fadd_rn(pt.gz, -vox_centre(pt.iz, grid));
        const float dist = __fsqrt_rn(__fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy))));
        gv[k] = (unsigned)((pt.ix * R + pt.iy) * R + pt.iz);
        q[k] = vox_quantise(dist, qscale);
      }
    }
  }
  vox_emit<PROJ_PIX, PROJ_THREADS>(gv, q, map, ws, P, s_hist);
}

template <bool W_FAST>
__global__ void __launch_bounds__(PROJ_THREADS)
cam_project_kernel(const CamProjArgs a) {
  extern __shared__ unsigned s_hist[];  // [ntiles] CTA-local tile histogram
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // let the splat grid start launching behind us
  cam_project_body<W_FAST>(a, blockIdx.x, blockIdx.y, s_hist);
}

static int cam_check(const float *depth, int64_t N, int64_t C, int64_t H, int64_t W, const float *fl,
                     const float *camdist, int res) {
  GB_REQUIRE(depth && fl && camdist, GENRE_B200_EINVAL, "cam_bp: null input pointer");
  GB_REQUIRE(N > 0 && C > 0 && H > 0 && W > 0, GENRE_B200_EINVAL, "cam_bp: empty depth tensor [%lld,%lld,%lld,%lld]",
             (long long)N, (long long)C, (long long)H, (long long)W);
  GB_REQUIRE(H < (1 << 20) && W < (1 << 20), GENRE_B200_EINVAL, "cam_bp: image too large");
  return vox_check_common(N * C, H * W, res);
}

// offsets inside one map must fit 32 bits (the kernels add them to a 64-bit per-map base)
static bool map_offsets_fit(int64_t H, int64_t W, int64_t sH, int64_t sW) {
  const long double span = (long double)(H - 1) * (long double)llabs(sH) + (long double)(W - 1) * (long double)llabs(sW);
  return span < 2147483647.0L;
}

static inline int log2_exact(int64_t v) {
  if (v <= 0 || (v & (v - 1))) return -1;
  int s = 0;
  while ((1ll << s) < v) ++s;
  return s;
}

static int cam_proj_args(const float *depth, int64_t N, int64_t C, int64_t H, int64_t W, int64_t sN, int64_t sC, int64_t sH,
                         int64_t sW, const float *fl, int64_t fN, int64_t fC, const float *camdist, int64_t dN, int64_t dC,
                         int res, const VoxWorkspace &w, CamProjArgs *a, bool *w_fast) {
  GB_REQUIRE(map_offsets_fit(H, W, sH, sW), GENRE_B200_EINVAL, "cam_bp: depth strides too large");
  *w_fast = llabs(sW) <= llabs(sH);  // map consecutive threads to the denser image axis
  a->depth = depth; a->C = (int)C; a->H = (int)H; a->W = (int)W; a->sN = sN; a->sC = sC; a->sH = (int)sH; a->sW = (int)sW;
  a->fl_in = fl; a->fN = fN; a->fC = fC; a->cd_in = camdist; a->dN = dN; a->dC = dC; a->R = res;
  a->qscale = (float)res * 16777216.0f;
  a->ws = w;
  a->fast_shift = log2_exact(*w_fast ? W : H);
  return 0;
}

static inline int cam_proj_ctas_per_map(int64_t P) {
  const int per_cta = PROJ_THREADS * PROJ_PIX;
  return (int)((P + per_cta - 1) / per_cta);
}

static int cam_project_launch(const float *depth, int64_t N, int64_t C, int64_t H, int64_t W, int64_t sN, int64_t sC,
                              int64_t sH, int64_t sW, const float *fl, int64_t fN, int64_t fC, const float *camdist,
                              int64_t dN, int64_t dC, int res, const VoxWorkspace &w, cudaStream_t st) {
  CamProjArgs a;
  bool w_fast = true;
  if (int rc = cam_proj_args(depth, N, C, H, W, sN, sC, sH, sW, fl, fN, fC, camdist, dN, dC, res, w, &a, &w_fast)) return rc;
  dim3 grid((unsigned)cam_proj_ctas_per_map(H * W), (unsigned)(N * C));
  const size_t smem = (size_t)w.ntiles * 4;
  if (w_fast) cam_project_kernel<true><<<grid, PROJ_THREADS, smem, st>>>(a);
  else cam_project_kernel<false><<<grid, PROJ_THREADS, smem, st>>>(a);
  return check_launch("cam_bp project kernel");
}

// ------------------------------------------------------------------------------------------------
// backward: one thread per pixel, gathers cnt / grad at its voxel
// (reference :365-471; cam_dist read with its own strides, not the :401 stride mix-up)
// ------------------------------------------------------------------------------------------------
constexpr int BWD_THREADS = 256;

__global__ void __launch_bounds__(BWD_THREADS)
cam_bp_backward_kernel(const float *__restrict__ depth, int C, int H, int W, long long sN, long long sC, long long sH,
                       long long sW, const float *__restrict__ fl_in, long long fN, long long fC,
                       const float *__restrict__ cd_in, long long dN, long long dC, const float *__restrict__ cnt,
                       const float *__restrict__ grad_tdf, int R, float *__restrict__ grad_depth,
                       float *__restrict__ grad_fl, float *__restrict__ grad_cd) {
  const int map = blockIdx.y;
  const int n = map / C, c = map - n * C;
  const int P = H * W;
  const int p = blockIdx.x * BWD_THREADS + threadIdx.x;  // dense grad_depth index: h * W + w
  float g_depth = 0.0f, g_fl = 0.0f, g_cd = 0.0f;
  if (p < P) {
    const int h = p / W, w = p - h * W;
    const float d = depth[n * sN + c * sC + h * sH + w * sW];
    if (!(d < 0.0f)) {
      const float fl = fl_in[n * fN + c * fC];
      const float cam_dist = cd_in[n * dN + c * dC];
      const float Rf = (float)R;
      const CamPoint pt = cam_unproject(d, fl, make_divisor(fl), cam_dist, h, w, __fadd_rn((float)H, -1.0f),
                                        __fadd_rn((float)W, -1.0f), R, Rf);
      if (pt.in_bounds) {
        // voxel centre: the reference's backward evaluates this in double (literals 0.5), :428-430
        const float cx = (float)((((double)(float)pt.ix + 0.5) / (double)Rf) - 0.5);
        const float cy = (float)((((double)(float)pt.iy + 0.5) / (double)Rf) - 0.5);
        const float cz = (float)((((double)(float)pt.iz + 0.5) / (double)Rf) - 0.5);
        float len = pt.norm;
        if ((double)len < 1e-5) len = 1e-5f;
        const float dirx = -fl / len, diry = pt.imw / len, dirz = pt.imh / len;
        const float ex = pt.gx - cx, ey = pt.gy - cy, ez = pt.gz - cz;
        float vlen = sqrtf(ex * ex + ey * ey + ez * ez);
        if ((double)vlen < 1e-5) vlen = 1e-5f;
        const float ux = ex / vlen, uy = ey / vlen, uz = ez / vlen;
        const float cos_cc = dirx * ux + diry * uy + dirz * uz;
        const size_t v = (size_t)map * R * R * R + ((size_t)pt.ix * R + pt.iy) * R + pt.iz;
        float ptnum = cnt[v];
        if (ptnum < 1.0f) ptnum = 1.0f;
        const float gd = grad_tdf[v];
        g_depth = -gd * cos_cc / ptnum;
        const float len3 = len * len * len;
        const float gfx = ux * (pt.imw * pt.imw + pt.imh * pt.imh) / len3;
        const float gfy = uy * (pt.imw * fl) / len3;
        const float gfz = uz * (pt.imh * fl) / len3;
        g_fl = (gfx + gfy + gfz) * gd * d / ptnum;
        g_cd = -ux * gd / ptnum;
      }
    }
    grad_depth[(size_t)map * P + p] = g_depth;
  }
  // block reduction of the two per-map scalars, then one atomic per CTA (reference: one per pixel, :464,469)
  __shared__ float s_fl[BWD_THREADS / 32], s_cd[BWD_THREADS / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    g_fl += __shfl_xor_sync(0xffffffffu, g_fl, o);
    g_cd += __shfl_xor_sync(0xffffffffu, g_cd, o);
  }
  if ((threadIdx.x & 31) == 0) { s_fl[threadIdx.x >> 5] = g_fl; s_cd[threadIdx.x >> 5] = g_cd; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, b = 0.f;
    for (int i = 0; i < BWD_THREADS / 32; ++i) { a += s_fl[i]; b += s_cd[i]; }
    if (a != 0.0f) atomicAdd(grad_fl + map, a);
    if (b != 0.0f) atomicAdd(grad_cd + map, b);
  }
}

// ------------------------------------------------------------------------------------------------
// surface mask: one thread per 4 consecutive voxels (reference :309-358, one voxel per thread, batch-fastest)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int floor_i_ref_d(double a) { return a < 0 ? (int)a - 1 : (int)a; }
// ROUND_I of the reference (:42-43) applied to a double argument
__device__ __forceinline__ int round_i_ref_d(double a) {
  const int fi = floor_i_ref_d(a);
  const float ff = (float)fi;
  return (a - ff > ff + 1.0 - a) ? fi + 1 : fi;
}

__device__ __forceinline__ float surface_mask_one(const float *__restrict__ dmap, int H, int W, long long sH,
                                                  long long sW, float fl, float cam_dist, float ptnum, int ix, int iy,
                                                  int iz, float Rf) {
  if ((double)ptnum > 1e-5) return 1.0f;
  const float cx = (float)((((double)(float)ix + 0.5) / (double)Rf) - 0.5);
  const float cy = (float)((((double)(float)iy + 0.5) / (double)Rf) - 0.5);
  const float cz = (float)((((double)(float)iz + 0.5) / (double)Rf) - 0.5);
  const float den = __fadd_rn(cx, cam_dist);
  const float im_h = __fdiv_rn(__fmul_rn(-cz, fl), den);
  const float im_w = __fdiv_rn(__fmul_rn(-cy, fl), den);
  const int idh = round_i_ref_d(__dadd_rn(__dmul_rn(0.5, (double)(float)H - 1.0), (double)im_h));
  const int idw = round_i_ref_d(__dadd_rn(__dmul_rn(0.5, (double)(float)W - 1.0), (double)im_w));
  if (idh < 0 || idh >= H || idw < 0 || idw >= W) return 1.0f;
  const float d = dmap[idh * sH + idw * sW];
  if (d < 0.0f) return 1.0f;
  const float ray = __fsqrt_rn(__fmaf_rn(cz, cz, __fmaf_rn(cy, cy, __fmul_rn(den, den))));
  return (d < ray) ? 0.0f : 1.0f;
}

__global__ void __launch_bounds__(256)
surface_mask_kernel(const float *__restrict__ depth, int C, int H, int W, long long sN, long long sC, long long sH,
                    long long sW, const float *__restrict__ fl_in, long long fN, long long fC,
                    const float *__restrict__ cd_in, long long dN, long long dC, const float *__restrict__ cnt,
                    float *__restrict__ mask, int R, long long nvox, bool vec) {
  const int map = blockIdx.y;
  const int n = map / C, c = map - n * C;
  const float fl = fl_in[n * fN + c * fC], cam_dist = cd_in[n * dN + c * dC];
  const float *dmap = depth + n * sN + c * sC;
  const float *cmap = cnt + (size_t)map * nvox;
  float *mmap = mask + (size_t)map * nvox;
  const float Rf = (float)R;
  const long long stride = (long long)gridDim.x * blockDim.x;
  if (vec) {
    for (long long v4 = blockIdx.x * (long long)blockDim.x + threadIdx.x; v4 * 4 < nvox; v4 += stride) {
      const long long v = v4 * 4;
      const float4 cn = *reinterpret_cast<const float4 *>(cmap + v);
      const int iz = (int)(v % R), iy = (int)((v / R) % R), ix = (int)(v / ((long long)R * R));
      // R % 4 == 0 on this path, so the four voxels share (ix, iy)
      float4 m;
      m.x = surface_mask_one(dmap, H, W, sH, sW, fl, cam_dist, cn.x, ix, iy, iz + 0, Rf);
      m.y = surface_mask_one(dmap, H, W, sH, sW, fl, cam_dist, cn.y, ix, iy, iz + 1, Rf);
      m.z = surface_mask_one(dmap, H, W, sH, sW, fl, cam_dist, cn.z, ix, iy, iz + 2, Rf);
      m.w = surface_mask_one(dmap, H, W, sH, sW, fl, cam_dist, cn.w, ix, iy, iz + 3, Rf);
      st_stream_f4(mmap + v, m);
    }
  } else {
    for (long long v = blockIdx.x * (long long)blockDim.x + threadIdx.x; v < nvox; v += stride) {
      const int iz = (int)(v % R), iy = (int)((v / R) % R), ix = (int)(v / ((long long)R * R));
      mmap[v] = surface_mask_one(dmap, H, W, sH, sW, fl, cam_dist, cmap[v], ix, iy, iz, Rf);
    }
  }
}

}  // namespace gb

using namespace gb;

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" int genre_b200_cam_bp_stage_project(const float *depth, int64_t N, int64_t C, int64_t H, int64_t W,
                                               int64_t sN, int64_t sC, int64_t sH, int64_t sW, const float *fl,
                                               int64_t fN, int64_t fC, const float *camdist, int64_t dN, int64_t dC,
                                               int res, void *workspace, size_t workspace_bytes, void *stream) {
  if (int rc = cam_check(depth, N, C, H, W, fl, camdist, res)) return rc;
  VoxWorkspace w;
  GB_REQUIRE(vox_carve(workspace, workspace_bytes, N * C, H * W, res, &w), GENRE_B200_EWORKSPACE,
             "cam_bp: workspace too small or misaligned (need %zu bytes)", vox_workspace_bytes(N * C, H * W, res));
  cudaStream_t st = as_stream(stream);
  if (int rc = vox_clear_counts(w, N * C, st)) return rc;
  return cam_project_launch(depth, N, C, H, W, sN, sC, sH, sW, fl, fN, fC, camdist, dN, dC, res, w, st);
}

extern "C" int genre_b200_cam_bp_forward(const float *depth, int64_t N, int64_t C, int64_t H, int64_t W, int64_t sN,
                                         int64_t sC, int64_t sH, int64_t sW, const float *fl, int64_t fN, int64_t fC,
                                         const float *camdist, int64_t dN, int64_t dC, float *tdf, float *cnt, int res,
                                         unsigned flags, void *workspace, size_t workspace_bytes, void *stream) {
  if (int rc = cam_check(depth, N, C, H, W, fl, camdist, res)) return rc;
  GB_REQUIRE(tdf != nullptr, GENRE_B200_EINVAL, "cam_bp: tdf is null");
  GB_REQUIRE((flags & ~(unsigned)GENRE_B200_FLAG_SHIFT_TDF) == 0, GENRE_B200_EINVAL,
             "cam_bp: unknown flag bits 0x%x (only GENRE_B200_FLAG_SHIFT_TDF = 1 is defined)", flags & ~(unsigned)GENRE_B200_FLAG_SHIFT_TDF);
  VoxWorkspace w;
  GB_REQUIRE(vox_carve(workspace, workspace_bytes, N * C, H * W, res, &w), GENRE_B200_EWORKSPACE,
             "cam_bp: workspace too small or misaligned (need %zu bytes)", vox_workspace_bytes(N * C, H * W, res));
  cudaStream_t st = as_stream(stream);
  // sum_q / count is the mean distance in units of 2^-24 voxel edges.
  //   raw  : tdf = mean               , background 1/R (cam_back_projection.py:23-24 + kernel bias :304,:829)
  //   shift: tdf = 1 - R * mean       , background 1 - R * (1/R)   (camera_backprojection_module.py:26-28)
  const float inv_r = (float)(1.0 / (double)res);
  float alpha, beta, bg;
  if (flags & GENRE_B200_FLAG_SHIFT_TDF) {
    alpha = 1.0f;
    beta = -(1.0f / 16777216.0f);
    bg = 1.0f - (float)res * inv_r;
  } else {
    alpha = 0.0f;
    beta = (float)((1.0 / 16777216.0) / (double)res);
    bg = inv_r;
  }
  if (int rc = vox_clear_counts(w, N * C, st)) return rc;
  if (int rc = cam_project_launch(depth, N, C, H, W, sN, sC, sH, sW, fl, fN, fC, camdist, dN, dC, res, w, st)) return rc;
  return vox_splat(w, N * C, H * W, res, tdf, cnt, alpha, beta, bg, st);
}

extern "C" int genre_b200_cam_bp_backward(const float *depth, int64_t N, int64_t C, int64_t H, int64_t W, int64_t sN,
                                          int64_t sC, int64_t sH, int64_t sW, const float *fl, int64_t fN, int64_t fC,
                                          const float *camdist, int64_t dN, int64_t dC, const float *cnt,
                                          const float *grad_tdf, int res, float *grad_depth, float *grad_fl,
                                          float *grad_camdist, void *stream) {
  if (int rc = cam_check(depth, N, C, H, W, fl, camdist, res)) return rc;
  GB_REQUIRE(cnt && grad_tdf && grad_depth && grad_fl && grad_camdist, GENRE_B200_EINVAL,
             "cam_bp backward: null pointer");
  cudaStream_t st = as_stream(stream);
  cudaError_t e = cudaMemsetAsync(grad_fl, 0, (size_t)(N * C) * sizeof(float), st);
  if (e == cudaSuccess) e = cudaMemsetAsync(grad_camdist, 0, (size_t)(N * C) * sizeof(float), st);
  if (e != cudaSuccess) {
    set_error("cam_bp backward: memset: %s", cudaGetErrorString(e));
    return (int)e;
  }
  const int64_t P = H * W;
  dim3 grid((unsigned)((P + BWD_THREADS - 1) / BWD_THREADS), (unsigned)(N * C));
  cam_bp_backward_kernel<<<grid, BWD_THREADS, 0, st>>>(depth, (int)C, (int)H, (int)W, sN, sC, sH, sW, fl, fN, fC,
                                                       camdist, dN, dC, cnt, grad_tdf, res, grad_depth, grad_fl,
                                                       grad_camdist);
  return check_launch("cam_bp backward kernel");
}

extern "C" int genre_b200_surface_mask(const float *depth, int64_t N, int64_t C, int64_t H, int64_t W, int64_t sN,
                                       int64_t sC, int64_t sH, int64_t sW, const float *fl, int64_t fN, int64_t fC,
                                       const float *camdist, int64_t dN, int64_t dC, const float *cnt, float *mask,
                                       int res, void *stream) {
  if (int rc = cam_check(depth, N, C, H, W, fl, camdist, res)) return rc;
  GB_REQUIRE(cnt && mask, GENRE_B200_EINVAL, "surface_mask: null pointer");
  const long long nvox = (long long)res * res * res;
  const bool vec = (res % 4 == 0) && aligned16(cnt) && aligned16(mask);
  const long long work = vec ? nvox / 4 : nvox;
  unsigned gx = (unsigned)((work + 255) / 256);
  if (gx > 148u * 16u) gx = 148u * 16u;
  dim3 grid(gx, (unsigned)(N * C));
  surface_mask_kernel<<<grid, 256, 0, as_stream(stream)>>>(depth, (int)C, (int)H, (int)W, sN, sC, sH, sW, fl, fN, fC,
                                                           camdist, dN, dC, cnt, mask, res, nvox, vec);
  return check_launch("surface mask kernel");
}
