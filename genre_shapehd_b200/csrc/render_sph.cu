// render_sph.cu — fused spherical renderer (voxel occupancy -> spherical depth map), forward + backward.
//
// Reference: toolbox/spherical_proj.py:31-72 (render_spherical):
//     grid   = dirs * 2 * (1 - linspace(0,1,Z))            [S,S,Z,3], fp64 numpy -> fp32      (:39-60)
//     prob   = grid_sample(vox.permute(0,1,4,3,2), grid)   trilinear, zero padding, torch-0.4.1
//              semantics == align_corners=True                                               (:63-65)
//     prob   = clamp(prob, 1e-5, 1 - 1e-5)                                                    (:66)
//     stop   = CalcStopProb(prob)                          calc_prob_kernel.cu:112-143        (:67)
//     out    = matmul(stop, linspace(0,1,Z)) + prod(1 - prob, dim=4)                          (:68-71)
// The reference materialises four [N,1,S,S,Z] tensors (256 MiB each at N=16).  Here one warp owns one
// ray: lanes take consecutive samples along the ray (neighbouring samples are ~0.5 voxel apart, so the
// 8-tap gathers of a warp land in a handful of cache lines), the transmittance crosses lanes with a
// shuffle product-scan and crosses 32-sample chunks through a register carry.  Only the [N,S,S] map
// is written.  Sample positions are formed in fp64 from the fp64 direction table exactly like the
// numpy code, then rounded to fp32, so they equal the reference's registered `grid` buffer.
#include "common.cuh"

namespace gb {

constexpr int RS_THREADS = 256;  // 8 rays per CTA
// resident CTAs per SM of the skipping renderer: bounds its registers (48, with 64 B of spills) and sizes its one-wave grid
constexpr int RS_OCC = 5;

struct Taps {
  int base;        // linear index of corner (x0, y0, z0); may be out of range, see masks
  float w[8];      // weights in order (x,y,z) = 000, 001, 010, 011, 100, 101, 110, 111
  unsigned valid;  // bit i set if tap i is inside the volume
};

__device__ __forceinline__ void make_taps(float gx, float gy, float gz, int R, Taps &t) {
  const float Rm1 = (float)(R - 1);
  // grid_sampler unnormalise, align_corners=True: ((coord + 1) / 2) * (size - 1)
  const float fx = __fmul_rn(__fmul_rn(__fadd_rn(gx, 1.0f), 0.5f), Rm1);
  const float fy = __fmul_rn(__fmul_rn(__fadd_rn(gy, 1.0f), 0.5f), Rm1);
  const float fz = __fmul_rn(__fmul_rn(__fadd_rn(gz, 1.0f), 0.5f), Rm1);
  const float x0f = floorf(fx), y0f = floorf(fy), z0f = floorf(fz);
  // clamp before the int conversion so far-away samples (|coord| up to 2) stay well defined
  const int x0 = (int)fminf(fmaxf(x0f, -2.0f), (float)R), y0 = (int)fminf(fmaxf(y0f, -2.0f), (float)R),
            z0 = (int)fminf(fmaxf(z0f, -2.0f), (float)R);
  const float wx1 = fx - x0f, wx0 = (x0f + 1.0f) - fx;
  const float wy1 = fy - y0f, wy0 = (y0f + 1.0f) - fy;
  const float wz1 = fz - z0f, wz0 = (z0f + 1.0f) - fz;
  t.base = (x0 * R + y0) * R + z0;
  t.w[0] = wx0 * wy0 * wz0; t.w[1] = wx0 * wy0 * wz1; t.w[2] = wx0 * wy1 * wz0; t.w[3] = wx0 * wy1 * wz1;
  t.w[4] = wx1 * wy0 * wz0; t.w[5] = wx1 * wy0 * wz1; t.w[6] = wx1 * wy1 * wz0; t.w[7] = wx1 * wy1 * wz1;
  const unsigned Rm = (unsigned)(R - 1);
  if (((unsigned)x0 < Rm) & ((unsigned)y0 < Rm) & ((unsigned)z0 < Rm)) {  // all 8 taps inside: the common case
    t.valid = 0xFFu;
    return;
  }
  const bool vx0 = (unsigned)x0 < (unsigned)R, vx1 = (unsigned)(x0 + 1) < (unsigned)R;
  const bool vy0 = (unsigned)y0 < (unsigned)R, vy1 = (unsigned)(y0 + 1) < (unsigned)R;
  const bool vz0 = (unsigned)z0 < (unsigned)R, vz1 = (unsigned)(z0 + 1) < (unsigned)R;
  t.valid = (unsigned)(vx0 & vy0 & vz0) | ((unsigned)(vx0 & vy0 & vz1) << 1) | ((unsigned)(vx0 & vy1 & vz0) << 2) |
            ((unsigned)(vx0 & vy1 & vz1) << 3) | ((unsigned)(vx1 & vy0 & vz0) << 4) |
            ((unsigned)(vx1 & vy0 & vz1) << 5) | ((unsigned)(vx1 & vy1 & vz0) << 6) |
            ((unsigned)(vx1 & vy1 & vz1) << 7);
}

__device__ __forceinline__ int tap_offset(int i, int R) {
  return ((i >> 2) & 1) * R * R + ((i >> 1) & 1) * R + (i & 1);
}

// Optional transform of every voxel value as it is fetched: v -> clamp(v * scale, lo, hi).  GenRe renders
// clamp(proj * 50, 1e-5, 1 - 1e-5) (depth_pred_with_sph_inpaint.py:124): applying the two elementwise ops here (same
// fp32 operations, same order) removes two dense passes over the volume.  Out-of-volume taps stay 0 (zero padding).
struct VoxPre {
  float scale, lo, hi;
};
template <bool PRE>
__device__ __forceinline__ float fetch_vox(const float *__restrict__ p, const VoxPre &pre) {
  const float v = __ldg(p);
  return PRE ? fminf(fmaxf(__fmul_rn(v, pre.scale), pre.lo), pre.hi) : v;
}

template <bool PRE>
__device__ __forceinline__ float sample_trilinear(const float *__restrict__ vol, const Taps &t, int R, const VoxPre &pre) {
  float acc = 0.0f;
  if (t.valid == 0xFFu) {  // interior: 4 pairs of z-adjacent taps
#pragma unroll
    for (int i = 0; i < 8; ++i) acc = fmaf(fetch_vox<PRE>(vol + t.base + tap_offset(i, R), pre), t.w[i], acc);
  } else if (t.valid) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (t.valid & (1u << i)) acc = fmaf(fetch_vox<PRE>(vol + t.base + tap_offset(i, R), pre), t.w[i], acc);
  }
  return acc;
}

// sample position k on the ray with fp64 direction (dx,dy,dz): (float)(dir*2*(1-alpha_k)), alpha = np.linspace(0,1,Z)
__device__ __forceinline__ void ray_point(double dx2, double dy2, double dz2, int k, int Z, double step, float &gx,
                                          float &gy, float &gz) {
  const double alpha = (k == Z - 1 && Z > 1) ? 1.0 : (double)k * step;
  const double f = 1.0 - alpha;
  gx = (float)(dx2 * f);
  gy = (float)(dy2 * f);
  gz = (float)(dz2 * f);
}

__device__ __forceinline__ float warp_excl_prod32(float v, float &total) {
  float incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const float u = __shfl_up_sync(0xffffffffu, incl, d);
    if ((threadIdx.x & 31) >= d) incl *= u;
  }
  total = __shfl_sync(0xffffffffu, incl, 31);
  float excl = __shfl_up_sync(0xffffffffu, incl, 1);
  if ((threadIdx.x & 31) == 0) excl = 1.0f;
  return excl;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

constexpr float RS_PMIN = 1e-5f;
constexpr float RS_PMAX = (float)(1.0 - 1e-5);

// forward pass over one ray; returns (sum_k s_k w_k, prod_k (1 - p_k)) to every lane
template <bool PRE>
__device__ __forceinline__ void render_ray(const float *__restrict__ vol, int R, double dx2, double dy2, double dz2,
                                           int Z, const float *__restrict__ depth_weight, const VoxPre &pre,
                                           float &exp_depth, float &trans) {
  const int lane = threadIdx.x & 31;
  const double step = Z > 1 ? 1.0 / (double)(Z - 1) : 0.0;
  float carry = 1.0f, acc = 0.0f;
  for (int k0 = 0; k0 < Z; k0 += 32) {
    const int k = k0 + lane;
    float p = 0.0f;  // lanes past the end behave like p = 0 (factor 1, no contribution)
    if (k < Z) {
      float gx, gy, gz;
      ray_point(dx2, dy2, dz2, k, Z, step, gx, gy, gz);
      Taps t;
      make_taps(gx, gy, gz, R, t);
      p = fminf(fmaxf(sample_trilinear<PRE>(vol, t, R, pre), RS_PMIN), RS_PMAX);
    }
    float total;
    const float before = carry * warp_excl_prod32(1.0f - p, total);
    if (k < Z) acc = fmaf(p * before, __ldg(depth_weight + k), acc);
    carry *= total;
    if (carry == 0.0f) break;  // transmittance underflowed: every later term is exactly 0 (warp-uniform)
  }
  exp_depth = warp_sum(acc);
  trans = carry;
}

template <bool PRE>
__global__ void __launch_bounds__(RS_THREADS)
render_spherical_forward_kernel(const float *__restrict__ vox, int R, const double *__restrict__ dirs, int S, int Z,
                                const float *__restrict__ depth_weight, float *__restrict__ out, long long n_rays,
                                const VoxPre pre) {
  const long long ray = (long long)blockIdx.x * (RS_THREADS / 32) + (threadIdx.x >> 5);
  if (ray >= n_rays) return;
  const int pix = (int)(ray % ((long long)S * S));
  const long long n = ray / ((long long)S * S);
  const float *vol = vox + (size_t)n * R * R * R;
  const double dx2 = dirs[pix * 3 + 0] * 2.0, dy2 = dirs[pix * 3 + 1] * 2.0, dz2 = dirs[pix * 3 + 2] * 2.0;
  float e, t;
  render_ray<PRE>(vol, R, dx2, dy2, dz2, Z, depth_weight, pre, e, t);
  if ((threadIdx.x & 31) == 0) out[ray] = e + t;
}

// ---- empty-space skipping (forward) ---------------------------------------------------------------------------------
// GenRe renders a thin shell: clamp(proj * 50, 1e-5, 1 - 1e-5) is 1e-5 everywhere except on the ~1 % of voxels the depth
// map hit, and a third of every ray lies outside the volume, yet the plain kernel pays ~200 instructions (fp64 position,
// 8 gathers, scan) for each of its 4.19 M samples per shape: it is issue-bound (ncu: 412 M warp instructions, 78 % issue
// active, profiles/r02_render_summary.md).  A sample whose 8 taps are all <= 1e-5 (or outside: zero padding) clamps to
// p = 1e-5 (up to a 1e-12 rounding of the interpolation), and a run of such samples has a closed form:
//     T after n samples = T * q^n,     sum_k s_k w_k over the run = 1e-5 * T * (S[b] - S[a]) / q^a,
//     q = 1 - 1e-5,   S[k] = sum_{j<k} q^j w_j  (prefix table built per CTA from the caller's depth_weight buffer).
//   pre-pass  (render_occupancy_*): one read of the volume -> a bit per 4^3 brick b, set when any voxel in [4b-1, 4b+5]
//             per dimension exceeds 1e-5: a sample at voxel coordinate f reads taps floor(f), floor(f)+1, so the brick
//             floor(f/4) covers both (+4), the -1 / +5 absorb the fp32 estimate of f used for the lookup;
//   render    a warp owns 4 neighbouring rays x 8 consecutive samples per step.  The bounding box of the marked bricks
//             gives each ray a sample range [K0, K1): everything before and after it is ONE closed-form update.  Inside,
//             every lane looks its sample's brick up in a 64^3-brick padded bitmask in shared memory (32 KB) (3 FMAs + 3 floors:
//             positions anywhere in [-2, 2]^3 index it without range checks); a step whose 32 samples are all empty is a
//             closed-form update, otherwise the lanes on occupied bricks take the exact path (fp64 positions, 8 taps) and the
//             transmittance is scanned inside each 8-lane group.
// Error against the sample-by-sample product: a few 1e-7 relative on T (measured <= 4e-6 on the output).
constexpr int RS_BRICK = 4;
constexpr int RS_NB_MAX = 32;         // bricks per dimension the padded mask covers (res <= 128)
constexpr int RS_PAD = 16;            // padding bricks on each side: |coord| <= 2  ->  brick index in [-16, 48)
constexpr int RS_PB = 64;             // padded bricks per dimension
constexpr int RS_MAX_Z = 1024;
constexpr float RS_LOG2_Q = -1.4427022e-05f;  // log2(1 - 1e-5)
constexpr float RS_INV_BRICK = 1.0f / RS_BRICK;

__host__ __device__ inline int rs_bricks(int R) { return (R + RS_BRICK - 1) / RS_BRICK; }
__host__ __device__ inline int rs_occ_words(int R) {
  const int nb = rs_bricks(R);
  return (nb * nb * nb + 31) / 32;
}

// generic pre-pass: one thread per 4 z-adjacent voxels (R % 4 == 0); blockIdx.y = volume
template <bool PRE>
__global__ void __launch_bounds__(256)
render_occupancy_kernel(const float *__restrict__ vox, int R, long long vox_per_vol4, unsigned *__restrict__ occ,
                        const VoxPre pre) {
  const long long i4 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i4 >= vox_per_vol4) return;
  const int n = blockIdx.y;
  const float4 v = *reinterpret_cast<const float4 *>(vox + ((size_t)n * vox_per_vol4 + i4) * 4);
  float a[4] = {v.x, v.y, v.z, v.w};
  int zlo = 4, zhi = -1;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float t = PRE ? fminf(fmaxf(__fmul_rn(a[i], pre.scale), pre.lo), pre.hi) : a[i];
    if (!(t <= RS_PMIN)) {  // NaN counts as occupied
      zlo = min(zlo, i);
      zhi = max(zhi, i);
    }
  }
  if (zhi < 0) return;
  const long long lin = i4 * 4;
  const int z = (int)(lin % R), y = (int)((lin / R) % R), x = (int)(lin / ((long long)R * R));
  const int nb = rs_bricks(R);
  // brick b is marked iff an occupied voxel lies in [4b - 1, 4b + 5]  <=>  b in [floor((v - 2) / 4), floor((v + 1) / 4)]
  const int bx0 = max(x - 2, 0) / RS_BRICK, bx1 = min(x + 1, R - 1) / RS_BRICK;
  const int by0 = max(y - 2, 0) / RS_BRICK, by1 = min(y + 1, R - 1) / RS_BRICK;
  const int bz0 = max(z + zlo - 2, 0) / RS_BRICK, bz1 = min(z + zhi + 1, R - 1) / RS_BRICK;
  unsigned *o = occ + (size_t)n * rs_occ_words(R);
  for (int bx = bx0; bx <= bx1; ++bx)
    for (int by = by0; by <= by1; ++by)
      for (int bz = bz0; bz <= bz1; ++bz) {
        const int bit = (bx * nb + by) * nb + bz;
        const unsigned m = 1u << (bit & 31);
        if (!(o[bit >> 5] & m)) atomicOr(&o[bit >> 5], m);
      }
}

// R = 128 pre-pass: a warp owns whole z rows (32 lanes x 4 voxels = 128), 4 rows in flight per iteration; a row's 32 z-brick
// bits are OR-reduced across the warp and merged into the (at most 2 x 2) brick columns its dilated (x, y) touches.
template <bool PRE>
__global__ void __launch_bounds__(256)
render_occupancy128_kernel(const float *__restrict__ vox, unsigned *__restrict__ occ, const VoxPre pre) {
  constexpr int R = 128, ROWS = 4, NB = R / RS_BRICK;
  static_assert(NB == 32, "one 32-bit word per (bx, by) brick column");
  const int n = blockIdx.y, lane = threadIdx.x & 31;
  const int warp_global = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int row0 = warp_global * ROWS;  // row index = x * R + y
  if (row0 >= R * R) return;
  const float4 *base = reinterpret_cast<const float4 *>(vox + (size_t)n * R * R * R) + (size_t)row0 * 32 + lane;
  float4 v[ROWS];
#pragma unroll
  for (int r = 0; r < ROWS; ++r) v[r] = __ldcs(base + r * 32);
  unsigned *o = occ + (size_t)n * rs_occ_words(R);
#pragma unroll
  for (int r = 0; r < ROWS; ++r) {
    const float a[4] = {v[r].x, v[r].y, v[r].z, v[r].w};
    unsigned zmask = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float t = PRE ? fminf(fmaxf(__fmul_rn(a[i], pre.scale), pre.lo), pre.hi) : a[i];
      if (!(t <= RS_PMIN)) {
        const int z = lane * 4 + i;
        zmask |= (1u << (max(z - 2, 0) / RS_BRICK)) | (1u << (min(z + 1, R - 1) / RS_BRICK));
      }
    }
    zmask = __reduce_or_sync(0xffffffffu, zmask);
    if (zmask == 0 || lane >= 4) continue;
    const int row = row0 + r, x = row >> 7, y = row & 127;
    const int bx = ((lane & 1) ? min(x + 1, R - 1) : max(x - 2, 0)) / RS_BRICK;
    const int by = ((lane & 2) ? min(y + 1, R - 1) : max(y - 2, 0)) / RS_BRICK;
    unsigned *w = o + bx * NB + by;   // bit = (bx*32 + by)*32 + bz: one word per brick column
    if ((*w & zmask) != zmask) atomicOr(w, zmask);
  }
}

template <bool PRE>
__global__ void __launch_bounds__(RS_THREADS, RS_OCC)
render_spherical_forward_skip_kernel(const float *__restrict__ vox, int R, const double *__restrict__ dirs, int S, int Z,
                                     const float *__restrict__ depth_weight, const unsigned *__restrict__ occ,
                                     float *__restrict__ out, const VoxPre pre) {
  __shared__ unsigned long long s_occ[RS_PB * RS_PB];  // padded brick mask: word = X * 64 + Y, bit = Z (padded brick coordinates)
  __shared__ float s_S[RS_MAX_Z + 1];                  // S[k] = sum_{j<k} q^j w_j
  __shared__ int s_box[7];                             // marked-brick bounding box: min x,y,z, max x,y,z (unpadded); [6] = marked bricks
  const int n = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nb = rs_bricks(R), words = rs_occ_words(R);
  if (tid < 3) s_box[tid] = nb;
  else if (tid < 6) s_box[tid] = -1;
  else if (tid == 6) s_box[6] = 0;
  // prefix table of q^j w_j: warp 0, 32 entries per pass
  if (warp == 0) {
    float run = 0.0f;
    for (int k0 = 0; k0 < Z; k0 += 32) {
      const int k = k0 + lane;
      float v = k < Z ? exp2f((float)k * RS_LOG2_Q) * __ldg(depth_weight + k) : 0.0f;
      float incl = v;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const float u = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += u;
      }
      if (k < Z) s_S[k + 1] = run + incl;
      run += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (lane == 0) s_S[0] = 0.0f;
  }
  __syncthreads();
  // padded mask: thread-owned words (no atomics).  Padded column (X, Y) holds brick column (X - PAD, Y - PAD); a sample with
  // f in (-1, 0) reads voxel 0 but floors to brick -1, so column -1 (and bit -1) copy column 0 (bit 0).
  const unsigned *cocc = occ + (size_t)n * words;
  for (int wi = tid; wi < RS_PB * RS_PB; wi += RS_THREADS) {
    int bx = wi / RS_PB - RS_PAD, by = wi % RS_PB - RS_PAD;
    const bool own = bx >= 0 && by >= 0;      // not a boundary copy: contributes to the bounding box
    if (bx == -1) bx = 0;
    if (by == -1) by = 0;
    unsigned long long row = 0;
    if (bx >= 0 && bx < nb && by >= 0 && by < nb) {
      const int bit0 = (bx * nb + by) * nb;   // nb <= 32 consecutive bits of the compact mask
      const int w0 = bit0 >> 5, sh = bit0 & 31;
      unsigned long long win = cocc[w0];
      if (sh + nb > 32 && w0 + 1 < words) win |= (unsigned long long)cocc[w0 + 1] << 32;
      const unsigned bits = (unsigned)(win >> sh) & (nb == 32 ? 0xffffffffu : ((1u << nb) - 1u));
      if (bits) {
        row = ((unsigned long long)bits << RS_PAD) | ((unsigned long long)(bits & 1u) << (RS_PAD - 1));
        if (own) {
          atomicMin(&s_box[0], bx); atomicMin(&s_box[1], by); atomicMin(&s_box[2], __ffs(bits) - 1);
          atomicMax(&s_box[3], bx); atomicMax(&s_box[4], by); atomicMax(&s_box[5], 31 - __clz(bits));
          atomicAdd(&s_box[6], __popc(bits));
        }
      }
    }
    s_occ[wi] = row;
  }
  __syncthreads();
  const bool any = s_box[3] >= 0;
  // a volume with occupied voxels in most bricks (nothing to skip) takes every step of the box range on the exact path
  // without the per-sample tests
  const bool dense = s_box[6] * 5 > nb * nb * nb * 2;
  // sample-space box: a sample looks up brick floor(f / 4) (f in [-4, 0) finds the copies of boundary marks)
  float blo[3], bhi[3];
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    blo[d] = s_box[d] == 0 ? -(float)RS_BRICK - 0.01f : (float)(RS_BRICK * s_box[d]) - 0.01f;
    bhi[d] = (float)(RS_BRICK * (s_box[3 + d] + 1)) + 0.01f;
  }
  const float h = 0.5f * (float)(R - 1), stepf = Z > 1 ? 1.0f / (float)(Z - 1) : 0.0f;
  const double step = Z > 1 ? 1.0 / (double)(Z - 1) : 0.0;
  const float *vol = vox + (size_t)n * R * R * R;
  const int j = lane & 7, grp = lane >> 3;
  const int nsteps = (Z + 7) / 8;
  const int ngroups = (S * S + 3) / 4;
  // 4-ray groups in a strided order: neighbouring groups (similar cost) go to different warps; the next group's direction
  // is fetched while the current one is marched
  const int gstride = gridDim.x * (RS_THREADS / 32);
  int g = blockIdx.x * (RS_THREADS / 32) + warp;
  double ndx = 0.0, ndy = 0.0, ndz = 0.0;
  if (g < ngroups) {
    const int pc = min(g * 4 + grp, S * S - 1);
    ndx = __ldg(dirs + pc * 3 + 0); ndy = __ldg(dirs + pc * 3 + 1); ndz = __ldg(dirs + pc * 3 + 2);
  }
  for (; g < ngroups; g += gstride) {
    const double dx = ndx, dy = ndy, dz = ndz;
    if (g + gstride < ngroups) {
      const int pc = min((g + gstride) * 4 + grp, S * S - 1);
      ndx = __ldg(dirs + pc * 3 + 0); ndy = __ldg(dirs + pc * 3 + 1); ndz = __ldg(dirs + pc * 3 + 2);
    }
    const int pix = g * 4 + grp;
    const bool ray_ok = pix < S * S;
    const double dx2 = dx * 2.0, dy2 = dy * 2.0, dz2 = dz * 2.0;
    // voxel coordinate of sample k (fp32 estimate): f = h + d*h*2*(1 - k*step) = A - Bk * k
    const float A[3] = {h + 2.0f * (float)dx * h, h + 2.0f * (float)dy * h, h + 2.0f * (float)dz * h};
    const float Bk[3] = {2.0f * (float)dx * h * stepf, 2.0f * (float)dy * h * stepf, 2.0f * (float)dz * h * stepf};
    // this ray's sample range inside the box (slab test on the real-valued sample index)
    float kmin = 0.0f, kmax = (float)Z;
    if (!any || !ray_ok) kmax = -1.0f;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      if (fabsf(Bk[d]) > 1e-12f) {
        const float inv = __frcp_rn(Bk[d]);
        const float k1 = (A[d] - blo[d]) * inv, k2 = (A[d] - bhi[d]) * inv;
        kmin = fmaxf(kmin, fminf(k1, k2));
        kmax = fminf(kmax, fmaxf(k1, k2));
      } else if (A[d] < blo[d] || A[d] > bhi[d]) {
        kmax = -1.0f;
      }
    }
    int s0 = nsteps, s1 = 0;  // steps [s0, s1) need per-sample tests
    if (kmax >= kmin) {
      s0 = max(0, (int)floorf(kmin) - 1) >> 3;
      s1 = min(nsteps, (min(Z, (int)ceilf(kmax) + 2) + 7) >> 3);
      if (s1 <= s0) { s0 = nsteps; s1 = 0; }
    }
    s0 = __reduce_min_sync(0xffffffffu, s0);
    s1 = __reduce_max_sync(0xffffffffu, s1);
    float T = 1.0f, acc = 0.0f, acc_u = 0.0f;
    int kdone = 0;  // samples [0, kdone) are accounted for
    // phase A: occupancy of every sample of every candidate step, independent iterations (the loads and conversions of
    // several steps are in flight together); windows of 32 steps
    const float Ab[3] = {A[0] * RS_INV_BRICK + RS_PAD, A[1] * RS_INV_BRICK + RS_PAD, A[2] * RS_INV_BRICK + RS_PAD};
    const float Bb[3] = {Bk[0] * RS_INV_BRICK, Bk[1] * RS_INV_BRICK, Bk[2] * RS_INV_BRICK};
    for (int w0 = s0; w0 < s1; w0 += 32) {   // warp-uniform bounds (ballots inside)
      const int w1 = min(w0 + 32, s1);
      unsigned mine = 0;       // bit i: this lane's sample of step w0 + i is occupied
      unsigned steps_any = 0;  // bit i: some lane's sample of step w0 + i is occupied (warp-uniform)
      if (dense) {
        steps_any = w1 - w0 == 32 ? 0xffffffffu : (1u << (w1 - w0)) - 1u;
        mine = ray_ok ? steps_any : 0u;
      } else
#pragma unroll 4
      for (int s = w0; s < w1; ++s) {
        const int k = 8 * s + j;
        const float kf = (float)k;
        const int X = (int)floorf(fmaf(-Bb[0], kf, Ab[0])), Y = (int)floorf(fmaf(-Bb[1], kf, Ab[1])),
                  Zb = (int)floorf(fmaf(-Bb[2], kf, Ab[2]));
        const bool occupied = ((s_occ[(X & (RS_PB - 1)) * RS_PB + (Y & (RS_PB - 1))] >> (Zb & (RS_PB - 1))) & 1ull) && k < Z && ray_ok;
        mine |= (unsigned)occupied << (s - w0);
        steps_any |= (__ballot_sync(0xffffffffu, occupied) ? 1u : 0u) << (s - w0);
      }
      // phase B: jump from occupied step to occupied step
      while (steps_any) {
        const int i = __ffs(steps_any) - 1;
        steps_any &= steps_any - 1;
        const int s = w0 + i, kstart = 8 * s, k = kstart + j;
        if (kstart > kdone) {  // the empty run [kdone, kstart) in closed form
          acc_u = fmaf(RS_PMIN * T, (s_S[kstart] - s_S[kdone]) * exp2f(-(float)kdone * RS_LOG2_Q), acc_u);
          T *= exp2f((float)(kstart - kdone) * RS_LOG2_Q);
        }
        float p = 0.0f;  // lanes past the end behave like p = 0 (factor 1, no contribution)
        if (k < Z) {
          p = RS_PMIN;
          if ((mine >> i) & 1u) {
            float gx, gy, gz;
            ray_point(dx2, dy2, dz2, k, Z, step, gx, gy, gz);
            Taps t;
            make_taps(gx, gy, gz, R, t);
            p = fminf(fmaxf(sample_trilinear<PRE>(vol, t, R, pre), RS_PMIN), RS_PMAX);
          }
        }
        float incl = 1.0f - p;
#pragma unroll
        for (int d = 1; d < 8; d <<= 1) {
          const float u = __shfl_up_sync(0xffffffffu, incl, d, 8);
          if (j >= d) incl *= u;
        }
        const float total = __shfl_sync(0xffffffffu, incl, 7, 8);
        float excl = __shfl_up_sync(0xffffffffu, incl, 1, 8);
        if (j == 0) excl = 1.0f;
        if (k < Z) acc = fmaf(p * (T * excl), __ldg(depth_weight + k), acc);
        T *= total;
        kdone = min(kstart + 8, Z);
        if (__all_sync(0xffffffffu, T == 0.0f)) { steps_any = 0; }  // every later term of all four rays is exactly 0
      }
      if (__all_sync(0xffffffffu, T == 0.0f)) break;
    }
    // tail: samples [kdone, Z) in closed form (T == 0 contributes exactly 0)
    if (kdone < Z) {
      acc_u = fmaf(RS_PMIN * T, (s_S[Z] - s_S[kdone]) * exp2f(-(float)kdone * RS_LOG2_Q), acc_u);
      T *= exp2f((float)(Z - kdone) * RS_LOG2_Q);
    }
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o, 8);
    if (j == 0 && ray_ok) out[(size_t)n * S * S + pix] = acc + acc_u + T;
  }
}

// backward: d out / d p_k = T_k w_k - (A_k + T_Z) / (1 - p_k),  A_k = sum_{m>k} w_m s_m, scattered through the
// trilinear weights (zero where the clamp was active, as torch.clamp's backward).  Pass 1 walks the ray
// forward keeping the raw samples and prefix transmittances in registers; pass 2 walks it backward so
// A_k is a plain running sum of non-negative terms (no cancellation against 1/(1-p) ~ 1e5).
constexpr int RS_MAX_CHUNKS = 8;  // backward keeps Z/32 samples per lane in registers -> Z <= 256

__global__ void __launch_bounds__(RS_THREADS)
render_spherical_backward_kernel(const float *__restrict__ vox, int R, const double *__restrict__ dirs, int S, int Z,
                                 const float *__restrict__ depth_weight, const float *__restrict__ grad_out,
                                 float *__restrict__ grad_vox, long long n_rays) {
  const long long ray = (long long)blockIdx.x * (RS_THREADS / 32) + (threadIdx.x >> 5);
  if (ray >= n_rays) return;
  const int lane = threadIdx.x & 31;
  const int pix = (int)(ray % ((long long)S * S));
  const long long n = ray / ((long long)S * S);
  const float *vol = vox + (size_t)n * R * R * R;
  float *gvol = grad_vox + (size_t)n * R * R * R;
  const float g = grad_out[ray];
  if (g == 0.0f) return;
  const double dx2 = dirs[pix * 3 + 0] * 2.0, dy2 = dirs[pix * 3 + 1] * 2.0, dz2 = dirs[pix * 3 + 2] * 2.0;
  const double step = Z > 1 ? 1.0 / (double)(Z - 1) : 0.0;

  float raw[RS_MAX_CHUNKS], Tk[RS_MAX_CHUNKS];
  float carry = 1.0f;
  int last_chunk = 0;
#pragma unroll
  for (int c = 0; c < RS_MAX_CHUNKS; ++c) {
    raw[c] = 0.0f;
    Tk[c] = 0.0f;
    const int k = c * 32 + lane;
    if (c * 32 < Z && carry != 0.0f) {  // warp-uniform
      float p = 0.0f;
      if (k < Z) {
        float gx, gy, gz;
        ray_point(dx2, dy2, dz2, k, Z, step, gx, gy, gz);
        Taps t;
        make_taps(gx, gy, gz, R, t);
        raw[c] = sample_trilinear<false>(vol, t, R, VoxPre{});
        p = fminf(fmaxf(raw[c], RS_PMIN), RS_PMAX);
      }
      float total;
      Tk[c] = carry * warp_excl_prod32(1.0f - p, total);
      carry *= total;
      last_chunk = c;
    }
  }
  const float t_all = carry;  // prod over the whole ray (0 if it underflowed; later samples then have zero gradient)

  float suffix = 0.0f;  // sum_{m in later chunks} w_m s_m
#pragma unroll
  for (int c = RS_MAX_CHUNKS - 1; c >= 0; --c) {
    if (c > last_chunk) continue;  // warp-uniform
    const int k = c * 32 + lane;
    const bool live = k < Z;
    const float p = live ? fminf(fmaxf(raw[c], RS_PMIN), RS_PMAX) : 0.0f;
    const float wk = live ? __ldg(depth_weight + k) : 0.0f;
    const float ws = wk * p * Tk[c];
    // exclusive suffix sum over lanes
    float incl = ws;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const float u = __shfl_down_sync(0xffffffffu, incl, d);
      if (lane + d < 32) incl += u;
    }
    float excl = __shfl_down_sync(0xffffffffu, incl, 1);
    if (lane == 31) excl = 0.0f;
    const float Ak = suffix + excl;
    suffix += __shfl_sync(0xffffffffu, incl, 0);
    if (live && raw[c] >= RS_PMIN && raw[c] <= RS_PMAX) {
      const float dp = g * (Tk[c] * wk - (Ak + t_all) / (1.0f - p));
      if (dp != 0.0f) {
        float gx, gy, gz;
        ray_point(dx2, dy2, dz2, k, Z, step, gx, gy, gz);
        Taps t;
        make_taps(gx, gy, gz, R, t);
#pragma unroll
        for (int i = 0; i < 8; ++i)
          if (t.valid & (1u << i)) atomicAdd(gvol + t.base + tap_offset(i, R), dp * t.w[i]);
      }
    }
  }
}

static int rs_check(const float *vox, int64_t N, int res, const double *dirs, int S, int Z, const float *dw) {
  GB_REQUIRE(vox && dirs && dw, GENRE_B200_EINVAL, "render_spherical: null pointer");
  GB_REQUIRE(N > 0 && res >= 2 && (int64_t)res * res * res < (1ll << 31) && S > 0 && Z > 0, GENRE_B200_EINVAL,
             "render_spherical: bad shape (N=%lld, R=%d, S=%d, Z=%d)", (long long)N, res, S, Z);
  GB_REQUIRE(((int64_t)N * S * S + 7) / 8 < (1ll << 31), GENRE_B200_EINVAL, "render_spherical: too many rays");
  return 0;
}

}  // namespace gb

using namespace gb;

extern "C" int genre_b200_render_spherical_forward(const float *vox, int64_t N, int res, const double *dirs,
                                                   int sph_res, int z_res, const float *depth_weight, float *out,
                                                   void *stream) {
  if (int rc = rs_check(vox, N, res, dirs, sph_res, z_res, depth_weight)) return rc;
  GB_REQUIRE(out != nullptr, GENRE_B200_EINVAL, "render_spherical: out is null");
  const long long n_rays = (long long)N * sph_res * sph_res;
  const unsigned grid = (unsigned)((n_rays + RS_THREADS / 32 - 1) / (RS_THREADS / 32));
  render_spherical_forward_kernel<false><<<grid, RS_THREADS, 0, as_stream(stream)>>>(vox, res, dirs, sph_res, z_res,
                                                                                     depth_weight, out, n_rays, VoxPre{});
  return check_launch("render_spherical forward kernel");
}

// Same renderer over clamp(vox * pre_scale, pre_lo, pre_hi) without materialising that volume (forward only: the
// fused GenRe inference path, depth_pred_with_sph_inpaint.py:124 `render_spherical(clamp(proj * 50, 1e-5, 1 - 1e-5))`).
extern "C" int genre_b200_render_spherical_forward_pre(const float *vox, int64_t N, int res, const double *dirs,
                                                       int sph_res, int z_res, const float *depth_weight,
                                                       float pre_scale, float pre_lo, float pre_hi, float *out,
                                                       void *stream) {
  if (int rc = rs_check(vox, N, res, dirs, sph_res, z_res, depth_weight)) return rc;
  GB_REQUIRE(out != nullptr, GENRE_B200_EINVAL, "render_spherical: out is null");
  GB_REQUIRE(pre_lo <= pre_hi, GENRE_B200_EINVAL, "render_spherical: empty clamp range");
  const long long n_rays = (long long)N * sph_res * sph_res;
  const unsigned grid = (unsigned)((n_rays + RS_THREADS / 32 - 1) / (RS_THREADS / 32));
  render_spherical_forward_kernel<true><<<grid, RS_THREADS, 0, as_stream(stream)>>>(
      vox, res, dirs, sph_res, z_res, depth_weight, out, n_rays, VoxPre{pre_scale, pre_lo, pre_hi});
  return check_launch("render_spherical forward kernel (pre-transform)");
}

extern "C" int genre_b200_render_spherical_backward(const float *vox, int64_t N, int res, const double *dirs,
                                                    int sph_res, int z_res, const float *depth_weight,
                                                    const float *grad_out, float *grad_vox, void *stream) {
  if (int rc = rs_check(vox, N, res, dirs, sph_res, z_res, depth_weight)) return rc;
  GB_REQUIRE(grad_out && grad_vox, GENRE_B200_EINVAL, "render_spherical backward: null pointer");
  GB_REQUIRE(z_res <= 32 * RS_MAX_CHUNKS, GENRE_B200_EINVAL, "render_spherical backward: z_res %d > %d unsupported",
             z_res, 32 * RS_MAX_CHUNKS);
  const long long n_rays = (long long)N * sph_res * sph_res;
  const unsigned grid = (unsigned)((n_rays + RS_THREADS / 32 - 1) / (RS_THREADS / 32));
  render_spherical_backward_kernel<<<grid, RS_THREADS, 0, as_stream(stream)>>>(vox, res, dirs, sph_res, z_res,
                                                                               depth_weight, grad_out, grad_vox, n_rays);
  return check_launch("render_spherical backward kernel");
}

extern "C" size_t genre_b200_render_spherical_workspace_bytes(int64_t N, int res) {
  if (N <= 0 || res < 2) return 0;
  return (size_t)N * rs_occ_words(res) * sizeof(unsigned);   // one bit per 4^3 brick
}

// The same renderer with empty-space skipping (see the header of the skipping section): identical results up to ~1e-6.
//   use_pre != 0: render clamp(vox * pre_scale, pre_lo, pre_hi) without materialising it
//   workspace: genre_b200_render_spherical_workspace_bytes(N, res) bytes, caller-owned, zeroed here (memset node)
// Supported: res % 4 == 0, res <= 128, z_res <= 1024, 16-byte aligned vox; otherwise the call is forwarded to the plain kernel.
extern "C" int genre_b200_render_spherical_forward_skip(const float *vox, int64_t N, int res, const double *dirs,
                                                        int sph_res, int z_res, const float *depth_weight, int use_pre,
                                                        float pre_scale, float pre_lo, float pre_hi, float *out,
                                                        void *workspace, size_t workspace_bytes, void *stream) {
  if (int rc = rs_check(vox, N, res, dirs, sph_res, z_res, depth_weight)) return rc;
  GB_REQUIRE(out != nullptr, GENRE_B200_EINVAL, "render_spherical: out is null");
  GB_REQUIRE(!use_pre || pre_lo <= pre_hi, GENRE_B200_EINVAL, "render_spherical: empty clamp range");
  const size_t need = genre_b200_render_spherical_workspace_bytes(N, res);
  const bool can_skip = res % 4 == 0 && rs_bricks(res) <= RS_NB_MAX && z_res <= RS_MAX_Z && aligned16(vox) && N < 65536;
  if (!can_skip) {
    if (use_pre) return genre_b200_render_spherical_forward_pre(vox, N, res, dirs, sph_res, z_res, depth_weight, pre_scale, pre_lo, pre_hi, out, stream);
    return genre_b200_render_spherical_forward(vox, N, res, dirs, sph_res, z_res, depth_weight, out, stream);
  }
  GB_REQUIRE(workspace && workspace_bytes >= need && ((uintptr_t)workspace & 3) == 0, GENRE_B200_EINVAL,
             "render_spherical: workspace of %zu bytes needed (got %zu)", need, workspace_bytes);
  cudaStream_t st = as_stream(stream);
  cudaError_t e = cudaMemsetAsync(workspace, 0, need, st);
  if (e != cudaSuccess) return fail_arg((int)e, "render_spherical: cudaMemsetAsync: %s", cudaGetErrorString(e));
  const VoxPre pre = use_pre ? VoxPre{pre_scale, pre_lo, pre_hi} : VoxPre{};
  if (res == 128) {
    dim3 og((unsigned)(128 * 128 / (8 * 4)), (unsigned)N);  // 8 warps x 4 rows per CTA
    if (use_pre) render_occupancy128_kernel<true><<<og, 256, 0, st>>>(vox, (unsigned *)workspace, pre);
    else render_occupancy128_kernel<false><<<og, 256, 0, st>>>(vox, (unsigned *)workspace, pre);
  } else {
    const long long v4 = (long long)res * res * res / 4;
    dim3 og((unsigned)((v4 + 255) / 256), (unsigned)N);
    if (use_pre) render_occupancy_kernel<true><<<og, 256, 0, st>>>(vox, res, v4, (unsigned *)workspace, pre);
    else render_occupancy_kernel<false><<<og, 256, 0, st>>>(vox, res, v4, (unsigned *)workspace, pre);
  }
  if (int rc = check_launch("render_spherical occupancy kernel")) return rc;
  const int ngroups = (sph_res * sph_res + 3) / 4;
  // one wave of resident CTAs over the whole batch (RS_OCC per SM, 148 SMs), warps stride over the ray groups
  int ctas = (int)((148 * RS_OCC) / N);
  const int max_ctas = (ngroups + RS_THREADS / 32 - 1) / (RS_THREADS / 32);
  if (ctas > max_ctas) ctas = max_ctas;
  if (ctas < 1) ctas = 1;
  dim3 rg((unsigned)ctas, (unsigned)N);
  if (use_pre)
    render_spherical_forward_skip_kernel<true><<<rg, RS_THREADS, 0, st>>>(vox, res, dirs, sph_res, z_res, depth_weight,
                                                                         (const unsigned *)workspace, out, pre);
  else
    render_spherical_forward_skip_kernel<false><<<rg, RS_THREADS, 0, st>>>(vox, res, dirs, sph_res, z_res, depth_weight,
                                                                          (const unsigned *)workspace, out, pre);
  return check_launch("render_spherical forward kernel (empty-space skipping)");
}
