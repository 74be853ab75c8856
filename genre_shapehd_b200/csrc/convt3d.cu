// convt3d.cu — stride-2 ConvTranspose3d forward as a tcgen05 (5th-gen tensor core) implicit GEMM, TF32 in / FP32 out.
//
// Reference layers: networks/networks.py:162-167 (Unet_3D.dec2..dec6 = Deconv3d_skip: cat(x, skip) ->
// ConvTranspose3d(k, s=2, p) [-> BatchNorm3d -> LeakyReLU]), :253-256,:40-57 (VoxelDecoder / VoxelGenerator
// deconv3d_2x).  The dominant one, dec5 = ConvT(80 -> 20, k=8, s=2, p=3) on 32^3, is 53.7 of Unet_3D's 78 GFLOP.
//
// Formulation.  o = 2 i - p + k splits the output into 8 parity classes (o = 2 j + par); class `par` only sees
// the taps k = k0 + 2 t, t < T = K/2, at input positions i = j + base - t: a stride-1 T^3-tap convolution.
//     GEMM per class:  M = B * D*H*W positions,  N = Cout (padded to NPAD),  K = T^3 * Cin
// Activations are kept channel-BLOCKED: [B*D][C/4][H][W][4] (16 bytes per position and channel group), so
//   * a shared-memory halo [cg][y][x][4] is exactly tcgen05's canonical K-major NO-SWIZZLE operand layout
//     (core matrix = 8 consecutive x positions x 16 B; next y row = SBO; next channel group = LBO), and
//   * the operand of ANY tap is the same halo at a different 16-byte-aligned start address: one halo load feeds
//     T*T (y,x) taps and MT M-tiles, which is what keeps the kernel off the L2 bandwidth wall at N = 20.
// The two sources of the skip concatenation are two tensors walked one after the other along K (the cat is never
// materialised).  Weights are pre-packed on the host into the exact shared-memory image of each (parity, z-tap,
// K-chunk) stage and arrive with ONE cp.async.bulk per stage.
//
// CTA = one (b, z, 16 y-rows, full W) output slab of one parity class: MT = W/8 M-tiles of 128 rows, accumulators
// MT x NPAD fp32 columns in TMEM.  Warps 0-3: halo producer (one thread issues the tensor copies, zero-fill = padding),
// then epilogue (tcgen05.ld -> scale/shift/LeakyReLU -> blocked store).  Warp 4: TMEM allocation + single-thread MMA issue.
// Pipeline: STAGES-deep ring of (halo chunk, weight chunk) with full/empty mbarriers; tcgen05.commit frees a slot.
#include <cuda.h>   // CUtensorMap + the cuTensorMapEncodeTiled prototype (the entry point is resolved through the runtime: no -lcuda)
#include <cstring>
#include "common.cuh"
#include "tc_ptx.cuh"

namespace gb {

constexpr int CT_THREADS = 160;       // 4 producer/epilogue warps + 1 MMA warp
constexpr int CT_BY = 16;             // y rows per CTA (16 core-matrix groups of 8 x positions = M 128)
constexpr int CT_KCG = 2;             // channel groups (of 4) per stage = one K=8 TF32 MMA per tap and M-tile

struct ConvTParams {
  const float *src0, *src1;  // blocked activations [B*D][cg][H][W][16 bytes]; src1 may be null (cg1 = 0).
                             // A channel group is 16 bytes per position: 4 fp32 (TF32 path) or 8 fp16 (F16 path).
  int cg0, cg1;
  int B, D, H, W;            // input extent
  const float *wpack;        // [8 parity][T ztap][nchunk][T*T taps][2 kcore][NPAD/8][8][4]
  const float *scale, *shift;  // per output channel (NPAD entries): y = act(acc * scale + shift)
  float slope;               // LeakyReLU slope (1 = identity)
  float *out;                // blocked [B*2D][cgo][2H][2W][4]
  int cgo;                   // output channel groups
  int base[2];               // input index = j + base[par] - t
  int xtiles;                // the CTA tile is 8*MT positions wide; W = xtiles * 8 * MT (set by the launcher)
  int act_sigmoid = 0;       // MODE 4: apply a sigmoid after the bias
  int srcpar_cgs;            // 0, or: the K range is 8 parity sub-volumes of srcpar_cgs channel groups each (strided
                             // Conv3d k=4 s=2 p=1 after space-to-depth); sub-volume s = (pz,py,px) uses base 1 - p per dim
};

// ---- the kernel ----------------------------------------------------------------------------------------------
// T: taps per dimension of a parity class (K/2: 2 for k=4, 4 for k=8); NPAD: padded Cout (32 or 64); MT = W/8.
// X2: the fp32-accurate fp16 hi/lo operand split.  Activations arrive as [B*D][2 parts: hi, lo'][cg][H][W][8 fp16] with
// lo' = (a - hi) * 2^11, weights as [W_hi | W_lo'] side by side along N (lo' = (w - hi) * 2^11).  Per K step and tap:
//     A_hi  x [W_hi | W_lo']  ->  TMEM columns [0, 2*NPAD)         (one MMA, N = 2*NPAD)
//     A_lo' x  W_hi           ->  TMEM columns [NPAD, 2*NPAD)      (one MMA, N = NPAD)
// so the hi*hi products and the 2^11-scaled cross terms keep separate accumulators (the tensor core's fp32 accumulator
// truncates: a step's error scales with the partial sum it joins, and the cross terms would otherwise ride on the big one),
// and the epilogue returns acc_hi + 2^-11 * acc_cross.  2 MMAs per K step instead of the 3 of a K-expanded split.
// Halo: a channel group arrives as ONE cp.async.bulk.tensor (5-D tiled tensor map over [plane][cg][H][W][16 B], box
// [1][1][PY][PX][16 B], out-of-bounds elements zero-filled = the convolution's padding); each channel group starts on a
// 128-byte boundary of shared memory (the LBO of the A descriptor is that padded stride).
template <int T, int NPAD, int MT, bool X2 = false>
struct ConvTCfg {
  static constexpr int W = 8 * MT;
  static constexpr int PY = CT_BY + T - 1, PX = W + T - 1;     // halo extent
  static constexpr int PARTS = X2 ? 2 : 1;
  static constexpr int NACC = PARTS * NPAD;                    // accumulator columns per M-tile = width of the B operand
  static constexpr int A_CG_BYTES = PY * PX * 16;              // one channel group of the halo
  static constexpr int A_CG_STRIDE = ((A_CG_BYTES + 127) / 128) * 128;   // its pitch in shared memory = LBO of A
  static constexpr int A_BYTES = PARTS * CT_KCG * A_CG_STRIDE; // [part][channel group][halo]
  static constexpr int A_TX_BYTES = PARTS * CT_KCG * A_CG_BYTES;  // bytes the tensor copies of one stage deliver
  static constexpr int B_TAP_BYTES = 2 * (NACC / 8) * 128;     // one (y,x) tap: [2 kcore][NACC/8][8 rows][16 B]
  // A stage holds the halo of one (z tap, K chunk) and the weights of ROWS of its T tap rows; YS = T / ROWS (rounded up)
  // stages walk the same halo when all T*T taps do not fit twice into shared memory (X2 with 5x5 union taps: 128 KB).
  static constexpr int stage_bytes(int ys) { return ((A_BYTES + ((T + ys - 1) / ys) * T * B_TAP_BYTES + 127) / 128) * 128; }
  static constexpr int pick_ys() {
    for (int ys = 1; ys < T; ++ys)
      if (2 * stage_bytes(ys) <= 218 * 1024) return ys;
    return T;
  }
  static constexpr int YS = pick_ys();
  static constexpr int ROWS = (T + YS - 1) / YS;
  static constexpr int B_BYTES = ROWS * T * B_TAP_BYTES;
  static constexpr int STAGE_BYTES = stage_bytes(YS);
  static constexpr int TMEM_COLS = MT * NACC <= 32 ? 32 : MT * NACC <= 64 ? 64 : MT * NACC <= 128 ? 128 : MT * NACC <= 256 ? 256 : 512;
  // Two CTAs per SM whenever TMEM (<= 256 columns each) and shared memory (<= ~112 KB each) allow: one CTA's prologue
  // (TMEM alloc, pipeline fill) and epilogue (TMEM drain, stores) then overlap the other's MMA stream.
  static constexpr int S_ALONE = (218 * 1024) / STAGE_BYTES > 6 ? 6 : (218 * 1024) / STAGE_BYTES;
  static constexpr int S_PAIR = (112 * 1024) / STAGE_BYTES > 6 ? 6 : (112 * 1024) / STAGE_BYTES;
  static constexpr bool PAIR = TMEM_COLS <= 256 && S_PAIR >= 2;
  static constexpr int STAGES = PAIR ? S_PAIR : S_ALONE;
  static constexpr size_t SMEM = (size_t)STAGES * STAGE_BYTES + 256;
  static_assert(STAGES >= 2, "stage too large");
  static_assert(MT * NACC <= 512, "accumulators exceed TMEM");
  static_assert(NACC <= 256 && NACC % 16 == 0 && NPAD % 16 == 0 || !X2, "X2: MMA N must be a multiple of 16, at most 256");
};

// MODE 0: 8 parity classes (blockIdx.y), output at 2*j + parity (ConvTranspose3d stride 2); TZ = T = K/2 taps
// MODE 1: one class, output at j (stride-1 tap convolution; strided Conv3d arrives here after space-to-depth)
// MODE 2: ConvTranspose3d stride 2 with the four (y,x) parity classes MERGED along N (blockIdx.y = z parity): the
//         classes read the same halo at offsets that overlap in all but one tap per dimension, so one MMA over the
//         union of T = K/2 + 1 taps with N = 4 * Cout columns (n = (py*2+px)*Cout + co, zero weights where a class
//         does not use a tap) replaces four N = Cout MMAs.  An M128 MMA costs about the same 64+ cycles for any
//         N <= 128 (the A operand streams from shared memory at a fixed rate), so this is ~2.5x fewer tensor cycles.
//         TZ = K/2 z taps of the CTA's z parity.
// MODE 3: a stride-1 T-tap convolution whose N columns are the 8 output classes of a 2x upsampled grid
//         (n = ((qz*2+qy)*2+qx)*Cout + co, written to output position 2*j + q): a strided Conv3d(k 8, s 2, p 3) on
//         a 4x space-to-depth input (Unet_3D.enc1: 2 -> 128 channels, 3 taps, N = 8 x 20) - the same "few wide
//         MMAs instead of many narrow ones" trade as MODE 2, for a forward convolution.
// MODE 4: ConvTranspose3d(k 4, s 2, p 1) to ONE output channel (the last layer of every decoder): MODE 3's geometry with
//         N = 16 columns of which 8 are the output classes; the epilogue adds the bias (shift[0]), optionally applies
//         the sigmoid, and writes the NCDHW fp32 volume directly.
// OP: operand type: 0 = TF32 (fp32 storage), 1 = fp16, 2 = fp16 hi/lo split (X2, see ConvTCfg)
template <int TZ, int T, int NPAD, int MT, int MODE, int OP>
__global__ void __launch_bounds__(CT_THREADS, 1)
convt3d_s2_kernel(const ConvTParams p, const __grid_constant__ CUtensorMap tmap0, const __grid_constant__ CUtensorMap tmap1) {
  constexpr bool F16 = OP != 0, X2 = OP == 2;
  using Cfg = ConvTCfg<T, NPAD, MT, X2>;
  constexpr int NACC = Cfg::NACC;
  constexpr float LO_SCALE = 1.0f / 2048.0f;   // the cross-term accumulators hold 2^11 x their value
  constexpr bool PAR = MODE == 0, MERGE = MODE == 2, MERGE8 = MODE == 3, C1 = MODE == 4;
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t *stages = smem;
  uint64_t *full = reinterpret_cast<uint64_t *>(smem + (size_t)Cfg::STAGES * Cfg::STAGE_BYTES);
  uint64_t *empty = full + Cfg::STAGES;
  uint64_t *accum_full = empty + Cfg::STAGES;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(accum_full + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int par = blockIdx.y;  // parity class: bit 2 = z, bit 1 = y, bit 0 = x
  const int pz = MERGE ? par : (par >> 2) & 1, py = (par >> 1) & 1, px = par & 1;
  const int ytiles = p.H / CT_BY;
  const int xt = blockIdx.x % p.xtiles;
  const int tile = blockIdx.x / p.xtiles;
  const int yt = tile % ytiles;
  const int zj = (tile / ytiles) % p.D;
  const int b = tile / (ytiles * p.D);
  const int y0 = yt * CT_BY, x0 = xt * Cfg::W;
  const int nchunk = (p.cg0 + p.cg1) / CT_KCG;

  // Stage enumeration shared by the producer and the MMA issuer: q = tz * nchunk + kc, skipped when the z tap plane
  // of that K chunk lies outside the input (it contributes nothing).  The per-dimension base offset of a chunk is
  // uniform (parity class / plain convolution) or a function of the chunk's source sub-volume (strided conv).
  auto stage_of = [&](int q, int &tz, int &kc, int &ys, int &bz, int &by, int &bx) -> bool {
    ys = q % Cfg::YS;
    const int qq = q / Cfg::YS;
    tz = qq / nchunk;
    kc = qq - tz * nchunk;
    if (p.srcpar_cgs) {
      const int sv = ((kc * CT_KCG) / p.srcpar_cgs) & 7;  // & 7: the K range may hold several blocks of 8 sub-volumes (3xTF32)
      bz = 1 - ((sv >> 2) & 1);
      by = 1 - ((sv >> 1) & 1);
      bx = 1 - (sv & 1);
    } else {
      bz = p.base[pz];
      by = MERGE ? T / 2 : p.base[py];
      bx = MERGE ? T / 2 : p.base[px];
    }
    const int zi = zj + bz - tz;
    return zi >= 0 && zi < p.D;
  };
  const int n_q = TZ * nchunk * Cfg::YS;

  if (tid == 0) {
    for (int s = 0; s < Cfg::STAGES; ++s) {
      mbar_init(&full[s], 1);   // the one expect_tx arrival (halo + weight bytes)
      mbar_init(&empty[s], 1);  // the tcgen05.commit of the MMAs that read the slot
    }
    mbar_init(accum_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 4) {  // TMEM allocation is warp-wide
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "n"(Cfg::TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 4) {
    // ===================== producer: ONE thread issues the tensor copies of every stage ==========================
    if (tid == 0) {
      int it = 0;
      for (int q = 0; q < n_q; ++q) {
        int tz, kc, ys, bz, by, bx;
        if (!stage_of(q, tz, kc, ys, bz, by, bx)) continue;
        const int s = it % Cfg::STAGES, use = it / Cfg::STAGES;
        ++it;
        if (use > 0) mbar_wait(&empty[s], (use - 1) & 1);
        uint8_t *sa = stages + (size_t)s * Cfg::STAGE_BYTES;
        // weights of tap rows [ys*ROWS, ...) of this (class, z tap, K chunk): a contiguous slice of its T*T-tap block
        const int rows = (ys + 1) * Cfg::ROWS <= T ? Cfg::ROWS : T - ys * Cfg::ROWS;
        const uint32_t wbytes = (uint32_t)(rows * T * Cfg::B_TAP_BYTES);
        const float *wsrc = p.wpack + ((((size_t)par * TZ + tz) * nchunk + kc) * (size_t)(T * T * Cfg::B_TAP_BYTES / 4)) +
                            (size_t)ys * Cfg::ROWS * T * (Cfg::B_TAP_BYTES / 4);
        mbar_arrive_expect_tx(&full[s], wbytes + (uint32_t)Cfg::A_TX_BYTES);
        bulk_g2s(sa + Cfg::A_BYTES, wsrc, wbytes, &full[s]);
        const int zi = zj + bz - tz;
        const int gy0 = y0 + by - (T - 1), gx0 = x0 + bx - (T - 1);  // halo row r holds input row gy0 + r
#pragma unroll
        for (int part = 0; part < Cfg::PARTS; ++part) {
#pragma unroll
          for (int c = 0; c < CT_KCG; ++c) {
            int cg = kc * CT_KCG + c;
            const CUtensorMap *tm = &tmap0;
            if (cg >= p.cg0) { cg -= p.cg0; tm = &tmap1; }
            tma_load_5d(sa + (part * CT_KCG + c) * Cfg::A_CG_STRIDE, tm, gx0, gy0, cg, (b * p.D + zi) * Cfg::PARTS + part, &full[s]);
          }
        }
      }
    }
    // ===================== epilogue: TMEM -> registers -> act(acc*scale+shift) -> blocked global store =========
    mbar_wait(accum_full, 0);
    tc_fence_after();
    const int m = warp * 32 + lane;  // accumulator row = TMEM lane
    const int yy = m >> 3, xx = m & 7;
    constexpr bool UP = PAR || MERGE || MERGE8 || C1;
    const int Ho = UP ? 2 * p.H : p.H, Wo = UP ? 2 * p.W : p.W, Do = UP ? 2 * p.D : p.D;
    const int oz_plain = UP ? 2 * zj + pz : zj, oy = PAR ? 2 * (y0 + yy) + py : y0 + yy;
    if constexpr (C1) {
      const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16);
      const float bias = __ldg(p.shift);
#pragma unroll
      for (int mt = 0; mt < MT; ++mt) {
        float v[8];
        tmem_ld8(trow + (uint32_t)(mt * NACC), v);
        if constexpr (X2) {
          float l[8];
          tmem_ld8(trow + (uint32_t)(mt * NACC + NPAD), l);
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] = fmaf(l[i], LO_SCALE, v[i]);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          v[i] += bias;
          if (p.act_sigmoid) v[i] = 1.0f / (1.0f + __expf(-v[i]));
        }
        const int oxb = 2 * (x0 + 8 * mt + xx);
#pragma unroll
        for (int qzy = 0; qzy < 4; ++qzy) {
          float *dst = p.out + (((size_t)b * Do + 2 * zj + (qzy >> 1)) * Ho + 2 * (y0 + yy) + (qzy & 1)) * (size_t)Wo + oxb;
          *reinterpret_cast<float2 *>(dst) = make_float2(v[qzy * 2], v[qzy * 2 + 1]);
        }
      }
    } else if constexpr (MERGE || MERGE8) {
      constexpr int NZ = MERGE8 ? 2 : 1;      // z classes held by this CTA's accumulators
      constexpr int CP = NPAD / (4 * NZ);     // output channels per class
      static_assert(CP % 4 == 0, "merged classes must be whole channel groups");
      const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16);
#pragma unroll
      for (int mt = 0; mt < MT; ++mt) {
        const int oxb = 2 * (x0 + 8 * mt + xx);
#pragma unroll
        for (int qzy = 0; qzy < 2 * NZ; ++qzy) {
          const int qz = MERGE8 ? qzy >> 1 : 0, qy = qzy & 1;
          const int oyy = 2 * (y0 + yy) + qy;
          const int oz = MERGE8 ? 2 * zj + qz : 2 * zj + pz;
#pragma unroll
          for (int cgo = 0; cgo < CP / 4; ++cgo) {
            if (cgo >= p.cgo) continue;  // uniform across the CTA
            float v[8];
            tmem_ld4x2(trow + (uint32_t)(mt * NACC + (qzy * 2) * CP + cgo * 4),
                       trow + (uint32_t)(mt * NACC + (qzy * 2 + 1) * CP + cgo * 4), v);
            if constexpr (X2) {
              float l[8];
              tmem_ld4x2(trow + (uint32_t)(mt * NACC + NPAD + (qzy * 2) * CP + cgo * 4),
                         trow + (uint32_t)(mt * NACC + NPAD + (qzy * 2 + 1) * CP + cgo * 4), l);
#pragma unroll
              for (int i = 0; i < 8; ++i) v[i] = fmaf(l[i], LO_SCALE, v[i]);
            }
            float4 o[2];
#pragma unroll
            for (int qx = 0; qx < 2; ++qx) {
              float *po = &o[qx].x;
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int n = cgo * 4 + e;
                const float t = fmaf(v[qx * 4 + e], __ldg(p.scale + n), __ldg(p.shift + n));
                po[e] = t > 0.0f ? t : t * p.slope;
              }
            }
            float *dst = p.out + (((((size_t)b * Do + oz) * p.cgo + cgo) * Ho + oyy) * (size_t)Wo + oxb) * 4;
            *reinterpret_cast<float4 *>(dst) = o[0];
            *reinterpret_cast<float4 *>(dst + 4) = o[1];
          }
        }
      }
    } else {
#pragma unroll
    for (int mt = 0; mt < MT; ++mt) {
      const int ox = PAR ? 2 * (x0 + 8 * mt + xx) + px : x0 + 8 * mt + xx;
#pragma unroll
      for (int nb = 0; nb < NPAD / 32; ++nb) {
        float v[32];
        tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(mt * NACC + nb * 32), v);
        if constexpr (X2) {
          float l[32];
          tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(mt * NACC + NPAD + nb * 32), l);
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = fmaf(l[i], LO_SCALE, v[i]);
        }
#pragma unroll
        for (int g4 = 0; g4 < 8; ++g4) {
          const int cgo = nb * 8 + g4;
          if (cgo < p.cgo) {
            float4 o;
            float *po = &o.x;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int n = cgo * 4 + e;
              float t = fmaf(v[g4 * 4 + e], __ldg(p.scale + n), __ldg(p.shift + n));
              po[e] = t > 0.0f ? t : t * p.slope;
            }
            float *dst = p.out + (((((size_t)b * Do + oz_plain) * p.cgo + cgo) * Ho + oy) * (size_t)Wo + ox) * 4;
            *reinterpret_cast<float4 *>(dst) = o;
          }
        }
      }
    }
    }
    tc_fence_before();
  } else if (lane == 0) {
    // ===================== MMA issuer (one thread) =============================================================
    constexpr uint32_t idesc = F16 ? umma_idesc_f16(128, NACC) : umma_idesc_tf32(128, NACC);
    constexpr uint32_t idesc_lo = umma_idesc_f16(128, NPAD);   // X2: A_lo' x W_hi, the first NPAD columns of the same B tile
    bool first = true;
    int it = 0;
    for (int q = 0; q < n_q; ++q) {
      int tz, kc, ys, bz, by, bx;
      if (!stage_of(q, tz, kc, ys, bz, by, bx)) continue;
      const int s = it % Cfg::STAGES, use = it / Cfg::STAGES;
      ++it;
      mbar_wait(&full[s], use & 1);
      tc_fence_after();
      const uint32_t sa = smem_u32(stages + (size_t)s * Cfg::STAGE_BYTES);
      const uint32_t sb = sa + Cfg::A_BYTES;
      const int ty0 = ys * Cfg::ROWS;
#pragma unroll
      for (int r = 0; r < Cfg::ROWS; ++r) {
        const int ty = ty0 + r;
        if (ty >= T) break;
#pragma unroll
        for (int tx = 0; tx < T; ++tx) {
          const uint64_t bdesc = umma_desc(sb + (r * T + tx) * Cfg::B_TAP_BYTES, (NACC / 8) * 128, 128);
#pragma unroll
          for (int mt = 0; mt < MT; ++mt) {
            // rows of this M-tile under tap (ty,tx): halo row (T-1-ty) + y, column (T-1-tx) + 8*mt + x
            const uint32_t a0 = sa + (((T - 1 - ty) * Cfg::PX) + (T - 1 - tx) + 8 * mt) * 16;
            const uint64_t adesc = umma_desc(a0, Cfg::A_CG_STRIDE, Cfg::PX * 16);
            const bool acc = !first || (r | tx);
            if (F16) umma_f16(tmem_base + mt * NACC, adesc, bdesc, idesc, acc);
            else umma_tf32(tmem_base + mt * NACC, adesc, bdesc, idesc, acc);
            if constexpr (X2) {
              const uint64_t adesc_lo = umma_desc(a0 + CT_KCG * Cfg::A_CG_STRIDE, Cfg::A_CG_STRIDE, Cfg::PX * 16);
              umma_f16(tmem_base + mt * NACC + NPAD, adesc_lo, bdesc, idesc_lo, true);
            }
          }
        }
      }
      first = false;
      umma_commit(&empty[s]);  // frees the slot when the MMAs that read it are done (implies fence::before_thread_sync)
    }
    umma_commit(accum_full);
  }
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(Cfg::TMEM_COLS) : "memory");
  }
}

// ---- tensor maps of the activation operands (host) ------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn tmap_encoder() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void *p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
    cudaGetLastError();
  }
  return fn;
}
// blocked activations [planes][ncg][H][W][16 B] as a 5-D map of 4-byte elements (4, W, H, ncg, planes); box = one channel
// group's halo (4, PX, PY, 1, 1); elements outside [0,W) x [0,H) are delivered as zeros
static bool make_halo_tmap(EncodeTiledFn enc, CUtensorMap *m, const void *base, long long planes, int ncg, int H, int W, int PX,
                           int PY) {
  if (!base || ncg <= 0) return false;
  const cuuint64_t gdim[5] = {4, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)ncg, (cuuint64_t)planes};
  const cuuint64_t gstr[4] = {16, (cuuint64_t)W * 16, (cuuint64_t)H * W * 16, (cuuint64_t)ncg * H * W * 16};
  const cuuint32_t box[5] = {4, (cuuint32_t)PX, (cuuint32_t)PY, 1, 1};
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_UINT32, 5, const_cast<void *>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
template <int TZ, int T, int NPAD, int MT, int MODE, int OP>
static int launch_convt_variant(const ConvTParams &p, cudaStream_t st) {
  using Cfg = ConvTCfg<T, NPAD, MT, OP == 2>;
  auto kern = convt3d_s2_kernel<TZ, T, NPAD, MT, MODE, OP>;
  static bool configured[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!configured[dev & 63]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM);
    if (e != cudaSuccess) {
      set_error("convt3d: cudaFuncSetAttribute(%zu bytes): %s", Cfg::SMEM, cudaGetErrorString(e));
      return (int)e;
    }
    configured[dev & 63] = true;
  }
  ConvTParams q = p;
  q.xtiles = p.W / Cfg::W;
  if (q.xtiles < 1 || q.xtiles * Cfg::W != p.W) return fail_arg(GENRE_B200_EINVAL, "convt3d: W=%d is not a multiple of the %d-wide tile", p.W, Cfg::W);
  const EncodeTiledFn enc = tmap_encoder();
  if (!enc) return fail_arg(GENRE_B200_EINVAL, "convt3d: the CUDA driver does not provide cuTensorMapEncodeTiled");
  CUtensorMap tm0, tm1;
  memset(&tm0, 0, sizeof(tm0));
  memset(&tm1, 0, sizeof(tm1));
  const long long planes = (long long)p.B * p.D * Cfg::PARTS;
  if (!make_halo_tmap(enc, &tm0, p.src0, planes, p.cg0, p.H, p.W, Cfg::PX, Cfg::PY))
    return fail_arg(GENRE_B200_EINVAL, "convt3d: cuTensorMapEncodeTiled failed for the first operand");
  if (p.cg1 > 0 && !make_halo_tmap(enc, &tm1, p.src1, planes, p.cg1, p.H, p.W, Cfg::PX, Cfg::PY))
    return fail_arg(GENRE_B200_EINVAL, "convt3d: cuTensorMapEncodeTiled failed for the second operand");
  dim3 grid((unsigned)(p.B * p.D * (p.H / CT_BY) * q.xtiles), MODE == 0 ? 8 : MODE == 2 ? 2 : 1);
  kern<<<grid, CT_THREADS, Cfg::SMEM, st>>>(q, tm0, tm1);
  return check_launch("convt3d_s2 kernel");
}

static thread_local int g_conv_op = 0;  // operand type of the next launch (set by the C ABI entry points): 0 TF32, 1 fp16, 2 fp16 hi/lo
// X2 doubles the accumulator columns: halve the M-tiles per CTA until MT * 2 * NPAD fits the 512 TMEM columns
template <int TZ, int T, int NPAD, int MT, int MODE>
static int launch_convt_x2(const ConvTParams &p, cudaStream_t st) {
  if constexpr (NPAD % 16 != 0 || 2 * NPAD > 256) {
    return fail_arg(GENRE_B200_EINVAL, "convt3d: the fp16 hi/lo mode needs N = %d to be a multiple of 16, at most 128", NPAD);
  } else if constexpr (MT * 2 * NPAD > 512) {
    return launch_convt_x2<TZ, T, NPAD, MT / 2, MODE>(p, st);
  } else {
    return launch_convt_variant<TZ, T, NPAD, MT, MODE, 2>(p, st);
  }
}
template <int TZ, int T, int NPAD, int MT, int MODE>
static int launch_convt_op(const ConvTParams &p, cudaStream_t st) {
  if (g_conv_op == 2) return launch_convt_x2<TZ, T, NPAD, MT, MODE>(p, st);
  return g_conv_op == 1 ? launch_convt_variant<TZ, T, NPAD, MT, MODE, 1>(p, st) : launch_convt_variant<TZ, T, NPAD, MT, MODE, 0>(p, st);
}
template <int T, int NPAD, int MT, bool PAR>
static int launch_convt(const ConvTParams &p, cudaStream_t st) {
  return launch_convt_op<T, T, NPAD, MT, PAR ? 0 : 1>(p, st);
}
template <int TZ, int T, int NPAD, int MT>
static int launch_convt_merged(const ConvTParams &p, cudaStream_t st) {
  return launch_convt_op<TZ, T, NPAD, MT, 2>(p, st);
}
template <int MT>
static int launch_convt_c1(const ConvTParams &p, cudaStream_t st) {
  if (g_conv_op == 2)   // not routed (ops_conv.convt_c1_tc): the exact FP32-pipe stencil serves the fp32-accurate modes
    return fail_arg(GENRE_B200_EINVAL, "convt_c1_tc: the fp16 hi/lo operand mode is not supported for the 1-channel layer");
  return g_conv_op == 1 ? launch_convt_variant<3, 3, 16, MT, 4, 1>(p, st) : launch_convt_variant<3, 3, 16, MT, 4, 0>(p, st);
}
template <int T, int NPAD, int MT>
static int launch_conv_merged8(const ConvTParams &p, cudaStream_t st) {
  return launch_convt_op<T, T, NPAD, MT, 3>(p, st);
}

}  // namespace gb

using namespace gb;

// ConvTranspose3d(kernel K in {4, 8}, stride 2, padding K/2 - 1) forward on channel-blocked activations.
//   src0 [B*D][cg0][H][W][4], src1 [B*D][cg1][H][W][4] or NULL: the two halves of the channel concatenation
//   wpack: weights packed by genre_shapehd_b200.ops_conv.pack_convt_weights (layout in the kernel header)
//   scale, shift [npad]: per-channel affine applied to the accumulator (bias and folded eval-mode BatchNorm),
//   slope: LeakyReLU slope (1 = none).   out [B*2D][cgo][2H][2W][4]
// Supported: W in {16, 32}, H % 16 == 0, cg0 + cg1 even, 4*cgo <= npad, npad in {32, 64}.
extern "C" int genre_b200_convt3d_s2_forward(const void *src0_, int cg0, const void *src1_, int cg1, int64_t B,
                                             int64_t D, int64_t H, int64_t W, const void *wpack_, int ksize, int npad,
                                             int f16, const float *scale, const float *shift, float slope, float *out,
                                             int cgo, void *stream) {
  const float *src0 = (const float *)src0_, *src1 = (const float *)src1_, *wpack = (const float *)wpack_;
  g_conv_op = f16;
  GB_REQUIRE(src0 && wpack && scale && shift && out, GENRE_B200_EINVAL, "convt3d: null pointer");
  GB_REQUIRE(ksize == 4 || ksize == 8, GENRE_B200_EINVAL, "convt3d: kernel size %d unsupported (4 or 8)", ksize);
  GB_REQUIRE(npad == 32 || npad == 64, GENRE_B200_EINVAL, "convt3d: npad %d unsupported (32 or 64)", npad);
  GB_REQUIRE(W == 16 || W == 32, GENRE_B200_EINVAL, "convt3d: input width %lld unsupported (16 or 32)", (long long)W);
  GB_REQUIRE(H % CT_BY == 0 && H > 0 && D > 0 && B > 0, GENRE_B200_EINVAL, "convt3d: bad extent");
  GB_REQUIRE(cg0 > 0 && cg1 >= 0 && (cg0 + cg1) % CT_KCG == 0 && (cg1 == 0 || src1), GENRE_B200_EINVAL,
             "convt3d: channel groups (%d + %d) must be even in total", cg0, cg1);
  GB_REQUIRE(cgo > 0 && 4 * cgo <= npad, GENRE_B200_EINVAL, "convt3d: %d output channels exceed npad %d", 4 * cgo, npad);
  GB_REQUIRE(B * D * (H / CT_BY) < (1ll << 31), GENRE_B200_EINVAL, "convt3d: grid too large");
  GB_REQUIRE(aligned16(src0) && aligned16(wpack) && aligned16(out) && (!src1 || aligned16(src1)), GENRE_B200_EALIGN,
             "convt3d: buffers must be 16-byte aligned");
  ConvTParams p;
  p.src0 = src0; p.src1 = src1; p.cg0 = cg0; p.cg1 = cg1;
  p.B = (int)B; p.D = (int)D; p.H = (int)H; p.W = (int)W;
  p.wpack = wpack; p.scale = scale; p.shift = shift; p.slope = slope; p.out = out; p.cgo = cgo;
  p.srcpar_cgs = 0;
  const int pad = ksize / 2 - 1;
  for (int par = 0; par < 2; ++par) {
    const int k0 = (par + pad) % 2;
    p.base[par] = (par + pad - k0) / 2;
  }
  cudaStream_t st = as_stream(stream);
  const int T = ksize / 2;
#define GB_CT(TT, NN, MM) return launch_convt<TT, NN, MM, true>(p, st)
  if (T == 4 && npad == 32 && W == 32) GB_CT(4, 32, 4);
  if (T == 4 && npad == 32 && W == 16) GB_CT(4, 32, 2);
  if (T == 2 && npad == 32 && W == 32) GB_CT(2, 32, 4);
  if (T == 2 && npad == 32 && W == 16) GB_CT(2, 32, 2);
  if (T == 2 && npad == 64 && W == 32) GB_CT(2, 64, 4);
  if (T == 2 && npad == 64 && W == 16) GB_CT(2, 64, 2);
  if (T == 4 && npad == 64 && W == 32) GB_CT(4, 64, 4);
  if (T == 4 && npad == 64 && W == 16) GB_CT(4, 64, 2);
#undef GB_CT
  return fail_arg(GENRE_B200_EINVAL, "convt3d: no kernel instance for k=%d npad=%d W=%lld", ksize, npad, (long long)W);
}

// ConvTranspose3d(kernel 8, stride 2, padding 3) with the four (y,x) output parity classes merged along N (kernel MODE 2):
// the layer that dominates Unet_3D, dec5 = ConvT(80 -> 20) on 32^3 (networks/networks.py:166).  Same operands as
// genre_b200_convt3d_s2_forward except
//   wpack [2 z-parity][4 z-tap][Cin chunk][5*5 union taps][2][npad/8][8][g], npad = 4 * cpad columns ordered
//         n = (py*2+px)*cpad + co  (ops_conv.pack_convt_merged_weights);  scale, shift [cpad].
// Supported: ksize 8, npad = 80 (Cout <= 20), W = 16 or a multiple of 32, H % 16 == 0.
extern "C" int genre_b200_convt3d_s2_merged_forward(const void *src0_, int cg0, const void *src1_, int cg1, int64_t B,
                                                    int64_t D, int64_t H, int64_t W, const void *wpack_, int ksize,
                                                    int npad, int f16, const float *scale, const float *shift,
                                                    float slope, float *out, int cgo, void *stream) {
  const float *src0 = (const float *)src0_, *src1 = (const float *)src1_, *wpack = (const float *)wpack_;
  g_conv_op = f16;
  GB_REQUIRE(src0 && wpack && scale && shift && out, GENRE_B200_EINVAL, "convt3d_merged: null pointer");
  GB_REQUIRE(ksize == 8, GENRE_B200_EINVAL, "convt3d_merged: kernel size %d unsupported (8)", ksize);
  GB_REQUIRE(npad == 80, GENRE_B200_EINVAL, "convt3d_merged: npad %d unsupported (80 = 4 classes x 20 channels)", npad);
  GB_REQUIRE(W == 16 || (W > 0 && W % 32 == 0), GENRE_B200_EINVAL,
             "convt3d_merged: input width %lld unsupported (16, or a multiple of 32 walked in 32-wide tiles)", (long long)W);
  GB_REQUIRE(H % CT_BY == 0 && H > 0 && D > 0 && B > 0, GENRE_B200_EINVAL, "convt3d_merged: bad extent");
  GB_REQUIRE(cg0 > 0 && cg1 >= 0 && (cg0 + cg1) % CT_KCG == 0 && (cg1 == 0 || src1), GENRE_B200_EINVAL,
             "convt3d_merged: channel groups (%d + %d) must be even in total", cg0, cg1);
  GB_REQUIRE(cgo > 0 && 16 * cgo <= npad, GENRE_B200_EINVAL, "convt3d_merged: %d output channels exceed npad/4", 4 * cgo);
  GB_REQUIRE(B * D * (H / CT_BY) < (1ll << 31), GENRE_B200_EINVAL, "convt3d_merged: grid too large");
  GB_REQUIRE(aligned16(src0) && aligned16(wpack) && aligned16(out) && (!src1 || aligned16(src1)), GENRE_B200_EALIGN,
             "convt3d_merged: buffers must be 16-byte aligned");
  ConvTParams p;
  p.src0 = src0; p.src1 = src1; p.cg0 = cg0; p.cg1 = cg1;
  p.B = (int)B; p.D = (int)D; p.H = (int)H; p.W = (int)W;
  p.wpack = wpack; p.scale = scale; p.shift = shift; p.slope = slope; p.out = out; p.cgo = cgo;
  p.srcpar_cgs = 0;
  const int pad = ksize / 2 - 1;
  for (int par = 0; par < 2; ++par) {
    const int k0 = (par + pad) % 2;
    p.base[par] = (par + pad - k0) / 2;
  }
  cudaStream_t st = as_stream(stream);
  if (W % 32 == 0) return launch_convt_merged<4, 5, 80, 4>(p, st);  // 32-wide x tiles
  return launch_convt_merged<4, 5, 80, 2>(p, st);
}

// Conv3d(kernel 8, stride 2, padding 3), few input channels, Cout <= 20, on a 4x space-to-depth input (kernel MODE 3):
// Unet_3D.enc1 = Conv3d(2 -> 20) on 128^3 (networks/networks.py:151).
//   src [B*D][cg][H][W][16 B]: D,H,W = input extent / 4, channels ((c*4+rz)*4+ry)*4+rx (genre_b200_ncdhw_to_blocked mode 3)
//   wpack [3 z-tap][chunk][9 taps][2][npad/8][8][g], npad = 160 columns n = ((qz*2+qy)*2+qx)*20 + co
//         (ops_conv.pack_conv_k8s2_s4d_weights);  scale, shift [20];  out [B*2D][cgo][2H][2W][4] fp32
// Supported: W % 16 == 0, H % 16 == 0, cg even.
extern "C" int genre_b200_conv3d_k8s2_s4d_forward(const void *src_, int cg, int64_t B, int64_t D, int64_t H, int64_t W,
                                                  const void *wpack_, int npad, int f16, const float *scale,
                                                  const float *shift, float slope, float *out, int cgo, void *stream) {
  const float *src = (const float *)src_, *wpack = (const float *)wpack_;
  g_conv_op = f16;
  GB_REQUIRE(src && wpack && scale && shift && out, GENRE_B200_EINVAL, "conv3d_k8s2_s4d: null pointer");
  GB_REQUIRE(npad == 160 || npad == 80, GENRE_B200_EINVAL,
             "conv3d_k8s2_s4d: npad %d unsupported (160 = 8 classes x 20 channels, or 80 = 4 (y,x) classes per z class)", npad);
  GB_REQUIRE(W > 0 && W % 16 == 0 && H > 0 && H % CT_BY == 0 && D > 0 && B > 0, GENRE_B200_EINVAL, "conv3d_k8s2_s4d: bad extent");
  GB_REQUIRE(cg > 0 && cg % CT_KCG == 0, GENRE_B200_EINVAL, "conv3d_k8s2_s4d: channel groups must be even");
  GB_REQUIRE(cgo > 0 && cgo <= 5, GENRE_B200_EINVAL, "conv3d_k8s2_s4d: too many output channels");
  GB_REQUIRE(B * D * (H / CT_BY) * (W / 16) < (1ll << 31), GENRE_B200_EINVAL, "conv3d_k8s2_s4d: grid too large");
  GB_REQUIRE(aligned16(src) && aligned16(wpack) && aligned16(out), GENRE_B200_EALIGN, "conv3d_k8s2_s4d: alignment");
  ConvTParams p;
  p.src0 = src; p.src1 = nullptr; p.cg0 = cg; p.cg1 = 0;
  p.B = (int)B; p.D = (int)D; p.H = (int)H; p.W = (int)W;
  p.wpack = wpack; p.scale = scale; p.shift = shift; p.slope = slope; p.out = out; p.cgo = cgo;
  p.srcpar_cgs = 0;
  p.base[0] = p.base[1] = 1;  // input cell = j + 1 - t
  // npad 80: the z class moves to blockIdx.y (MODE 2 with 3 z taps per class; wpack [2 qz][3][chunk][9][2][10][8][g]):
  // twice the MMAs of the 8-class form, but 256 TMEM columns and half the weight bytes per stage let two CTAs share an SM
  if (npad == 80) return launch_convt_merged<3, 3, 80, 2>(p, as_stream(stream));
  return launch_conv_merged8<3, 160, 2>(p, as_stream(stream));
}

// ConvTranspose3d(Cin -> 1, k 4, s 2, p 1) on the tensor cores (kernel MODE 4): the last layer of every decoder
// (Unet_3D.dec6 networks/networks.py:167-168, VoxelDecoder main.17 :57, VoxelGenerator :98).  3 union taps per dimension,
// the 8 output classes as N columns.
//   src0/src1 blocked operands [B*D][cg][H][W][16 B] (two halves of a skip concatenation; src1 may be NULL)
//   wpack [3][chunk][9][2][2][8][g] (ops_conv.pack_convt_c1_tc_weights), bias, act_sigmoid;  out [B][2D][2H][2W] fp32
// Supported: W in {16, 32, 64}, H % 16 == 0, cg0 + cg1 even.
extern "C" int genre_b200_convt_c1_tc_forward(const void *src0_, int cg0, const void *src1_, int cg1, int64_t B, int64_t D,
                                              int64_t H, int64_t W, const void *wpack_, int f16, const float *bias,
                                              int act_sigmoid, float *out, void *stream) {
  const float *src0 = (const float *)src0_, *src1 = (const float *)src1_, *wpack = (const float *)wpack_;
  g_conv_op = f16;
  GB_REQUIRE(src0 && wpack && bias && out, GENRE_B200_EINVAL, "convt_c1_tc: null pointer");
  GB_REQUIRE(W == 16 || W == 32 || W == 64, GENRE_B200_EINVAL, "convt_c1_tc: input width %lld unsupported", (long long)W);
  GB_REQUIRE(H % CT_BY == 0 && H > 0 && D > 0 && B > 0, GENRE_B200_EINVAL, "convt_c1_tc: bad extent");
  GB_REQUIRE(cg0 > 0 && cg1 >= 0 && (cg0 + cg1) % CT_KCG == 0 && (cg1 == 0 || src1), GENRE_B200_EINVAL,
             "convt_c1_tc: channel groups (%d + %d) must be even in total", cg0, cg1);
  GB_REQUIRE(B * D * (H / CT_BY) < (1ll << 31), GENRE_B200_EINVAL, "convt_c1_tc: grid too large");
  GB_REQUIRE(aligned16(src0) && aligned16(wpack) && ((uintptr_t)out & 7) == 0 && (!src1 || aligned16(src1)), GENRE_B200_EALIGN,
             "convt_c1_tc: alignment");
  ConvTParams p;
  p.src0 = src0; p.src1 = src1; p.cg0 = cg0; p.cg1 = cg1;
  p.B = (int)B; p.D = (int)D; p.H = (int)H; p.W = (int)W;
  p.wpack = wpack; p.scale = bias; p.shift = bias; p.slope = 1.0f; p.out = out; p.cgo = 1;
  p.srcpar_cgs = 0;
  p.act_sigmoid = act_sigmoid;
  p.base[0] = p.base[1] = 1;
  cudaStream_t st = as_stream(stream);
  if (W == 64) return launch_convt_c1<8>(p, st);
  if (W == 32) return launch_convt_c1<4>(p, st);
  return launch_convt_c1<2>(p, st);
}

// Stride-1 convolution with T taps per dimension on channel-blocked activations (same kernel, one output class):
//     out[b, z, y, x, n] = act(scale[n] * sum_{tz,ty,tx,c} in[b, z + base - tz, y + base - ty, x + base - tx, c] * Wt[...] + shift[n])
// A strided Conv3d reaches this form through space-to-depth (genre_shapehd_b200/ops_conv.py): Unet_3D.enc1 =
// Conv3d(2 -> 20, k=8, s=2, p=3) (networks/networks.py:151) is a 5-tap stride-1 convolution over the 16 s2d channels.
//   wpack [T z-tap][C/8 chunk][T*T taps][2][npad/8][8][4];  out [B*D][cgo][H][W][4]
// Supported: T in {3, 5}, W in {16, 32, 64}, H % 16 == 0, npad = 32 (or 64 with T = 3, 96 with T = 5).
extern "C" int genre_b200_conv3d_taps_forward(const void *src0_, int cg0, const void *src1_, int cg1, int64_t B,
                                              int64_t D, int64_t H, int64_t W, const void *wpack_, int taps, int base,
                                              int npad, int f16, const float *scale, const float *shift, float slope,
                                              float *out, int cgo, void *stream) {
  const float *src0 = (const float *)src0_, *src1 = (const float *)src1_, *wpack = (const float *)wpack_;
  g_conv_op = f16;
  GB_REQUIRE(src0 && wpack && scale && shift && out, GENRE_B200_EINVAL, "conv3d_taps: null pointer");
  GB_REQUIRE(taps == 3 || taps == 5, GENRE_B200_EINVAL, "conv3d_taps: %d taps unsupported (3 or 5)", taps);
  GB_REQUIRE(npad == 32 || (npad == 64 && taps == 3) || (npad == 96 && taps == 5), GENRE_B200_EINVAL,
             "conv3d_taps: npad %d unsupported (32; 64 with 3 taps; 96 with 5 taps)", npad);
  GB_REQUIRE(W == 16 || W == 32 || W == 64, GENRE_B200_EINVAL, "conv3d_taps: width %lld unsupported", (long long)W);
  GB_REQUIRE(H % CT_BY == 0 && H > 0 && D > 0 && B > 0, GENRE_B200_EINVAL, "conv3d_taps: bad extent");
  GB_REQUIRE(cg0 > 0 && cg1 >= 0 && (cg0 + cg1) % CT_KCG == 0 && (cg1 == 0 || src1), GENRE_B200_EINVAL,
             "conv3d_taps: channel groups (%d + %d) must be even in total", cg0, cg1);
  GB_REQUIRE(cgo > 0 && 4 * cgo <= npad, GENRE_B200_EINVAL, "conv3d_taps: too many output channels");
  GB_REQUIRE(B * D * (H / CT_BY) < (1ll << 31), GENRE_B200_EINVAL, "conv3d_taps: grid too large");
  GB_REQUIRE(aligned16(src0) && aligned16(wpack) && aligned16(out) && (!src1 || aligned16(src1)), GENRE_B200_EALIGN,
             "conv3d_taps: buffers must be 16-byte aligned");
  ConvTParams p;
  p.src0 = src0; p.src1 = src1; p.cg0 = cg0; p.cg1 = cg1;
  p.B = (int)B; p.D = (int)D; p.H = (int)H; p.W = (int)W;
  p.wpack = wpack; p.scale = scale; p.shift = shift; p.slope = slope; p.out = out; p.cgo = cgo;
  p.srcpar_cgs = 0;
  p.base[0] = p.base[1] = base;
  cudaStream_t st = as_stream(stream);
  // 3 taps, N = 64: Conv3d(1 -> 64, k4, s2, p1) over the 2x space-to-depth input (VoxelDiscriminator's first layer);
  // 32-wide tiles (256 TMEM columns) so that two CTAs share an SM
  if (taps == 3 && npad == 64) {
    if (W % 32 == 0) return launch_convt<3, 64, 4, false>(p, st);
    return launch_convt<3, 64, 2, false>(p, st);
  }
  // 5 taps, N = 96: Conv3d(20 -> 80, k8, s2, p3) over the 2x space-to-depth input = the input gradient of Unet_3D.dec5
  // (ConvTranspose3d 80 -> 20); 32- or 16-wide tiles (384 / 192 TMEM columns)
  if (taps == 5 && npad == 96) {
    if (W % 32 == 0) return launch_convt<5, 96, 4, false>(p, st);
    return launch_convt<5, 96, 2, false>(p, st);
  }
#define GB_CV(TT, MM) return launch_convt<TT, 32, MM, false>(p, st)
  if (taps == 5 && W == 64) GB_CV(5, 8);
  if (taps == 5 && W == 32) GB_CV(5, 4);
  if (taps == 5 && W == 16) GB_CV(5, 2);
  if (taps == 3 && W == 64) GB_CV(3, 8);
  if (taps == 3 && W == 32) GB_CV(3, 4);
  if (taps == 3 && W == 16) GB_CV(3, 2);
#undef GB_CV
  return fail_arg(GENRE_B200_EINVAL, "conv3d_taps: no kernel instance");
}

// Conv3d(kernel 4, stride 2, padding 1) forward (VoxelDiscriminator networks/networks.py:247-250 conv3d_half, Unet_3D
// enc2..enc5 :152-155) on the same kernel: the input arrives as its 8 parity sub-volumes in ONE channel-blocked tensor
//   src [B*D'][8*cgs][H'][W'][16 B]   (D' = D/2 ...; channel group index = s*cgs + c, s = (pz*2+py)*2+px)
// and sub-volume s is a K range with 2 taps per dimension: in[2(o+delta)+p] with delta = (1-p) - t, k = 3 - 2t - p.
//   wpack [2 z-tap][kblocks*8*cgs/2 chunk][4 taps][2][npad/8][8][g];  out [B*D'][cgo][H'][W'][4] fp32
//   kblocks (1, or 3 for the hi|lo|hi operand of the 3xTF32 mode): how many such 8-sub-volume blocks the K range holds
// Supported: W' in {16, 32}, H' % 16 == 0, cgs even, npad in {32, 64, 96, 128}.
extern "C" int genre_b200_conv3d_k4s2_forward(const void *src_, int cgs, int kblocks, int64_t B, int64_t D, int64_t H,
                                              int64_t W, const void *wpack_, int npad, int f16, const float *scale,
                                              const float *shift, float slope, float *out, int cgo, void *stream) {
  const float *src = (const float *)src_, *wpack = (const float *)wpack_;
  g_conv_op = f16;
  GB_REQUIRE(src && wpack && scale && shift && out, GENRE_B200_EINVAL, "conv3d_k4s2: null pointer");
  GB_REQUIRE(npad == 32 || npad == 64 || npad == 96 || npad == 128, GENRE_B200_EINVAL, "conv3d_k4s2: npad %d", npad);
  GB_REQUIRE(W == 16 || W == 32, GENRE_B200_EINVAL, "conv3d_k4s2: output width %lld unsupported (16 or 32)", (long long)W);
  GB_REQUIRE(H % CT_BY == 0 && H > 0 && D > 0 && B > 0, GENRE_B200_EINVAL, "conv3d_k4s2: bad extent");
  GB_REQUIRE(cgs > 0 && cgs % CT_KCG == 0, GENRE_B200_EINVAL, "conv3d_k4s2: channel groups per sub-volume must be even");
  GB_REQUIRE(cgo > 0 && 4 * cgo <= npad, GENRE_B200_EINVAL, "conv3d_k4s2: too many output channels");
  GB_REQUIRE(B * D * (H / CT_BY) < (1ll << 31), GENRE_B200_EINVAL, "conv3d_k4s2: grid too large");
  GB_REQUIRE(aligned16(src) && aligned16(wpack) && aligned16(out), GENRE_B200_EALIGN, "conv3d_k4s2: alignment");
  ConvTParams p;
  p.src0 = src; p.src1 = nullptr; p.cg0 = 8 * cgs * (kblocks > 0 ? kblocks : 1); p.cg1 = 0;
  p.B = (int)B; p.D = (int)D; p.H = (int)H; p.W = (int)W;
  p.wpack = wpack; p.scale = scale; p.shift = shift; p.slope = slope; p.out = out; p.cgo = cgo;
  p.srcpar_cgs = cgs;
  p.base[0] = p.base[1] = 0;
  cudaStream_t st = as_stream(stream);
#define GB_CS(NN, MM) return launch_convt<2, NN, MM, false>(p, st)
  if (W == 32) {
    if (npad == 32) GB_CS(32, 4);
    if (npad == 64) GB_CS(64, 4);
    if (npad == 96) GB_CS(96, 4);
    if (npad == 128) GB_CS(128, 4);
  } else {
    if (npad == 32) GB_CS(32, 2);
    if (npad == 64) GB_CS(64, 2);
    if (npad == 96) GB_CS(96, 2);
    if (npad == 128) GB_CS(128, 2);
  }
#undef GB_CS
  return fail_arg(GENRE_B200_EINVAL, "conv3d_k4s2: no kernel instance");
}
