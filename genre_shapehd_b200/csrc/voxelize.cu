// voxelize.cu — workspace + splat stage of the voxelisation pipeline (see voxelize.cuh for the design).
#include "voxelize.cuh"

namespace gb {

// ------------------------------------------------------------------------------------------------
// workspace
// ------------------------------------------------------------------------------------------------
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

static size_t counters_words(int64_t n_maps, size_t nt) { return (size_t)n_maps * nt + (size_t)n_maps; }
static size_t counters_bytes(int64_t n_maps, size_t nt) { return align_up(counters_words(n_maps, nt) * 4, 256); }

size_t vox_workspace_bytes(int64_t n_maps, int64_t P, int res) {
  const size_t nt = (size_t)vox_ntiles(res);
  size_t b = counters_bytes(n_maps, nt);                         // counts + ovf_count (contiguous: one memset)
  b += align_up((size_t)n_maps * nt * VOX_BUCKET * 8, 256);      // buckets
  b += align_up((size_t)n_maps * P * 8, 256);                    // overflow lists
  return b;
}

bool vox_carve(void *ws, size_t ws_bytes, int64_t n_maps, int64_t P, int res, VoxWorkspace *out) {
  if (!ws || !aligned16(ws) || ws_bytes < vox_workspace_bytes(n_maps, P, res)) return false;
  const size_t nt = (size_t)vox_ntiles(res);
  char *p = (char *)ws;
  out->counts = (unsigned *)p;
  out->ovf_count = out->counts + (size_t)n_maps * nt;
  p += counters_bytes(n_maps, nt);
  out->buckets = (uint2 *)p;
  p += align_up((size_t)n_maps * nt * VOX_BUCKET * 8, 256);
  out->ovf = (uint2 *)p;
  out->ntiles = (int)nt;
  return true;
}

int vox_clear_counts(const VoxWorkspace &w, int64_t n_maps, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(w.counts, 0, counters_words(n_maps, (size_t)w.ntiles) * 4, st);
  if (e != cudaSuccess) {
    set_error("voxelize: clearing tile counters: %s", cudaGetErrorString(e));
    return (int)e;
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// splat: one CTA per output tile
// ------------------------------------------------------------------------------------------------
template <bool VEC, bool WRITE_CNT>
__global__ void __launch_bounds__(VOX_SPLAT_THREADS)
vox_splat_kernel(const SplatArgs a) {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  vox_splat_body<VEC, WRITE_CNT>(a, blockIdx.x, blockIdx.y);
}

template <bool VEC, bool WRITE_CNT>
static int launch_splat(const VoxWorkspace &w, int64_t n_maps, int64_t P, long long nvox, float *tdf, float *cnt,
                        float alpha, float beta, float bg, cudaStream_t st, bool pdl, long long out_stride) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)w.ntiles, (unsigned)n_maps);
  cfg.blockDim = dim3(VOX_SPLAT_THREADS);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;  // overlap this launch with the project kernel's tail
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;  // stand-alone launches (stage entry point, used for timing) keep plain stream ordering
  const SplatArgs a = vox_splat_args(w, P, nvox, tdf, cnt, alpha, beta, bg, out_stride);
  cudaError_t e = cudaLaunchKernelEx(&cfg, vox_splat_kernel<VEC, WRITE_CNT>, a);
  if (e != cudaSuccess) {
    set_error("voxelize splat kernel: %s", cudaGetErrorString(e));
    cudaGetLastError();
    return (int)e;
  }
  return check_launch("voxelize splat kernel");
}

int vox_splat(const VoxWorkspace &w, int64_t n_maps, int64_t P, int res, float *tdf, float *cnt, float alpha,
              float beta, float bg, cudaStream_t st, bool pdl, long long out_stride) {
  const long long nvox = (long long)res * res * res;
  if (out_stride <= 0) out_stride = nvox;
  const bool vec = (nvox % 4 == 0) && (out_stride % 4 == 0) && aligned16(tdf) && (!cnt || aligned16(cnt));
  if (vec) {
    return cnt ? launch_splat<true, true>(w, n_maps, P, nvox, tdf, cnt, alpha, beta, bg, st, pdl, out_stride)
               : launch_splat<true, false>(w, n_maps, P, nvox, tdf, cnt, alpha, beta, bg, st, pdl, out_stride);
  }
  return cnt ? launch_splat<false, true>(w, n_maps, P, nvox, tdf, cnt, alpha, beta, bg, st, pdl, out_stride)
             : launch_splat<false, false>(w, n_maps, P, nvox, tdf, cnt, alpha, beta, bg, st, pdl, out_stride);
}

// arguments shared by both back-projections
int vox_check_common(int64_t n_maps, int64_t P, int res) {
  GB_REQUIRE(n_maps > 0 && n_maps <= 65535, GENRE_B200_EINVAL, "N*C = %lld must be in [1, 65535]", (long long)n_maps);
  GB_REQUIRE(P > 0 && P <= VOX_MAX_PIXELS, GENRE_B200_EINVAL, "H*W = %lld must be in [1, 2^20)", (long long)P);
  GB_REQUIRE(res > 0 && (int64_t)res * res * res < (1ll << 31), GENRE_B200_EINVAL, "voxel resolution %d unsupported", res);
  GB_REQUIRE(vox_ntiles(res) <= VOX_MAX_TILES, GENRE_B200_EINVAL, "voxel resolution %d unsupported (too many tiles)", res);
  return 0;
}

}  // namespace gb

// ------------------------------------------------------------------------------------------------
// C ABI: workspace size + stage entry point
// ------------------------------------------------------------------------------------------------
extern "C" size_t genre_b200_voxelize_workspace_bytes(int64_t n_maps, int64_t pixels_per_map, int res) {
  if (n_maps <= 0 || pixels_per_map <= 0 || res <= 0) return 0;
  return gb::vox_workspace_bytes(n_maps, pixels_per_map, res);
}

extern "C" int genre_b200_voxelize_stage_splat(int64_t n_maps, int64_t P, int res, float *tdf, float *cnt,
                                               float hit_alpha, float hit_beta, float background, void *workspace,
                                               size_t workspace_bytes, void *stream) {
  if (int rc = gb::vox_check_common(n_maps, P, res)) return rc;
  GB_REQUIRE(tdf != nullptr, GENRE_B200_EINVAL, "tdf is null");
  gb::VoxWorkspace w;
  GB_REQUIRE(gb::vox_carve(workspace, workspace_bytes, n_maps, P, res, &w), GENRE_B200_EWORKSPACE,
             "workspace too small or misaligned (need %zu bytes)", gb::vox_workspace_bytes(n_maps, P, res));
  return gb::vox_splat(w, n_maps, P, res, tdf, cnt, hit_alpha, hit_beta, background, gb::as_stream(stream), false);
}
