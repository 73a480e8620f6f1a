// Shared declarations of the sm_100a rasterizer kernels (internal; the public surface is include/gsr_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <stdint.h>
#include <stddef.h>

#include "../../include/gsr_b200.h"

namespace gsr {

constexpr int TILE = 16;  // tile edge in pixels; fixed by the reference's binning (config.h:16-17) and
                          // therefore by the bit-exact tile-range contract
constexpr int TILE_PIX = TILE * TILE;

// ---- HBM layout ------------------------------------------------------------------------------------
// Per-Gaussian "splat record": everything the two render kernels need about a projected Gaussian, packed
// into 48 contiguous, 16-byte-aligned bytes so that one tile-list gather is three 128-bit loads
// (the reference gathers from five separate arrays: means2D, conic_opacity, rgb, depths, point ids).
//   q0 = { x, y, conic.a, conic.b }      q1 = { conic.c, opacity, view-depth, <unused> }
//   q2 = { r, g, b, radius (int bits; 0 = culled, the only field a culled record defines) }
struct __align__(16) SplatRecord {
  float4 q0, q1, q2;
};
static_assert(sizeof(SplatRecord) == 48, "record layout");

inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

struct GeometryWS {
  SplatRecord* records;     // [P]
  uint32_t* tiles_touched;  // [P]
  uint8_t* clamped;         // [P]
  uint32_t* depth_keys;     // [P] fp32 view-depth bits, 0xFFFFFFFF for culled
  uint32_t* ident;          // [P] 0..P-1
  uint32_t* depth_keys_sorted;
  uint32_t* depth_order;    // [P] Gaussian indices in (depth, index) order
  uint32_t* offsets;        // [P] inclusive scan of tiles_touched in depth order
  uint32_t* R_dev;          // [4]  word 0: number of instances (tile_binning.cu: tile_count_kernel)
  int32_t* tile_diff;       // [MAX_TILE_DIFF] 2-D difference array of the tile rectangles, (gy+1) x (gx+1), directly
                            //      behind R_dev so that one memset clears both
  void* cub_temp;
  size_t cub_temp_bytes;
  size_t total;
};
// (gx+1)*(gy+1) <= 2*65536 + 1 for every grid with gx*gy < 65536 tiles (the limit of the 16-bit tile keys)
constexpr int MAX_TILE_DIFF = 4 * (2 * 65536 + 64);  // 2 MB: room for 64 replicas of a 1600x1200 grid
// The corner updates are global atomics and a scene concentrates them on the few hundred entries around the screen
// centre (same-address atomics serialise in L2: measured +65 us on the 1M-Gaussian preprocess). The reservation is used
// for up to 64 REPLICAS of the array (Gaussian i updates replica i & (copies-1)); the readers add the replicas up.
inline int tile_diff_copies(int gx, int gy) {
  const long long nent = (long long)(gx + 1) * (gy + 1);
  int c = 1;  // + 1: behind the replicas lies their sum, written by tile_count_kernel and read by tile_prefix_kernel
  // up to 64 replicas, but no more than ~0.5 MB in total: beyond that the memset and the replica sum cost more than the
  // contention they remove (measured at 1600x1200: 16 replicas 0.075 ms, 64 replicas 0.081 ms for the preprocess stage)
  while (c < 64 && (2LL * c + 1) * nent <= MAX_TILE_DIFF / 4) c *= 2;
  return c;
}
struct BinningWS {
  uint32_t* keys_unsorted;  // [R] tile id
  uint32_t* keys_sorted;    // [R]
  uint32_t* vals_unsorted;  // [R] Gaussian index
  uint32_t* point_list;     // [R] sorted
  void* cub_temp;
  size_t cub_temp_bytes;
  // tile_binning.cu (own radix passes with decoupled look-back): per pass and sort tile one status word per digit,
  // plus [0..1] ticket counters and [2 .. 2+512) the exclusive digit bases of both passes
  uint32_t* sort_state;
  size_t sort_state_bytes;
  size_t total;
};
struct ImageWS {
  float* final_T;       // [Npix]
  uint32_t* n_contrib;  // [Npix]
  uint2* ranges;        // [Ntile]
  uint32_t* tile_last;  // [Ntile] max n_contrib over the tile's pixels: where the backward walk starts
  size_t total;
};

// Tile ownership of the Gaussian-sharded multi-GPU path (gsr_b200.h: gsr_tile_owner): this rank bins and renders the
// tile rows ty with ty % stride == phase. {1, 0} = every tile (single-GPU path).
struct TileOwner {
  int stride = 1, phase = 0;
  int owned_rows(int gy) const { return phase < gy ? (gy - phase + stride - 1) / stride : 0; }
};

// Carve a workspace out of `base` (may be null for a pure size query).
bool carve_geometry(void* base, int P, GeometryWS& ws);
bool carve_binning(void* base, int P, int64_t R, int W, int H, BinningWS& ws);
void carve_image(void* base, int W, int H, ImageWS& ws);

// Backward scratch: per-Gaussian accumulators of the nine 2-D gradients (+3 pad -> 48 B, 16-B aligned):
//   [0..2] dL/dcolor  [3..4] dL/dmean2D  [5..7] dL/dconic (a,b,c)  [8] dL/dopacity
//   [9] dL/d(view depth), written only by the depth-gradient backward (gsr_backward_depth), zero otherwise
constexpr int ACC_STRIDE = 12;

// ---- options -----------------------------------------------------------------------------------------
struct Options {
  int render_fwd_variant = 3;  // 0 CTA/tile, 1/2/3 = 1/2/4 warps per tile
  int render_bwd_variant = 14;  // 0 CTA/tile, 1/2/3 branchy, 4..9 branch-light, 10/11 mask-skip, 12..14 register caps (14: 96 regs + hit-skip)
  int preprocess_variant = 1;
  int profile = 0;
  int tile_key_bits = 16;
  int binning_variant = 1;     // 0 = emit kernel + CUB tile sort + tile_ranges, 1 = tile_binning.cu
  int depth_sort_variant = 0;  // 0 = CUB radix sort + CUB scan (default: faster at 1M keys), 1 = depth_sort.cu
};
enum Stage { ST_PRE_FWD = 0, ST_DEPTH_SCAN, ST_EMIT, ST_TILE_SORT, ST_RANGES, ST_RENDER_FWD, ST_RENDER_BWD, ST_PRE_BWD, ST_APPLY_W };
// RAII stage timer: records two events on `st` when profiling is on, otherwise free.
struct StageScope {
  int stage; cudaStream_t st; void* rec;
  StageScope(int stage, cudaStream_t st);
  ~StageScope();
};
extern Options g_opt;
extern unsigned long long* g_stats_dev;  // device counters when option "stats" is on (instrumentation only)
extern std::atomic<long long> g_launches;

// ---- error plumbing ------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what);
int check_launch(const char* what, bool debug, cudaStream_t st);
int validate_cloud(const gsr_settings* s, const gsr_cloud* c);  // argument checks of the reference's Python/C++ glue

// ---- stage entry points (host side; each file owns its kernels) ------------------------------------------
// peer_records/npeers: fused all-gather of the sharded path (every rank's view of this shard's record slice), else 0
// raw selects the RAW variant (fused activations): c.opacities / c.scales / c.rotations are then the raw parameters,
// c.shs is features_dc [P,1,3] and features_rest [P,M-1,3] holds the other coefficients (may be null when M == 1).
int launch_preprocess_fwd(const gsr_settings& s, const gsr_cloud& c, const GeometryWS& g, int32_t* radii,
                          cudaStream_t st, SplatRecord* const* peer_records = nullptr, int npeers = 0, bool raw = false,
                          const float* features_rest = nullptr, bool count_tiles = false);
// depth_sort.cu: depth order + offsets scan without CUB; scratch lives in GeometryWS::cub_temp
size_t depth_sort_scratch_bytes(int P);
int run_depth_sort_own(int P, const GeometryWS& g, cudaStream_t st, bool debug);
int run_depth_order_and_scan(const gsr_cloud& c, const GeometryWS& g, int32_t* num_rendered_host, cudaStream_t st,
                             bool debug);
// Sharded path: recompute tiles_touched (owned tile rows only) and the sort identity for all P gathered Gaussians.
int launch_retouch(const gsr_settings& s, int P, const GeometryWS& g, int32_t* radii, const TileOwner& own,
                   cudaStream_t st);
int run_binning(const gsr_settings& s, const gsr_cloud& c, int R, bool speculative, const GeometryWS& g,
                const BinningWS& b, const ImageWS& im, const int32_t* radii, cudaStream_t st,
                const TileOwner& own = TileOwner());
// tile_binning.cu: ranges from the tile-count difference array, emission fused into the first of two own radix passes
constexpr int SORT_TILE = 4096;  // instances per CTA of a radix pass
bool tile_binning_supported(int gx, int gy);
int run_tile_binning(const gsr_settings& s, int P, int R, bool speculative, const GeometryWS& g, const BinningWS& b,
                     const ImageWS& im, const int32_t* radii, cudaStream_t st, const TileOwner& own);
// clears R_dev + the difference array of a gx x gy grid (before the kernel that accumulates them)
int clear_tile_counts(const GeometryWS& g, int gx, int gy, cudaStream_t st);
// g.R_dev[0] = number of instances in the owned tile rows = a weighted sum over the difference array (no prefix needed)
int launch_tile_count(const GeometryWS& g, int gx, int gy, const TileOwner& own, cudaStream_t st);
int launch_render_fwd(const gsr_settings& s, const GeometryWS& g, const BinningWS& b, const ImageWS& im,
                      float* out_color, float* out_depth, cudaStream_t st, const TileOwner& own = TileOwner());
int launch_render_bwd(const gsr_settings& s, const GeometryWS& g, const BinningWS& b, const ImageWS& im,
                      const float* dL_dpix, float* acc, cudaStream_t st, const TileOwner& own = TileOwner(),
                      const float* dL_dalpha_img = nullptr, const float* dL_ddepth = nullptr);
// raw != nullptr: RAW variant -- gradients w.r.t. the raw parameters (gr.dL_dsh = d features_dc, raw->dL_dfeatures_rest)
struct RawBackward {
  const float* features_rest;
  float* dL_dfeatures_rest;
};
// cam != nullptr: also dL/dviewmatrix [16], dL/dprojmatrix [16], dL/dcampos [3] (opt-in; scratch = camera_scratch_bytes(P))
// depth: acc slot 9 holds dL/d(view depth) (gsr_backward_depth) and enters dL/dt.z
struct CameraBackward {
  float* dL_dviewmatrix;
  float* dL_dprojmatrix;
  float* dL_dcampos;
  float* scratch;
};
size_t camera_scratch_bytes(int P);
int launch_preprocess_bwd(const gsr_settings& s, const gsr_cloud& c, const GeometryWS& g, const int32_t* radii,
                          const float* acc, const gsr_grads& gr, cudaStream_t st, const RawBackward* raw = nullptr,
                          const CameraBackward* cam = nullptr, bool depth = false);
// out_alpha[i] = 1 - final_T[i]  (the reference keeps final_T as ImageState::accum_alpha, rasterizer_impl.h:50)
int launch_alpha_image(const float* final_T, size_t n, float* out_alpha, cudaStream_t st);
int launch_mark_visible(int P, const float* means3D, const float* viewmatrix, uint8_t* present, cudaStream_t st);
int launch_apply_weights(const gsr_settings& s, const GeometryWS& g, const BinningWS& b, const ImageWS& im,
                         const float* image_weights, int CH, float* weights, int32_t* cnt, cudaStream_t st);

#ifdef __CUDACC__
// ---- device helpers ---------------------------------------------------------------------------------

// Reference numerics of one (pixel, splat) evaluation, fixed with explicit round-to-nearest intrinsics so the
// compiler can neither re-associate nor contract differently. The sequence is what nvcc emits for
// forward.cu:335-338 / backward.cu:491-494 at sm_100a (SASS of the unmodified reference, see DESIGN.md):
//   power = fma( fma(dx, A*dx, (C*dy)*dy), -0.5, -((B*dx)*dy) )
__device__ __forceinline__ float splat_power(float dx, float dy, float A, float B, float C) {
  float t0 = __fmul_rn(__fmul_rn(dy, C), dy);
  float t1 = __fmul_rn(dx, A);
  float t2 = __fmul_rn(__fmul_rn(dx, B), dy);
  float s = __fmaf_rn(dx, t1, t0);
  return __fmaf_rn(s, -0.5f, -t2);
}

// Which 8x4 sub-blocks of tile (X0,Y0) can a splat reach with alpha >= 1/255?  alpha = o*exp(power) >= 1/255 iff
// q(dx,dy) = A dx^2 + 2B dx dy + C dy^2 <= 2 ln(255 o), so sub-block k is reachable iff the minimum of the convex
// quadratic q over its pixel rectangle is below that threshold. The exact box minimum of a convex quadratic whose
// unconstrained minimiser is the origin is min(q on the line v = v_c, q on the line u = u_c) with (u_c, v_c) the box
// point closest to the origin and the free coordinate clamped to the box (two 1-D parabola minima). The rectangle is
// grown by 0.02 px and the threshold by 0.1 % + 2e-3, far beyond fp32 rounding of `power`, so the test only ever
// rejects splats every pixel of the sub-block would skip at `alpha < 1/255` (results unchanged, n_contrib included).
// Returns a mask over this warp's NSB sub-blocks (global sub-block index part*NSB + k, column k&1, row pair k>>1).
template <int NSB>
__device__ __forceinline__ uint32_t splat_subblock_mask(const float4 q0, const float4 q1, float X0, float Y0, int part) {
  const float A = q0.z, B = q0.w, C = q1.x, o = q1.y;
  if (o < 1.0f / 255.0f) return 0u;  // alpha = o*exp(power<=0) can never reach 1/255
  const float det = A * C - B * B;
  if (!(det > 0.0f) || !(A > 0.0f) || !(C > 0.0f) || !(A < 1e30f) || !(C < 1e30f)) return (1u << NSB) - 1u;
  const float thr = 2.0f * (__logf(o * 255.0f) * 1.001f + 1e-3f);
  const float nBA = -B / A, nBC = -B / C;
  const float cx = q0.x - X0, cy = q0.y - Y0;  // splat centre relative to the tile origin
  uint32_t mask = 0;
#pragma unroll
  for (int k = 0; k < NSB; k++) {
    const int kg = part * NSB + k;
    const float ua = (float)(8 * (kg & 1)) - 0.02f - cx, ub = ua + 7.04f;   // u = pixel_x - centre_x over the block
    const float va = (float)(4 * (kg >> 1)) - 0.02f - cy, vb = va + 3.04f;
    const float uc = fminf(fmaxf(0.f, ua), ub), vc = fminf(fmaxf(0.f, va), vb);
    const float us = fminf(fmaxf(nBA * vc, ua), ub);                          // argmin_u q(u, vc) over [ua, ub]
    const float vs = fminf(fmaxf(nBC * uc, va), vb);                          // argmin_v q(uc, v) over [va, vb]
    const float q1v = A * us * us + (2.0f * B * us + C * vc) * vc;
    const float q2v = C * vs * vs + (2.0f * B * vs + A * uc) * uc;
    if (fminf(q1v, q2v) <= thr) mask |= 1u << k;
  }
  return mask;
}

// n-th tile (row-major over the owned rows) of a rank that owns the tile rows ty = phase + k*stride
__device__ __forceinline__ int owned_tile(int n, int gx, int stride, int phase) {
  const int r = n / gx;
  return (phase + r * stride) * gx + (n - r * gx);
}

// the four corners of a tile rectangle [rmin, rmax) in replica (idx & (copies-1)) of the (gy+1) x (gx+1) difference array
__device__ __forceinline__ void add_tile_rect(int32_t* diff, int gx, int gy, int copies, uint32_t idx, uint32_t x0, uint32_t y0,
                                              uint32_t x1, uint32_t y1) {
  const int stride = gx + 1;
  int32_t* d = diff + (size_t)(idx & (uint32_t)(copies - 1)) * (size_t)(stride * (gy + 1));
  atomicAdd(d + y0 * stride + x0, 1);
  atomicAdd(d + y0 * stride + x1, -1);
  atomicAdd(d + y1 * stride + x0, -1);
  atomicAdd(d + y1 * stride + x1, 1);
}

// 128-bit streaming loads/stores
__device__ __forceinline__ float4 ldg4(const float4* p) { return __ldg(p); }

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// mbarrier + bulk async copy (TMA unit; SASS: UBLKCP / SYNCS)
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t phase) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tWAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}" ::"r"(smem_u32(bar)),
      "r"(phase)
      : "memory");
}
// global -> shared bulk copy, completion counted in bytes on `bar`; size and both addresses multiples of 16
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// shared -> global bulk copy (bulk async-group completion)
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
#endif  // __CUDACC__

}  // namespace gsr
