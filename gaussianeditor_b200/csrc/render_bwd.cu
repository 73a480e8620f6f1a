// Backward of the alpha blending for sm_100a: per-pixel dL/dcolor -> per-Gaussian 2-D gradients
// (dL/dcolor, dL/dmean2D, dL/dconic, dL/dopacity), accumulated into the 48-byte-per-Gaussian scratch `acc`.
//
// Semantics: renderCUDA (bwd) of the reference (cuda_rasterizer/backward.cu:399-557): walk each tile's list
// back to front, skip list positions behind the pixel's last contributor, recompute G = exp(power) and alpha
// with the forward's arithmetic (same skip decisions), T <- T/(1-alpha), and accumulate nine partial sums per
// (pixel, splat) hit.
//
// The reference issues nine global float atomics PER HIT (~10^9 REDG at config 3) and walks every tile list
// from its very end.  Here:
//   * the walk starts at tile_last = max n_contrib of the tile (written by the forward): on a saturated scene
//     three quarters of every list lie behind the last contributor of all 256 pixels and are never loaded;
//   * warp variants (1/2/3 branchy, 4..9 branch-light, 10/11 skip by sub-block mask, 12..14 register caps; DEFAULT 14 =
//     one warp per half tile, 96 registers -> 5 CTAs/SM, updates of sub-blocks without a hit skipped warp-uniformly:
//     0.544 ms at config 3; the A/B of all of them is in DESIGN.md section 3): a
//     warp owns a whole tile, half or a quarter of it, each lane owns one pixel of each of its
//     8x4 sub-blocks; the nine partial sums are first accumulated over the lane's own pixels in registers,
//     then summed across the warp with a transposing butterfly (16 shuffles for 9 values instead of 45), and
//     only then added to global memory: 9 atomics per (tile, splat) instead of 9 per (pixel, splat);
//   * the same opacity-aware sub-block culling as the forward (render_fwd.cu) removes splats whose
//     alpha>=1/255 ellipse misses the sub-block before any pixel looks at them.
// Variant 0: the reference's CTA-per-tile structure with a plain warp-shuffle reduction before the atomics.
//
// Gradients are sums of floats in a different order than the reference's atomics (which are themselves
// non-deterministic), so parity is to tolerance (tests: rel L2 <= 1e-4), not bit-exact.
#include "common.cuh"

namespace gsr {

namespace {

struct BwdArgs {
  const uint2* ranges;
  const uint32_t* point_list;
  const SplatRecord* records;
  const uint32_t* tile_last;
  int W, H, gx, gy;
  const float* bg;
  const float* final_T;
  const uint32_t* n_contrib;
  const float* dL_dpix;
  const float* dL_dalpha_img;  // optional [H*W]: gradient of the alpha image 1 - final_T (gsr_backward_alpha)
  float* acc;  // [P, ACC_STRIDE]
  int own_stride, own_phase;  // tile-row ownership (1, 0 = all tiles)
};
// The DEPTH kernels take dL/d(depth image) [H*W] (gsr_backward_depth) as a separate last kernel parameter: BwdArgs keeps
// its layout, so the instantiations without depth compile to exactly the code they had before the depth gradient.

// One (pixel, splat) hit. `ar` tracks the reference's accum_rec (backward.cu:515) dotted with dL_dpixel, updated
// eagerly; `bgT` = T_final * (bg . dL_dpixel).
//
// The nine sums of backward.cu:523-554 are accumulated as moments of w = dL_dG * G over the pixels,
//   g[3..7] = sum w*{dx, dy, dx*dx, dx*dy, dy*dy},  g[8] = sum w,  g[0..2] = sum alpha*T*dL_dpixel,
// and turned into the reference's quantities once per (tile, splat) by finish_sums() -- the per-splat factors
// (conic, opacity, 0.5*W, 0.5*H) are constant over the pixels, so this is the same sum with the common factor
// pulled out (8 instead of 17 operations per hit).
//
// DEPTH (gsr_backward_depth): the depth image D = sum d_i*alpha_i*T_i is a fourth colour channel without a background
// term, with the record's view depth d_i as its colour and dD = dL/dD(pixel) as its upstream gradient. It joins the
// scalar recurrence (s += d_i*dD) and adds one more per-Gaussian sum, g[9] = sum alpha*T*dD = dL/dd_i (acc slot 9).
struct PixState {
  float T, ar, d0, d1, d2, bgT;   // ar = accum_rec . dL_dpixel (scalar; see hit_update)
  float dD;                       // DEPTH only: dL/d(depth image) at this pixel
};
constexpr int nsums(bool depth) { return depth ? 10 : 9; }

// What multiplies dT_final/dalpha_i = -T_final/(1-alpha_i) in dL/dalpha_i: the background term of the colour
// (backward.cu:505-511: bg . dL_dpixel) and, when the caller asked for the alpha image A = 1 - T_final, -dL/dA.
__device__ __forceinline__ float bg_term(const BwdArgs& a, size_t pix_id, float bg0, float bg1, float bg2, const PixState& p) {
  float t = bg0 * p.d0 + bg1 * p.d1 + bg2 * p.d2;
  if (a.dL_dalpha_img != nullptr) t -= a.dL_dalpha_img[pix_id];
  return t;
}

template <bool DEPTH>
__device__ __forceinline__ void hit_update(PixState& p, float* g, float dx, float dy, float G, float alpha, float o,
                                           float c0, float c1, float c2, float depth) {
  const float oma = 1.f - alpha;
  float rcp;  // 1-alpha is in [0.01, 1]: the bare MUFU.RCP (<= 1 ulp here) needs no range fix-up
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rcp) : "f"(oma));
  rcp = alpha > 0.f ? rcp : 1.0f;          // (alpha, G) = (0, 0) encodes "no hit" in the branch-light variants: exact no-op
  p.T = p.T * rcp;                         // T / (1 - alpha)
  const float dchannel_dcolor = alpha * p.T;
  // backward.cu:515-519 keeps the blended colour behind the splat per channel (accum_rec) and forms
  // sum_ch (c_ch - accum_rec_ch) * dL_dpixel_ch. Only that dot product is ever used, and the recurrence
  // accum_rec' = alpha*c + (1-alpha)*accum_rec is linear, so the scalar ar = accum_rec . dL_dpixel obeys
  // ar' = ar + alpha*(c.dL_dpixel - ar): one state variable and 5 operations instead of three and 9.
  float s = fmaf(c2, p.d2, fmaf(c1, p.d1, c0 * p.d0));
  if constexpr (DEPTH) s = fmaf(depth, p.dD, s);  // the depth channel: colour d_i, no background
  float dL_dalpha = s - p.ar;
  g[0] = fmaf(dchannel_dcolor, p.d0, g[0]);
  g[1] = fmaf(dchannel_dcolor, p.d1, g[1]);
  g[2] = fmaf(dchannel_dcolor, p.d2, g[2]);
  if constexpr (DEPTH) g[9] = fmaf(dchannel_dcolor, p.dD, g[9]);
  p.ar = fmaf(alpha, dL_dalpha, p.ar);
  dL_dalpha = fmaf(dL_dalpha, p.T, -p.bgT * rcp);
  const float w = (o * dL_dalpha) * G;  // dL_dG * G
  const float wdx = w * dx, wdy = w * dy;
  g[3] += wdx;
  g[4] += wdy;
  g[5] = fmaf(wdx, dx, g[5]);
  g[6] = fmaf(wdx, dy, g[6]);
  g[7] = fmaf(wdy, dy, g[7]);
  g[8] += w;
}

// Warp totals of the moments -> the reference's nine gradient contributions (acc layout: 0..2 dcolor, 3..4 dmean2D,
// 5..7 dconic a,b,c, 8 dopacity). After warp_sum9 lane 4*j holds the total of moment j (j = 0..7) and every lane holds
// sw = sum w. Output j is a two-term combination  ka*tot + kb*other  with `other` = the partner moment of the
// (w*dx, w*dy) pair (lanes 12..15 <-> 16..19, one shuffle) and lane-constant selectors -- no divergent code:
//   j<3: tot | j=3: -(A*s_x + B*s_y)*0.5W | j=4: -(C*s_y + B*s_x)*0.5H | j=5..7: -0.5*tot | opacity: sw / o
struct LaneRole {
  bool is_x, is_y, writer, opac;  // moment-3 group, moment-4 group, lane that issues the atomic, opacity lane
  bool dep;                       // DEPTH: the lane that adds dL/d(view depth) into slot 9 (neither a writer nor lane 1)
  float kconst;                   // 1 for the colour groups, -0.5 for the conic groups
  int slot;
};
__device__ __forceinline__ LaneRole lane_role(int lane) {
  LaneRole r;
  r.slot = lane >> 2;
  r.is_x = r.slot == 3;
  r.is_y = r.slot == 4;
  r.writer = (lane & 3) == 0;
  r.opac = lane == 1;
  r.dep = lane == 2;
  r.kconst = r.slot < 3 ? 1.0f : -0.5f;
  return r;
}
template <bool DEPTH>
__device__ __forceinline__ void finish_and_add(float* dst, float tot, float sw, float sd, const LaneRole& role, float A,
                                               float B, float C, float o, float ddelx_dx, float ddely_dy) {
  const float other = __shfl_xor_sync(0xffffffffu, tot, 28);  // s_x <-> s_y between lanes 12..15 and 16..19
  const float nBx = -B * ddelx_dx, nBy = -B * ddely_dy;
  const float ka = role.is_x ? -A * ddelx_dx : (role.is_y ? -C * ddely_dy : role.kconst);
  const float kb = role.is_x ? nBx : (role.is_y ? nBy : 0.0f);
  const float v = fmaf(kb, other, ka * tot);
  if (role.writer) atomicAdd(dst + role.slot, v);
  if (role.opac) atomicAdd(dst + 8, __fdividef(sw, o));  // dL/dopacity = sum G*dL_dalpha = (sum w) / o
  if constexpr (DEPTH) {
    if (role.dep) atomicAdd(dst + 9, sd);  // dL/d(view depth) = sum alpha*T*dL/dD
  }
}

// Sum nine per-lane values over the warp. g[0..7] go through a transposing butterfly: after it, lane 4*j (and
// its three neighbours) holds the warp total of g[j]; g[8] takes a plain butterfly. Returns this lane's total of
// value (lane>>2), and the total of g[8] in `g8`. DEPTH: g[9] takes a plain butterfly too, its total in `g9`.
template <bool DEPTH>
__device__ __forceinline__ float warp_sum9(const float* g, int lane, float& g8, float& g9) {
  const unsigned F = 0xffffffffu;
  float a[4], b[2], c;
  {
    const bool up = lane & 16;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const float keep = up ? g[4 + i] : g[i];
      const float send = up ? g[i] : g[4 + i];
      a[i] = keep + __shfl_xor_sync(F, send, 16);
    }
  }
  {
    const bool up = lane & 8;
#pragma unroll
    for (int i = 0; i < 2; i++) {
      const float keep = up ? a[2 + i] : a[i];
      const float send = up ? a[i] : a[2 + i];
      b[i] = keep + __shfl_xor_sync(F, send, 8);
    }
  }
  {
    const bool up = lane & 4;
    const float keep = up ? b[1] : b[0];
    const float send = up ? b[0] : b[1];
    c = keep + __shfl_xor_sync(F, send, 4);
  }
  c += __shfl_xor_sync(F, c, 2);
  c += __shfl_xor_sync(F, c, 1);
  float t = g[8];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(F, t, o);
  g8 = t;
  if constexpr (DEPTH) {
    float d = g[9];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(F, d, o);
    g9 = d;
  }
  return c;
}

// ------------------------------------------------------------------------------------------------------
// Variant 1: NSB sub-blocks per warp (8 = one warp per tile, 4 = two warps per tile)
// ------------------------------------------------------------------------------------------------------
constexpr int BW_WARPS = 4;

template <int NSB, bool DEPTH = false>
__global__ void __launch_bounds__(BW_WARPS * 32) render_bwd_warp_kernel(const BwdArgs a, const int ntiles,
                                                                        const float* dL_ddepth) {
  __shared__ float4 s_stage[BW_WARPS][3][32];
  __shared__ uint32_t s_id[BW_WARPS][32];
  constexpr int PARTS = 8 / NSB;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int gw = blockIdx.x * BW_WARPS + warp;
  const int part = gw % PARTS;
  if (gw / PARTS >= ntiles) return;
  const int tile = owned_tile(gw / PARTS, a.gx, a.own_stride, a.own_phase);  // ntiles counts the OWNED tiles
  float4(*stg)[32] = s_stage[warp];
  uint32_t* sid = s_id[warp];

  const int tx = tile % a.gx, ty = tile / a.gx;
  const int lx = lane & 7, ly = lane >> 3;
  const float X0 = (float)(tx * TILE), Y0 = (float)(ty * TILE);
  const float fx = X0 + (float)lx, fy = Y0 + (float)ly;
  const uint2 range = a.ranges[tile];
  if (a.tile_last[tile] == 0) return;
  const size_t HW = (size_t)a.H * a.W;
  const float bg0 = a.bg[0], bg1 = a.bg[1], bg2 = a.bg[2];
  const float ddelx_dx = 0.5f * a.W, ddely_dy = 0.5f * a.H;
  const LaneRole role = lane_role(lane);

  PixState ps[NSB];
  uint32_t nc[NSB], sblast[NSB];
  uint32_t my_last = 0;
#pragma unroll
  for (int k = 0; k < NSB; k++) {
    const int kg = part * NSB + k;
    const int px = tx * TILE + 8 * (kg & 1) + lx, py = ty * TILE + 4 * (kg >> 1) + ly;
    PixState p;
    p.T = 0.f; p.ar = 0.f; p.d0 = p.d1 = p.d2 = 0.f; p.bgT = 0.f; p.dD = 0.f;
    nc[k] = 0;
    if (px < a.W && py < a.H) {
      const size_t pix_id = (size_t)a.W * py + px;
      const float Tf = a.final_T[pix_id];
      p.T = Tf;
      p.d0 = a.dL_dpix[pix_id];
      p.d1 = a.dL_dpix[HW + pix_id];
      p.d2 = a.dL_dpix[2 * HW + pix_id];
      p.bgT = Tf * bg_term(a, pix_id, bg0, bg1, bg2, p);
      if constexpr (DEPTH) p.dD = dL_ddepth[pix_id];
      nc[k] = a.n_contrib[pix_id];
    }
    ps[k] = p;
    sblast[k] = __reduce_max_sync(0xffffffffu, nc[k]);
    my_last = max(my_last, sblast[k]);
  }

  for (int hi = (int)my_last; hi > 0; hi -= 32) {
    // ---- stage positions hi, hi-1, ... (1-based), cull, compact (descending order is preserved) ----
    const int pos = hi - lane;
    uint32_t mask = 0, id = 0;
    float4 q0, q1, q2;
    if (pos >= 1) {
      id = a.point_list[range.x + pos - 1];
      const float4* r = reinterpret_cast<const float4*>(a.records + id);
      q0 = __ldg(r);
      q1 = __ldg(r + 1);
      q2 = __ldg(r + 2);
      mask = splat_subblock_mask<NSB>(q0, q1, X0, Y0, part);
    }
    const uint32_t keep = __ballot_sync(0xffffffffu, mask != 0);
    const int cnt = __popc(keep);
    if (mask != 0) {
      const int slot = __popc(keep & ((1u << lane) - 1u));
      q1.w = __uint_as_float(mask);
      q2.w = __uint_as_float((uint32_t)pos);
      stg[0][slot] = q0;
      stg[1][slot] = q1;
      stg[2][slot] = q2;
      sid[slot] = id;
    }
    __syncwarp();
    const uint32_t lo = (uint32_t)max(hi - 31, 1);
    uint32_t act = 0;  // sub-blocks that can still have a contributor at these positions
#pragma unroll
    for (int k = 0; k < NSB; k++)
      if (sblast[k] >= lo) act |= 1u << k;

    for (int j = 0; j < cnt; j++) {
      const float4 s1 = stg[1][j];
      const uint32_t m = __float_as_uint(s1.w) & act;
      if (m == 0) continue;
      const float4 s0 = stg[0][j];
      const float4 s2 = stg[2][j];
      const uint32_t spos = __float_as_uint(s2.w);
      float dxv[2], dxA[2], dxB[2], dyv[NSB / 2], t0[NSB / 2];
#pragma unroll
      for (int c = 0; c < 2; c++) {
        dxv[c] = s0.x - (fx + 8.0f * c);
        dxA[c] = __fmul_rn(dxv[c], s0.z);
        dxB[c] = __fmul_rn(dxv[c], s0.w);
      }
#pragma unroll
      for (int r = 0; r < NSB / 2; r++) {
        dyv[r] = s0.y - (fy + 4.0f * (float)(part * (NSB / 2) + r));
        t0[r] = __fmul_rn(__fmul_rn(dyv[r], s1.x), dyv[r]);
      }
      float g[nsums(DEPTH)];
#pragma unroll
      for (int i = 0; i < nsums(DEPTH); i++) g[i] = 0.f;
      bool any = false;
#pragma unroll
      for (int k = 0; k < NSB; k++) {
        if (!((m >> k) & 1u)) continue;  // warp-uniform
        const int c = k & 1, r = k >> 1;  // NSB is even, so the column parity of sub-block part*NSB+k is k&1
        const float dx = dxv[c], dy = dyv[r];
        const float s = __fmaf_rn(dx, dxA[c], t0[r]);
        const float power = __fmaf_rn(s, -0.5f, -__fmul_rn(dxB[c], dy));
        if (power > 0.0f || spos > nc[k]) continue;
        const float G = expf(power);
        const float alpha = fminf(0.99f, __fmul_rn(s1.y, G));
        if (alpha < 1.0f / 255.0f) continue;
        any = true;
        hit_update<DEPTH>(ps[k], g, dx, dy, G, alpha, s1.y, s2.x, s2.y, s2.z, s1.z);
      }
      if (__any_sync(0xffffffffu, any)) {
        float m8, m9;
        const float tot = warp_sum9<DEPTH>(g, lane, m8, m9);
        finish_and_add<DEPTH>(a.acc + (size_t)sid[j] * ACC_STRIDE, tot, m8, m9, role, s0.z, s0.w, s1.x, s1.y, ddelx_dx,
                              ddely_dy);
      }
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------------------------
// Variant 4/5: same mapping as variant 2 (NSB sub-blocks per warp) with a branch-light inner body.
// The profile of variant 2 is latency-bound (33 % of the stall samples are fixed-latency dependency waits, 11 % branch
// resolution, 16 warps/SM): here the NSB evaluations of a splat are issued as independent straight-line chains
// (instruction-level parallelism NSB), hit / no-hit is folded into (alpha, G) = (0, 0) so the gradient arithmetic
// needs no per-pixel branch, and G uses ex2.approx -- the skip decision alpha < 1/255 still equals the forward's
// (which uses libdevice expf) because evaluations within 1e-5 of the threshold are re-done with expf.
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

template <int NSB, int MINB, bool SKIP = false, bool MASKSKIP = false, bool DEPTH = false>
__global__ void __launch_bounds__(BW_WARPS * 32, MINB) render_bwd_flat_kernel(const BwdArgs a, const int ntiles,
                                                                                 const float* dL_ddepth) {
  __shared__ float4 s_stage[BW_WARPS][3][32];
  __shared__ uint32_t s_id[BW_WARPS][32];
  constexpr int PARTS = 8 / NSB;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int gw = blockIdx.x * BW_WARPS + warp;
  const int part = gw % PARTS;
  if (gw / PARTS >= ntiles) return;
  const int tile = owned_tile(gw / PARTS, a.gx, a.own_stride, a.own_phase);  // ntiles counts the OWNED tiles
  float4(*stg)[32] = s_stage[warp];
  uint32_t* sid = s_id[warp];

  const int tx = tile % a.gx, ty = tile / a.gx;
  const int lx = lane & 7, ly = lane >> 3;
  const float X0 = (float)(tx * TILE), Y0 = (float)(ty * TILE);
  const float fx = X0 + (float)lx, fy = Y0 + (float)ly;
  const uint2 range = a.ranges[tile];
  if (a.tile_last[tile] == 0) return;
  const size_t HW = (size_t)a.H * a.W;
  const float bg0 = a.bg[0], bg1 = a.bg[1], bg2 = a.bg[2];
  const float ddelx_dx = 0.5f * a.W, ddely_dy = 0.5f * a.H;
  const LaneRole role = lane_role(lane);

  PixState ps[NSB];
  uint32_t nc[NSB], sblast[NSB];
  uint32_t my_last = 0;
#pragma unroll
  for (int k = 0; k < NSB; k++) {
    const int kg = part * NSB + k;
    const int px = tx * TILE + 8 * (kg & 1) + lx, py = ty * TILE + 4 * (kg >> 1) + ly;
    PixState p;
    p.T = 0.f; p.ar = 0.f; p.d0 = p.d1 = p.d2 = 0.f; p.bgT = 0.f; p.dD = 0.f;
    nc[k] = 0;
    if (px < a.W && py < a.H) {
      const size_t pix_id = (size_t)a.W * py + px;
      const float Tf = a.final_T[pix_id];
      p.T = Tf;
      p.d0 = a.dL_dpix[pix_id];
      p.d1 = a.dL_dpix[HW + pix_id];
      p.d2 = a.dL_dpix[2 * HW + pix_id];
      p.bgT = Tf * bg_term(a, pix_id, bg0, bg1, bg2, p);
      if constexpr (DEPTH) p.dD = dL_ddepth[pix_id];
      nc[k] = a.n_contrib[pix_id];
    }
    ps[k] = p;
    sblast[k] = __reduce_max_sync(0xffffffffu, nc[k]);
    my_last = max(my_last, sblast[k]);
  }

  for (int hi = (int)my_last; hi > 0; hi -= 32) {
    const int pos = hi - lane;
    uint32_t mask = 0, id = 0;
    float4 q0, q1, q2;
    if (pos >= 1) {
      id = a.point_list[range.x + pos - 1];
      const float4* r = reinterpret_cast<const float4*>(a.records + id);
      q0 = __ldg(r);
      q1 = __ldg(r + 1);
      q2 = __ldg(r + 2);
      mask = splat_subblock_mask<NSB>(q0, q1, X0, Y0, part);
    }
    const uint32_t keep = __ballot_sync(0xffffffffu, mask != 0);
    const int cnt = __popc(keep);
    if (mask != 0) {
      const int slot = __popc(keep & ((1u << lane) - 1u));
      q1.w = __uint_as_float(mask);
      q2.w = __uint_as_float((uint32_t)pos);
      stg[0][slot] = q0;
      stg[1][slot] = q1;
      stg[2][slot] = q2;
      sid[slot] = id;
    }
    __syncwarp();
    const uint32_t lo = (uint32_t)max(hi - 31, 1);
    uint32_t act = 0;
#pragma unroll
    for (int k = 0; k < NSB; k++)
      if (sblast[k] >= lo) act |= 1u << k;

    for (int j = 0; j < cnt; j++) {
      const float4 s1 = stg[1][j];
      const uint32_t m = __float_as_uint(s1.w) & act;
      if (m == 0) continue;
      const float4 s0 = stg[0][j];
      const float4 s2 = stg[2][j];
      const uint32_t spos = __float_as_uint(s2.w);
      float dxv[2], dxA[2], dxB[2], dyv[NSB / 2], t0[NSB / 2];
#pragma unroll
      for (int c = 0; c < 2; c++) {
        dxv[c] = s0.x - (fx + 8.0f * c);
        dxA[c] = __fmul_rn(dxv[c], s0.z);
        dxB[c] = __fmul_rn(dxv[c], s0.w);
      }
#pragma unroll
      for (int r = 0; r < NSB / 2; r++) {
        dyv[r] = s0.y - (fy + 4.0f * (float)(part * (NSB / 2) + r));
        t0[r] = __fmul_rn(__fmul_rn(dyv[r], s1.x), dyv[r]);
      }
      // ---- NSB independent evaluations ----
      float G[NSB], al[NSB], pw[NSB];
      bool near = false;
#pragma unroll
      for (int k = 0; k < NSB; k++) {
        if (MASKSKIP && !((m >> k) & 1u)) {  // warp-uniform: the splat's alpha >= 1/255 ellipse misses this sub-block
          pw[k] = 1.0f; G[k] = 0.f; al[k] = 0.f;
          continue;
        }
        const int c = k & 1, r = k >> 1;
        const float s = __fmaf_rn(dxv[c], dxA[c], t0[r]);
        pw[k] = __fmaf_rn(s, -0.5f, -__fmul_rn(dxB[c], dyv[r]));
        G[k] = ex2_approx(pw[k] * 1.4426950408889634f);
        al[k] = fminf(0.99f, s1.y * G[k]);
        near |= fabsf(al[k] - 1.0f / 255.0f) <= (1.0f / 255.0f) * 1e-5f;
      }
      if (near) {  // rare: too close to the 1/255 threshold to call with ex2.approx -> the forward's exact arithmetic
#pragma unroll
        for (int k = 0; k < NSB; k++) {
          if (MASKSKIP && !((m >> k) & 1u)) continue;
          G[k] = expf(pw[k]);
          al[k] = fminf(0.99f, __fmul_rn(s1.y, G[k]));
        }
      }
      bool anyhit = false;
      uint32_t hitk = 0;  // SKIP: warp-uniform mask of sub-blocks with at least one hit
#pragma unroll
      for (int k = 0; k < NSB; k++) {
        const bool ok = ((m >> k) & 1u) && !(pw[k] > 0.0f) && spos <= nc[k] && !(al[k] < 1.0f / 255.0f);
        G[k] = ok ? G[k] : 0.f;
        al[k] = ok ? al[k] : 0.f;
        anyhit |= ok;
        if (SKIP && __any_sync(0xffffffffu, ok)) hitk |= 1u << k;
      }
      if (SKIP ? hitk == 0 : !__any_sync(0xffffffffu, anyhit)) continue;
      float g[nsums(DEPTH)];
#pragma unroll
      for (int i = 0; i < nsums(DEPTH); i++) g[i] = 0.f;
#pragma unroll
      for (int k = 0; k < NSB; k++) {
        // (alpha, G) = (0, 0) makes every update below an exact no-op: 1/(1-0) = 1, +0 contributions
        if (SKIP && !((hitk >> k) & 1u)) continue;
        if (MASKSKIP && !((m >> k) & 1u)) continue;
        hit_update<DEPTH>(ps[k], g, dxv[k & 1], dyv[k >> 1], G[k], al[k], s1.y, s2.x, s2.y, s2.z, s1.z);
      }
      float m8, m9;
      const float tot = warp_sum9<DEPTH>(g, lane, m8, m9);
      finish_and_add<DEPTH>(a.acc + (size_t)sid[j] * ACC_STRIDE, tot, m8, m9, role, s0.z, s0.w, s1.x, s1.y, ddelx_dx,
                            ddely_dy);
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------------------------
// Variant 0: CTA per tile, one pixel per thread, butterfly reduction of the nine sums per splat
// ------------------------------------------------------------------------------------------------------
template <bool DEPTH = false>
__global__ void __launch_bounds__(TILE_PIX) render_bwd_cta_kernel(const BwdArgs a, const float* dL_ddepth) {
  __shared__ float4 s_q0[TILE_PIX], s_q1[TILE_PIX], s_q2[TILE_PIX];
  __shared__ uint32_t s_ids[TILE_PIX];
  const int tile = blockIdx.y * a.gx + blockIdx.x;
  const int tid = threadIdx.y * TILE + threadIdx.x;
  const int lane = tid & 31;
  const uint2 pix = make_uint2(blockIdx.x * TILE + threadIdx.x, blockIdx.y * TILE + threadIdx.y);
  const bool inside = pix.x < (unsigned)a.W && pix.y < (unsigned)a.H;
  const size_t pix_id = (size_t)a.W * pix.y + pix.x;
  const float2 pixf = make_float2((float)pix.x, (float)pix.y);
  const uint2 range = a.ranges[tile];
  const int tl = (int)a.tile_last[tile];  // block-uniform
  const size_t HW = (size_t)a.H * a.W;

  PixState p;
  p.T = 0.f; p.ar = 0.f; p.d0 = p.d1 = p.d2 = 0.f; p.bgT = 0.f; p.dD = 0.f;
  uint32_t nc = 0;
  if (inside) {
    const float Tf = a.final_T[pix_id];
    p.T = Tf;
    p.d0 = a.dL_dpix[pix_id]; p.d1 = a.dL_dpix[HW + pix_id]; p.d2 = a.dL_dpix[2 * HW + pix_id];
    p.bgT = Tf * bg_term(a, pix_id, a.bg[0], a.bg[1], a.bg[2], p);
    if constexpr (DEPTH) p.dD = dL_ddepth[pix_id];
    nc = a.n_contrib[pix_id];
  }
  const float ddelx_dx = 0.5f * a.W, ddely_dy = 0.5f * a.H;
  const LaneRole role = lane_role(lane);

  for (int hi = tl; hi > 0; hi -= TILE_PIX) {
    __syncthreads();
    const int pos = hi - tid;
    if (pos >= 1) {
      const uint32_t id = a.point_list[range.x + pos - 1];
      const float4* r = reinterpret_cast<const float4*>(a.records + id);
      s_q0[tid] = __ldg(r); s_q1[tid] = __ldg(r + 1); s_q2[tid] = __ldg(r + 2);
      s_ids[tid] = id;
    }
    __syncthreads();
    const int n = min(TILE_PIX, hi);
    for (int j = 0; j < n; j++) {
      const uint32_t spos = (uint32_t)(hi - j);
      const float4 q0 = s_q0[j], q1 = s_q1[j];
      const float dx = q0.x - pixf.x, dy = q0.y - pixf.y;
      const float power = splat_power(dx, dy, q0.z, q0.w, q1.x);
      float g[nsums(DEPTH)];
#pragma unroll
      for (int i = 0; i < nsums(DEPTH); i++) g[i] = 0.f;
      bool hit = false;
      if (!(power > 0.0f) && spos <= nc) {
        const float G = expf(power);
        const float alpha = fminf(0.99f, __fmul_rn(q1.y, G));
        if (!(alpha < 1.0f / 255.0f)) {
          hit = true;
          const float4 q2 = s_q2[j];
          hit_update<DEPTH>(p, g, dx, dy, G, alpha, q1.y, q2.x, q2.y, q2.z, q1.z);
        }
      }
      if (__any_sync(0xffffffffu, hit)) {
        float m8, m9;
        const float tot = warp_sum9<DEPTH>(g, lane, m8, m9);
        finish_and_add<DEPTH>(a.acc + (size_t)s_ids[j] * ACC_STRIDE, tot, m8, m9, role, q0.z, q0.w, q1.x, q1.y, ddelx_dx,
                              ddely_dy);
      }
    }
  }
}

// One launch of render_bwd_variant v (see Options::render_bwd_variant); DEPTH picks the instantiation that also
// back-propagates the depth image. Every variant exists in both forms, so the variant option never drops dL/dD.
template <bool DEPTH>
void launch_variant(int v, const BwdArgs& a, int ntiles, const float* dL_ddepth, cudaStream_t st) {
  if (v == 0) {
    render_bwd_cta_kernel<DEPTH><<<dim3(a.gx, a.gy), dim3(TILE, TILE), 0, st>>>(a, dL_ddepth);
  } else if (v == 2) {
    const int warps = ntiles * 2;
    render_bwd_warp_kernel<4, DEPTH><<<(warps + BW_WARPS - 1) / BW_WARPS, BW_WARPS * 32, 0, st>>>(a, ntiles, dL_ddepth);
  } else if (v == 3) {
    const int warps = ntiles * 4;
    render_bwd_warp_kernel<2, DEPTH><<<(warps + BW_WARPS - 1) / BW_WARPS, BW_WARPS * 32, 0, st>>>(a, ntiles, dL_ddepth);
  } else if (v == 4) {
    render_bwd_flat_kernel<4, 1, false, false, DEPTH><<<(ntiles * 2 + BW_WARPS - 1) / BW_WARPS, BW_WARPS * 32, 0, st>>>(a, ntiles, dL_ddepth);
  } else if (v == 5) {
    render_bwd_flat_kernel<4, 6, false, false, DEPTH><<<(ntiles * 2 + BW_WARPS - 1) / BW_WARPS, BW_WARPS * 32, 0, st>>>(a, ntiles, dL_ddepth);
  } else if (v == 6) {
    render_bwd_flat_kernel<2, 1, false, false, DEPTH><<<(ntiles * 4 + BW_WARPS - 1) / BW_WARPS, BW_WARPS * 32, 0, st>>>(a, ntiles, dL_ddepth);
  } else if (v == 7) {
    render_bwd_flat_kernel<8, 1, false, false, DEPTH><<<(ntiles + BW_WARPS - 1) / BW_WARPS, BW_WARPS * 32, 0, st>>>(a, ntiles, dL_ddepth);
  } else if (v == 8) {
    render_bwd_flat_kernel<4, 1, true, false, DEPTH><<<(ntiles * 2 + BW_WARPS - 1) / BW_WARPS, BW_WARPS * 32, 0, st>>>(a, ntiles, dL_ddepth);
  } else if (v == 9) {
    render_bwd_flat_kernel<8, 1, true, false, DEPTH><<<(ntiles + BW_WARPS - 1) / BW_WARPS, BW_WARPS * 32, 0, st>>>(a, ntiles, dL_ddepth);
  } else if (v == 12) {  // register caps: 5 / 6 CTAs per SM, with and without the hit-skip
    render_bwd_flat_kernel<4, 5, false, false, DEPTH><<<(ntiles * 2 + BW_WARPS - 1) / BW_WARPS, BW_WARPS * 32, 0, st>>>(a, ntiles, dL_ddepth);
  } else if (v == 13) {
    render_bwd_flat_kernel<4, 6, true, false, DEPTH><<<(ntiles * 2 + BW_WARPS - 1) / BW_WARPS, BW_WARPS * 32, 0, st>>>(a, ntiles, dL_ddepth);
  } else if (v == 14) {
    // the DEPTH instantiation fits the same cap without spilling (96 registers, 5 CTAs/SM)
    render_bwd_flat_kernel<4, 5, true, false, DEPTH><<<(ntiles * 2 + BW_WARPS - 1) / BW_WARPS, BW_WARPS * 32, 0, st>>>(a, ntiles, dL_ddepth);
  } else if (v == 10) {  // variant 4 + sub-blocks outside the splat's mask skipped with warp-uniform branches
    render_bwd_flat_kernel<4, 1, false, true, DEPTH><<<(ntiles * 2 + BW_WARPS - 1) / BW_WARPS, BW_WARPS * 32, 0, st>>>(a, ntiles, dL_ddepth);
  } else if (v == 11) {  // the same for the quarter-tile mapping
    render_bwd_flat_kernel<2, 1, false, true, DEPTH><<<(ntiles * 4 + BW_WARPS - 1) / BW_WARPS, BW_WARPS * 32, 0, st>>>(a, ntiles, dL_ddepth);
  } else {
    render_bwd_warp_kernel<8, DEPTH><<<(ntiles + BW_WARPS - 1) / BW_WARPS, BW_WARPS * 32, 0, st>>>(a, ntiles, dL_ddepth);
  }
}

}  // namespace

int launch_render_bwd(const gsr_settings& s, const GeometryWS& g, const BinningWS& b, const ImageWS& im,
                      const float* dL_dpix, float* acc, cudaStream_t st, const TileOwner& own,
                      const float* dL_dalpha_img, const float* dL_ddepth) {
  BwdArgs a;
  a.dL_dalpha_img = dL_dalpha_img;
  a.own_stride = own.stride; a.own_phase = own.phase;
  a.ranges = im.ranges; a.point_list = b.point_list; a.records = g.records; a.tile_last = im.tile_last;
  a.W = s.image_width; a.H = s.image_height;
  a.gx = (a.W + TILE - 1) / TILE; a.gy = (a.H + TILE - 1) / TILE;
  a.bg = s.bg; a.final_T = im.final_T; a.n_contrib = im.n_contrib; a.dL_dpix = dL_dpix; a.acc = acc;
  const int ntiles = a.gx * own.owned_rows(a.gy);  // tiles this rank walks (all of them when own = {1,0})
  if (ntiles == 0) return GSR_OK;
  int v = g_opt.render_bwd_variant;
  if (v == 0 && own.stride != 1) v = 4;  // the CTA-per-tile kernel maps blockIdx to tiles directly: single-GPU only
  if (dL_ddepth != nullptr)
    launch_variant<true>(v, a, ntiles, dL_ddepth, st);
  else
    launch_variant<false>(v, a, ntiles, nullptr, st);
  g_launches++;
  return check_launch("render_bwd", s.debug != 0, st);
}

}  // namespace gsr
