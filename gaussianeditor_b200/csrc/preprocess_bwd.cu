// Backward of the per-Gaussian preprocess for sm_100a: 2-D gradients -> gradients of means3D, scales,
// rotations (or cov3D), SH coefficients (or colours) and opacity.
//
// Semantics: the reference's two kernels computeCov2DCUDA (cuda_rasterizer/backward.cu:144-274) and
// preprocessCUDA (bwd, :346-396 with computeColorFromSH :20-139 and computeCov3D :278-341), in the order of
// rasterizer_impl.cu:333-340 (the covariance kernel ASSIGNS dL/dmean, the second kernel adds the projection and
// SH view-direction terms).  Fused here into ONE pass over the cloud:
//   * every input byte of a Gaussian is read once (the reference reads mean/radii/cov3D twice and round-trips
//     dL/dcov3D and dL/dmean through HBM between its two kernels); cov3D is recomputed from scale/rotation
//     instead of being stored by the forward (saves 24 B/Gaussian written + read);
//   * the kernel writes EVERY gradient element itself -- zeros for culled Gaussians and for SH coefficients
//     above the active degree -- so the caller allocates outputs uninitialised and the reference's nine
//     zero-fill kernels (rasterize_points.cu:120-128; 300 MB of memset at config 3) disappear;
//   * SH rows (192 B in, 192 B out per Gaussian at degree 3) move through the TMA unit: cp.async.bulk
//     global->shared for visible Gaussians only, cp.async.bulk shared->global for the gradient rows, staged in
//     padded 208-byte shared-memory rows owned by one thread each (conflict-free 128-bit accesses, no
//     block-level synchronisation besides the load mbarrier).
#include "common.cuh"

namespace gsr {

namespace {

constexpr int PB_THREADS = 128;
constexpr int ROW_WORDS = 52;

struct M3 {
  float m[3][3];  // m[column][row]
};
__device__ __forceinline__ M3 mat_mul(const M3& A, const M3& B) {
  M3 R;
#pragma unroll
  for (int c = 0; c < 3; c++)
#pragma unroll
    for (int r = 0; r < 3; r++) R.m[c][r] = A.m[0][r] * B.m[c][0] + A.m[1][r] * B.m[c][1] + A.m[2][r] * B.m[c][2];
  return R;
}
__device__ __forceinline__ M3 mat_t(const M3& A) {
  M3 R;
#pragma unroll
  for (int c = 0; c < 3; c++)
#pragma unroll
    for (int r = 0; r < 3; r++) R.m[c][r] = A.m[r][c];
  return R;
}

struct PbArgs {
  int P, D, M, W, H;
  float tan_fovx, tan_fovy, h_x, h_y, scale_modifier;
  const float* means3D;
  const float* shs;
  const float* scales;
  const float* rotations;
  const float* cov3D_precomp;
  const float* view;
  const float* proj;
  const float* campos;
  const int32_t* radii;
  const uint8_t* clamped;
  const float* acc;
  float* dL_dmeans3D;
  float* dL_dmeans2D;
  float* dL_dcolors;
  float* dL_dopacity;
  float* dL_dcov3D;
  float* dL_dsh;
  float* dL_dscales;
  float* dL_drotations;
  // RAW variant (fused activations): shs = features_dc [P,1,3], dL_dsh = d features_dc, opacities = logits,
  // scales = log-scales, rotations = unnormalised; gradients are taken w.r.t. those raw parameters
  const float* opacities;
  const float* features_rest;
  float* dL_dfeatures_rest;
  float* cam_partial;  // CAM variant: [nblocks, CAM_STRIDE] block partial sums of the camera gradients
  int depth;           // acc slot 9 holds dL/d(view depth) (gsr_backward_depth): add it to dL/dt.z
};

__device__ __forceinline__ M3 quat_to_R(float r, float x, float y, float z) {
  M3 R;
  R.m[0][0] = 1.f - 2.f * (y * y + z * z); R.m[0][1] = 2.f * (x * y - r * z); R.m[0][2] = 2.f * (x * z + r * y);
  R.m[1][0] = 2.f * (x * y + r * z); R.m[1][1] = 1.f - 2.f * (x * x + z * z); R.m[1][2] = 2.f * (y * z - r * x);
  R.m[2][0] = 2.f * (x * z - r * y); R.m[2][1] = 2.f * (y * z + r * x); R.m[2][2] = 1.f - 2.f * (x * x + y * y);
  return R;
}

// Camera gradients (opt-in, gsr_backward_camera; the reference has none: its autograd returns None for the settings,
// diff_gaussian_rasterization/__init__.py:213-223). viewmatrix, projmatrix and campos are treated as INDEPENDENT inputs,
// exactly as the forward reads them; a caller that builds projmatrix / campos from the view matrix chains the three.
// Compact per-thread accumulator layout, CAM_N floats:
//   [4k + j]      dL/dview[k + 4j]   k = 0..2 (row of t = view * mean), j = 0..3 (x, y, z, 1)
//   [12 + 4r + j] dL/dproj[i + 4j]   i = (0, 1, 3)[r] (p_hom.x, .y, .w)
//   [24 + c]      dL/dcampos[c]
constexpr int CAM_N = 27, CAM_STRIDE = 32;

template <bool BULK, bool RAW = false, bool CAM = false>
__global__ void __launch_bounds__(PB_THREADS) preprocess_bwd_kernel(const PbArgs a) {
  static_assert(!(BULK && RAW), "the RAW variant stages its SH block itself");
  float cg[CAM ? CAM_N : 1];
  if (CAM) {
#pragma unroll
    for (int i = 0; i < CAM_N; i++) cg[i] = 0.f;
  }
  __shared__ __align__(16) float rows[BULK ? PB_THREADS * ROW_WORDS : 4];
  // RAW: the CTA's features_rest rows in (one bulk load), overwritten in place by their gradients, out (one bulk store)
  __shared__ __align__(128) float s_rest[RAW ? PB_THREADS * 45 : 1];
  __shared__ uint64_t bar;
  const int idx = blockIdx.x * PB_THREADS + threadIdx.x;
  const bool live = idx < a.P;
  const bool vis = live && a.radii[idx] > 0;
  const bool has_sh = a.shs != nullptr;
  float* row = BULK ? &rows[threadIdx.x * ROW_WORDS] : nullptr;
  const int nb = (a.D + 1) * (a.D + 1);  // active coefficients
  const int K3 = RAW ? (a.M - 1) * 3 : 0;
  bool rest_block = false, rest_loaded = false;
  if (RAW) {
    const int first = blockIdx.x * PB_THREADS;
    const uint32_t bytes = (uint32_t)(min(PB_THREADS, a.P - first) * K3 * 4);
    rest_block = bytes != 0 && (bytes & 15u) == 0;          // else: partial last block, plain loads / stores
    if (threadIdx.x == 0) {
      mbar_init(&bar, 1);
      fence_mbar_init();
    }
    rest_loaded = __syncthreads_or(vis) && rest_block && a.D > 0;
    if (rest_loaded && threadIdx.x == 0) {
      mbar_arrive_expect_tx(&bar, bytes);
      bulk_g2s(s_rest, a.features_rest + (size_t)first * K3, bytes, &bar);
    }
  }

  if (BULK) {
    if (threadIdx.x == 0) {
      mbar_init(&bar, PB_THREADS);
      fence_mbar_init();
    }
    __syncthreads();
    const uint32_t nbytes = (uint32_t)((nb * 12 + 15) & ~15);
    if (vis) {
      mbar_arrive_expect_tx(&bar, nbytes);
      bulk_g2s(row, a.shs + (size_t)idx * a.M * 3, nbytes, &bar);
    } else {
      mbar_arrive(&bar);
    }
  }

  float dmean[3] = {0.f, 0.f, 0.f}, dcov[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float dscale[3] = {0.f, 0.f, 0.f}, drot[4] = {0.f, 0.f, 0.f, 0.f};
  float4 acc0 = make_float4(0.f, 0.f, 0.f, 0.f), acc1 = acc0, acc2 = acc0;
  float3 mean = make_float3(0.f, 0.f, 0.f);
  float3 act_scale = make_float3(0.f, 0.f, 0.f);
  float4 qn = make_float4(0.f, 0.f, 0.f, 0.f);
  float raw_norm = 1.0f;

  if (vis) {
    const float4* ap = reinterpret_cast<const float4*>(a.acc + (size_t)idx * ACC_STRIDE);
    acc0 = __ldg(ap);      // dcolor.rgb, dmean2D.x
    acc1 = __ldg(ap + 1);  // dmean2D.y, dconic.a, dconic.b, dconic.c
    acc2 = __ldg(ap + 2);  // dopacity, dL/d(view depth) (slot 9; zero unless the depth gradient was requested)
    mean = make_float3(a.means3D[3 * idx], a.means3D[3 * idx + 1], a.means3D[3 * idx + 2]);

    // ---- 3-D covariance (recomputed; forward.cu:118-152) ----
    float cov3D[6];
    float3 sc = make_float3(0.f, 0.f, 0.f);
    float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
    M3 R, Mm;
    if (a.cov3D_precomp != nullptr) {
#pragma unroll
      for (int k = 0; k < 6; k++) cov3D[k] = a.cov3D_precomp[(size_t)idx * 6 + k];
    } else {
      act_scale = make_float3(a.scales[3 * idx], a.scales[3 * idx + 1], a.scales[3 * idx + 2]);
      q = __ldg(reinterpret_cast<const float4*>(a.rotations) + idx);
      if (RAW) {  // same activations as the RAW forward (preprocess_fwd.cu)
        act_scale = make_float3(expf(act_scale.x), expf(act_scale.y), expf(act_scale.z));
        raw_norm = fmaxf(sqrtf(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w), 1e-12f);
        q = make_float4(__fdiv_rn(q.x, raw_norm), __fdiv_rn(q.y, raw_norm), __fdiv_rn(q.z, raw_norm), __fdiv_rn(q.w, raw_norm));
      }
      sc = make_float3(a.scale_modifier * act_scale.x, a.scale_modifier * act_scale.y, a.scale_modifier * act_scale.z);
      R = quat_to_R(q.x, q.y, q.z, q.w);
      // M = S * R (GLM): M[c][r] = s_r * R[c][r]
#pragma unroll
      for (int c = 0; c < 3; c++) {
        Mm.m[c][0] = sc.x * R.m[c][0];
        Mm.m[c][1] = sc.y * R.m[c][1];
        Mm.m[c][2] = sc.z * R.m[c][2];
      }
      M3 Sigma = mat_mul(mat_t(Mm), Mm);
      cov3D[0] = Sigma.m[0][0]; cov3D[1] = Sigma.m[0][1]; cov3D[2] = Sigma.m[0][2];
      cov3D[3] = Sigma.m[1][1]; cov3D[4] = Sigma.m[1][2]; cov3D[5] = Sigma.m[2][2];
    }

    // ---- backward of the 2-D covariance / conic (backward.cu:164-273) ----
    {
      const float* vm = a.view;
      float3 t;
      t.x = vm[0] * mean.x + vm[4] * mean.y + vm[8] * mean.z + vm[12];
      t.y = vm[1] * mean.x + vm[5] * mean.y + vm[9] * mean.z + vm[13];
      t.z = vm[2] * mean.x + vm[6] * mean.y + vm[10] * mean.z + vm[14];
      const float limx = 1.3f * a.tan_fovx, limy = 1.3f * a.tan_fovy;
      const float txtz = t.x / t.z, tytz = t.y / t.z;
      t.x = fminf(limx, fmaxf(-limx, txtz)) * t.z;
      t.y = fminf(limy, fmaxf(-limy, tytz)) * t.z;
      const float x_grad_mul = (txtz < -limx || txtz > limx) ? 0.f : 1.f;
      const float y_grad_mul = (tytz < -limy || tytz > limy) ? 0.f : 1.f;
      M3 J;
      J.m[0][0] = a.h_x / t.z; J.m[0][1] = 0.f; J.m[0][2] = -(a.h_x * t.x) / (t.z * t.z);
      J.m[1][0] = 0.f; J.m[1][1] = a.h_y / t.z; J.m[1][2] = -(a.h_y * t.y) / (t.z * t.z);
      J.m[2][0] = 0.f; J.m[2][1] = 0.f; J.m[2][2] = 0.f;
      M3 Wm;
      Wm.m[0][0] = vm[0]; Wm.m[0][1] = vm[4]; Wm.m[0][2] = vm[8];
      Wm.m[1][0] = vm[1]; Wm.m[1][1] = vm[5]; Wm.m[1][2] = vm[9];
      Wm.m[2][0] = vm[2]; Wm.m[2][1] = vm[6]; Wm.m[2][2] = vm[10];
      M3 Vrk;
      Vrk.m[0][0] = cov3D[0]; Vrk.m[0][1] = cov3D[1]; Vrk.m[0][2] = cov3D[2];
      Vrk.m[1][0] = cov3D[1]; Vrk.m[1][1] = cov3D[3]; Vrk.m[1][2] = cov3D[4];
      Vrk.m[2][0] = cov3D[2]; Vrk.m[2][1] = cov3D[4]; Vrk.m[2][2] = cov3D[5];
      const M3 T = mat_mul(Wm, J);
      const M3 cov2D = mat_mul(mat_mul(mat_t(T), mat_t(Vrk)), T);
      const float ca = cov2D.m[0][0] + 0.3f, cb = cov2D.m[0][1], cc = cov2D.m[1][1] + 0.3f;
      const float gca = acc1.y, gcb = acc1.z, gcc = acc1.w;  // dL/dconic (a, b, c)
      const float denom = ca * cc - cb * cb;
      float dL_da = 0.f, dL_db = 0.f, dL_dc = 0.f;
      const float denom2inv = 1.0f / ((denom * denom) + 0.0000001f);
      if (denom2inv != 0.f) {
        dL_da = denom2inv * (-cc * cc * gca + 2 * cb * cc * gcb + (denom - ca * cc) * gcc);
        dL_dc = denom2inv * (-ca * ca * gcc + 2 * ca * cb * gcb + (denom - ca * cc) * gca);
        dL_db = denom2inv * 2 * (cb * cc * gca - (denom + 2 * cb * cb) * gcb + ca * cb * gcc);
        dcov[0] = (T.m[0][0] * T.m[0][0] * dL_da + T.m[0][0] * T.m[1][0] * dL_db + T.m[1][0] * T.m[1][0] * dL_dc);
        dcov[3] = (T.m[0][1] * T.m[0][1] * dL_da + T.m[0][1] * T.m[1][1] * dL_db + T.m[1][1] * T.m[1][1] * dL_dc);
        dcov[5] = (T.m[0][2] * T.m[0][2] * dL_da + T.m[0][2] * T.m[1][2] * dL_db + T.m[1][2] * T.m[1][2] * dL_dc);
        dcov[1] = 2 * T.m[0][0] * T.m[0][1] * dL_da + (T.m[0][0] * T.m[1][1] + T.m[0][1] * T.m[1][0]) * dL_db + 2 * T.m[1][0] * T.m[1][1] * dL_dc;
        dcov[2] = 2 * T.m[0][0] * T.m[0][2] * dL_da + (T.m[0][0] * T.m[1][2] + T.m[0][2] * T.m[1][0]) * dL_db + 2 * T.m[1][0] * T.m[1][2] * dL_dc;
        dcov[4] = 2 * T.m[0][2] * T.m[0][1] * dL_da + (T.m[0][1] * T.m[1][2] + T.m[0][2] * T.m[1][1]) * dL_db + 2 * T.m[1][1] * T.m[1][2] * dL_dc;
      }
      // u_i = row i of T against Vrk column j
      float u0[3], u1[3];
#pragma unroll
      for (int j = 0; j < 3; j++) {
        u0[j] = T.m[0][0] * Vrk.m[j][0] + T.m[0][1] * Vrk.m[j][1] + T.m[0][2] * Vrk.m[j][2];
        u1[j] = T.m[1][0] * Vrk.m[j][0] + T.m[1][1] * Vrk.m[j][1] + T.m[1][2] * Vrk.m[j][2];
      }
      const float dL_dT00 = 2 * u0[0] * dL_da + u1[0] * dL_db;
      const float dL_dT01 = 2 * u0[1] * dL_da + u1[1] * dL_db;
      const float dL_dT02 = 2 * u0[2] * dL_da + u1[2] * dL_db;
      const float dL_dT10 = 2 * u1[0] * dL_dc + u0[0] * dL_db;
      const float dL_dT11 = 2 * u1[1] * dL_dc + u0[1] * dL_db;
      const float dL_dT12 = 2 * u1[2] * dL_dc + u0[2] * dL_db;
      const float dL_dJ00 = Wm.m[0][0] * dL_dT00 + Wm.m[0][1] * dL_dT01 + Wm.m[0][2] * dL_dT02;
      const float dL_dJ02 = Wm.m[2][0] * dL_dT00 + Wm.m[2][1] * dL_dT01 + Wm.m[2][2] * dL_dT02;
      const float dL_dJ11 = Wm.m[1][0] * dL_dT10 + Wm.m[1][1] * dL_dT11 + Wm.m[1][2] * dL_dT12;
      const float dL_dJ12 = Wm.m[2][0] * dL_dT10 + Wm.m[2][1] * dL_dT11 + Wm.m[2][2] * dL_dT12;
      const float tz = 1.f / t.z, tz2 = tz * tz, tz3 = tz2 * tz;
      const float dL_dtx = x_grad_mul * -a.h_x * tz2 * dL_dJ02;
      const float dL_dty = y_grad_mul * -a.h_y * tz2 * dL_dJ12;
      float dL_dtz = -a.h_x * tz2 * dL_dJ00 - a.h_y * tz2 * dL_dJ11 + (2 * a.h_x * t.x) * tz3 * dL_dJ02 +
                     (2 * a.h_y * t.y) * tz3 * dL_dJ12;
      // the depth image reads d_i = t.z (unclamped): its gradient joins dL/dt.z and from there the mean, cov3D_precomp,
      // RAW and camera paths below. A uniform branch, not `+ 0`: without the flag the gradients stay bit-identical.
      if (a.depth) dL_dtz += acc2.y;
      // transformVec4x3Transpose (auxiliary.h:89-97)
      dmean[0] = vm[0] * dL_dtx + vm[1] * dL_dty + vm[2] * dL_dtz;
      dmean[1] = vm[4] * dL_dtx + vm[5] * dL_dty + vm[6] * dL_dtz;
      dmean[2] = vm[8] * dL_dtx + vm[9] * dL_dty + vm[10] * dL_dtz;
      if (CAM) {
        // through t = view * mean (same dL/dt, same clamp convention as the mean gradient above)
        const float dt[3] = {dL_dtx, dL_dty, dL_dtz};
        const float mj[4] = {mean.x, mean.y, mean.z, 1.0f};
#pragma unroll
        for (int k = 0; k < 3; k++)
#pragma unroll
          for (int j = 0; j < 4; j++) cg[4 * k + j] += dt[k] * mj[j];
        // through W (the rotation part of view) in T = W * J:  T[0][r] = W[0][r] J00 + W[2][r] J02,
        // T[1][r] = W[1][r] J11 + W[2][r] J12  with W[0] = (v0,v4,v8), W[1] = (v1,v5,v9), W[2] = (v2,v6,v10)
        const float J00 = J.m[0][0], J02 = J.m[0][2], J11 = J.m[1][1], J12 = J.m[1][2];
        const float dT0[3] = {dL_dT00, dL_dT01, dL_dT02}, dT1[3] = {dL_dT10, dL_dT11, dL_dT12};
#pragma unroll
        for (int r = 0; r < 3; r++) {
          cg[4 * 0 + r] += dT0[r] * J00;                    // view[0 + 4r]
          cg[4 * 1 + r] += dT1[r] * J11;                    // view[1 + 4r]
          cg[4 * 2 + r] += dT0[r] * J02 + dT1[r] * J12;     // view[2 + 4r]
        }
      }
    }

    // ---- projection term (backward.cu:372-387) ----
    {
      const float* proj = a.proj;
      const float hw = proj[3] * mean.x + proj[7] * mean.y + proj[11] * mean.z + proj[15];
      const float m_w = 1.0f / (hw + 0.0000001f);
      const float mul1 = (proj[0] * mean.x + proj[4] * mean.y + proj[8] * mean.z + proj[12]) * m_w * m_w;
      const float mul2 = (proj[1] * mean.x + proj[5] * mean.y + proj[9] * mean.z + proj[13]) * m_w * m_w;
      const float g2x = acc0.w, g2y = acc1.x;
      dmean[0] += (proj[0] * m_w - proj[3] * mul1) * g2x + (proj[1] * m_w - proj[3] * mul2) * g2y;
      dmean[1] += (proj[4] * m_w - proj[7] * mul1) * g2x + (proj[5] * m_w - proj[7] * mul2) * g2y;
      dmean[2] += (proj[8] * m_w - proj[11] * mul1) * g2x + (proj[9] * m_w - proj[11] * mul2) * g2y;
      if (CAM) {
        // p_proj = p_hom.xy / (p_hom.w + eps): dL/dp_hom.x = g2x m_w, .y = g2y m_w, .w = -(g2x hx + g2y hy) m_w^2
        const float dh[3] = {g2x * m_w, g2y * m_w, -(g2x * mul1 + g2y * mul2)};
        const float mj[4] = {mean.x, mean.y, mean.z, 1.0f};
#pragma unroll
        for (int r = 0; r < 3; r++)
#pragma unroll
          for (int j = 0; j < 4; j++) cg[12 + 4 * r + j] += dh[r] * mj[j];
      }
    }

    // ---- 3-D covariance -> scale / rotation (backward.cu:278-341) ----
    if (a.cov3D_precomp == nullptr) {
      M3 dSig;
      dSig.m[0][0] = dcov[0]; dSig.m[0][1] = 0.5f * dcov[1]; dSig.m[0][2] = 0.5f * dcov[2];
      dSig.m[1][0] = 0.5f * dcov[1]; dSig.m[1][1] = dcov[3]; dSig.m[1][2] = 0.5f * dcov[4];
      dSig.m[2][0] = 0.5f * dcov[2]; dSig.m[2][1] = 0.5f * dcov[4]; dSig.m[2][2] = dcov[5];
      M3 twoM;
#pragma unroll
      for (int c = 0; c < 3; c++)
#pragma unroll
        for (int r = 0; r < 3; r++) twoM.m[c][r] = Mm.m[c][r] * 2.0f;
      const M3 dL_dM = mat_mul(twoM, dSig);
      const M3 Rt = mat_t(R);
      M3 dMt = mat_t(dL_dM);
      dscale[0] = Rt.m[0][0] * dMt.m[0][0] + Rt.m[0][1] * dMt.m[0][1] + Rt.m[0][2] * dMt.m[0][2];
      dscale[1] = Rt.m[1][0] * dMt.m[1][0] + Rt.m[1][1] * dMt.m[1][1] + Rt.m[1][2] * dMt.m[1][2];
      dscale[2] = Rt.m[2][0] * dMt.m[2][0] + Rt.m[2][1] * dMt.m[2][1] + Rt.m[2][2] * dMt.m[2][2];
#pragma unroll
      for (int k = 0; k < 3; k++) {
        dMt.m[0][k] *= sc.x;
        dMt.m[1][k] *= sc.y;
        dMt.m[2][k] *= sc.z;
      }
      const float r = q.x, x = q.y, y = q.z, z = q.w;
      drot[0] = 2 * z * (dMt.m[0][1] - dMt.m[1][0]) + 2 * y * (dMt.m[2][0] - dMt.m[0][2]) + 2 * x * (dMt.m[1][2] - dMt.m[2][1]);
      drot[1] = 2 * y * (dMt.m[1][0] + dMt.m[0][1]) + 2 * z * (dMt.m[2][0] + dMt.m[0][2]) + 2 * r * (dMt.m[1][2] - dMt.m[2][1]) - 4 * x * (dMt.m[2][2] + dMt.m[1][1]);
      drot[2] = 2 * x * (dMt.m[1][0] + dMt.m[0][1]) + 2 * r * (dMt.m[2][0] - dMt.m[0][2]) + 2 * z * (dMt.m[1][2] + dMt.m[2][1]) - 4 * y * (dMt.m[2][2] + dMt.m[0][0]);
      drot[3] = 2 * r * (dMt.m[0][1] - dMt.m[1][0]) + 2 * x * (dMt.m[2][0] + dMt.m[0][2]) + 2 * y * (dMt.m[1][2] + dMt.m[2][1]) - 4 * z * (dMt.m[1][1] + dMt.m[0][0]);
      qn = q;
    }
  }

  // ---- SH backward (backward.cu:20-139) ----
  // Coefficient by coefficient, four at a time (12 floats = three 128-bit row accesses): read sh[k], add its share to the
  // view-direction gradient, overwrite it IN PLACE with dL/dsh[k] = basis_k * dL/dRGB. Only one 12-float chunk is live
  // at a time (the first version kept all 48 + 48 values in registers: 113 regs, 16 warps/SM).
  if (BULK) mbar_wait(&bar, 0);
  if (RAW && rest_loaded) mbar_wait(&bar, 0);
  if (has_sh && live) {
    const float C0 = 0.28209479177387814f, C1 = 0.4886025119029199f;
    const float C2_0 = 1.0925484305920792f, C2_1 = -1.0925484305920792f, C2_2 = 0.31539156525252005f,
                C2_3 = -1.0925484305920792f, C2_4 = 0.5462742152960396f;
    const float C3_0 = -0.5900435899266435f, C3_1 = 2.890611442640554f, C3_2 = -0.4570457994644658f,
                C3_3 = 0.3731763325901154f, C3_4 = -0.4570457994644658f, C3_5 = 1.445305721320277f,
                C3_6 = -0.5900435899266435f;
    float x = 0.f, y = 0.f, z = 0.f, sum2 = 1.f;
    float3 dir_orig = make_float3(0.f, 0.f, 0.f);
    float dRGB[3] = {0.f, 0.f, 0.f};
    if (vis) {
      dir_orig = make_float3(mean.x - a.campos[0], mean.y - a.campos[1], mean.z - a.campos[2]);
      sum2 = dir_orig.x * dir_orig.x + dir_orig.y * dir_orig.y + dir_orig.z * dir_orig.z;
      const float len = sqrtf(sum2);
      x = dir_orig.x / len; y = dir_orig.y / len; z = dir_orig.z / len;
      const uint8_t cl = a.clamped[idx];
      dRGB[0] = acc0.x * ((cl & 1) ? 0.f : 1.f);   // clamped channels pass no gradient (backward.cu:31-34)
      dRGB[1] = acc0.y * ((cl & 2) ? 0.f : 1.f);
      dRGB[2] = acc0.z * ((cl & 4) ? 0.f : 1.f);
    }
    const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
    float ddir[3] = {0.f, 0.f, 0.f};
    const float* gsrc = a.shs + (size_t)idx * (RAW ? 3 : a.M * 3);     // RAW: features_dc row
    float* gdst = a.dL_dsh + (size_t)idx * (RAW ? 3 : a.M * 3);
    const float* rest_g = RAW ? a.features_rest + (size_t)idx * K3 : nullptr;
    float* drest_g = RAW ? a.dL_dfeatures_rest + (size_t)idx * K3 : nullptr;
    float* rest_s = s_rest + (RAW ? threadIdx.x * K3 : 0);
    const int nw = a.M * 3;
#pragma unroll
    for (int cchunk = 0; cchunk < 4; cchunk++) {
      if (12 * cchunk >= nw) break;  // M = 4: one chunk, M = 16: four (M*12 % 16 == 0 on the BULK path)
      float v[12];
      const bool need = vis && 4 * cchunk < nb;  // this chunk holds active coefficients of a visible Gaussian
      if (BULK) {
#pragma unroll
        for (int q = 0; q < 3; q++) {
          float4 t4 = make_float4(0.f, 0.f, 0.f, 0.f);
          if (need) t4 = *reinterpret_cast<const float4*>(row + 12 * cchunk + 4 * q);
          v[4 * q] = t4.x; v[4 * q + 1] = t4.y; v[4 * q + 2] = t4.z; v[4 * q + 3] = t4.w;
        }
      } else if (RAW) {
#pragma unroll
        for (int i = 0; i < 12; i++) {
          const int e = 12 * cchunk + i;  // element of the virtual [M,3] row: 0..2 = features_dc, the rest features_rest
          float t = 0.f;
          if (need && e < nb * 3) t = e < 3 ? gsrc[e] : (rest_loaded ? rest_s[e - 3] : rest_g[e - 3]);
          v[i] = t;
        }
      } else {
#pragma unroll
        for (int i = 0; i < 12; i++) v[i] = (need && 12 * cchunk + i < nb * 3) ? gsrc[12 * cchunk + i] : 0.f;
      }
      float o12[12];
#pragma unroll
      for (int kk = 0; kk < 4; kk++) {
        const int k = 4 * cchunk + kk;
        // basis_k and its gradient w.r.t. the unit view direction (derivatives as backward.cu:58-122)
        float bk = 0.f, bx = 0.f, by = 0.f, bz = 0.f;
        switch (k) {
          case 0: bk = C0; break;
          case 1: bk = -C1 * y; by = -C1; break;
          case 2: bk = C1 * z; bz = C1; break;
          case 3: bk = -C1 * x; bx = -C1; break;
          case 4: bk = C2_0 * xy; bx = C2_0 * y; by = C2_0 * x; break;
          case 5: bk = C2_1 * yz; by = C2_1 * z; bz = C2_1 * y; break;
          case 6: bk = C2_2 * (2.f * zz - xx - yy); bx = -2.f * C2_2 * x; by = -2.f * C2_2 * y; bz = 4.f * C2_2 * z; break;
          case 7: bk = C2_3 * xz; bx = C2_3 * z; bz = C2_3 * x; break;
          case 8: bk = C2_4 * (xx - yy); bx = 2.f * C2_4 * x; by = -2.f * C2_4 * y; break;
          case 9: bk = C3_0 * y * (3.f * xx - yy); bx = 6.f * C3_0 * xy; by = 3.f * C3_0 * (xx - yy); break;
          case 10: bk = C3_1 * xy * z; bx = C3_1 * yz; by = C3_1 * xz; bz = C3_1 * xy; break;
          case 11: bk = C3_2 * y * (4.f * zz - xx - yy); bx = -2.f * C3_2 * xy; by = C3_2 * (-3.f * yy + 4.f * zz - xx); bz = 8.f * C3_2 * yz; break;
          case 12: bk = C3_3 * z * (2.f * zz - 3.f * xx - 3.f * yy); bx = -6.f * C3_3 * xz; by = -6.f * C3_3 * yz; bz = 3.f * C3_3 * (2.f * zz - xx - yy); break;
          case 13: bk = C3_4 * x * (4.f * zz - xx - yy); bx = C3_4 * (-3.f * xx + 4.f * zz - yy); by = -2.f * C3_4 * xy; bz = 8.f * C3_4 * xz; break;
          case 14: bk = C3_5 * z * (xx - yy); bx = 2.f * C3_5 * xz; by = -2.f * C3_5 * yz; bz = C3_5 * (xx - yy); break;
          default: bk = C3_6 * x * (xx - 3.f * yy); bx = 3.f * C3_6 * (xx - yy); by = -6.f * C3_6 * xy; break;
        }
        const bool active = need && k < nb;
        // contribution of coefficient k to dL/ddir: (d basis_k / d dir) * (sh[k] . dL/dRGB)
        const float dot = v[3 * kk] * dRGB[0] + v[3 * kk + 1] * dRGB[1] + v[3 * kk + 2] * dRGB[2];
        if (active) {
          ddir[0] = fmaf(bx, dot, ddir[0]);
          ddir[1] = fmaf(by, dot, ddir[1]);
          ddir[2] = fmaf(bz, dot, ddir[2]);
        }
        o12[3 * kk] = active ? bk * dRGB[0] : 0.f;
        o12[3 * kk + 1] = active ? bk * dRGB[1] : 0.f;
        o12[3 * kk + 2] = active ? bk * dRGB[2] : 0.f;
      }
      if (BULK) {
#pragma unroll
        for (int q = 0; q < 3; q++)
          *reinterpret_cast<float4*>(row + 12 * cchunk + 4 * q) = make_float4(o12[4 * q], o12[4 * q + 1], o12[4 * q + 2], o12[4 * q + 3]);
      } else if (RAW) {
#pragma unroll
        for (int i = 0; i < 12; i++) {
          const int e = 12 * cchunk + i;
          if (e < 3) gdst[e] = o12[i];
          else if (e < nw) { if (rest_block) rest_s[e - 3] = o12[i]; else drest_g[e - 3] = o12[i]; }
        }
      } else {
#pragma unroll
        for (int i = 0; i < 12; i++)
          if (12 * cchunk + i < nw) gdst[12 * cchunk + i] = o12[i];
      }
    }
    if (vis) {
      // dnormvdv (auxiliary.h:107-117)
      const float invsum32 = 1.0f / sqrtf(sum2 * sum2 * sum2);
      dmean[0] += ((+sum2 - dir_orig.x * dir_orig.x) * ddir[0] - dir_orig.y * dir_orig.x * ddir[1] - dir_orig.z * dir_orig.x * ddir[2]) * invsum32;
      dmean[1] += (-dir_orig.x * dir_orig.y * ddir[0] + (sum2 - dir_orig.y * dir_orig.y) * ddir[1] - dir_orig.z * dir_orig.y * ddir[2]) * invsum32;
      dmean[2] += (-dir_orig.x * dir_orig.z * ddir[0] - dir_orig.y * dir_orig.z * ddir[1] + (sum2 - dir_orig.z * dir_orig.z) * ddir[2]) * invsum32;
      if (CAM) {  // dir = mean - campos: the camera position receives minus what the mean receives through the SH direction
        cg[24] -= ((+sum2 - dir_orig.x * dir_orig.x) * ddir[0] - dir_orig.y * dir_orig.x * ddir[1] - dir_orig.z * dir_orig.x * ddir[2]) * invsum32;
        cg[25] -= (-dir_orig.x * dir_orig.y * ddir[0] + (sum2 - dir_orig.y * dir_orig.y) * ddir[1] - dir_orig.z * dir_orig.y * ddir[2]) * invsum32;
        cg[26] -= (-dir_orig.x * dir_orig.z * ddir[0] - dir_orig.y * dir_orig.z * ddir[1] + (sum2 - dir_orig.z * dir_orig.z) * ddir[2]) * invsum32;
      }
    }
    if (BULK) {
      fence_proxy_async_smem();
      bulk_s2g(gdst, row, (uint32_t)(nw * 4));
      bulk_commit();
    }
  }

  if (live) {
    a.dL_dmeans3D[3 * idx] = dmean[0]; a.dL_dmeans3D[3 * idx + 1] = dmean[1]; a.dL_dmeans3D[3 * idx + 2] = dmean[2];
    a.dL_dmeans2D[3 * idx] = acc0.w; a.dL_dmeans2D[3 * idx + 1] = acc1.x; a.dL_dmeans2D[3 * idx + 2] = 0.f;
    if (a.dL_dcolors) { a.dL_dcolors[3 * idx] = acc0.x; a.dL_dcolors[3 * idx + 1] = acc0.y; a.dL_dcolors[3 * idx + 2] = acc0.z; }
    float dopac = acc2.x;
    if (RAW) {
      // chain rule through the activations: sigmoid' = o(1-o), exp' = exp, and F.normalize: (I - q q^T) / |raw|
      if (vis) {
        const float o = 1.0f / (1.0f + expf(-a.opacities[idx]));
        dopac *= o * (1.0f - o);
      }
      dscale[0] *= act_scale.x; dscale[1] *= act_scale.y; dscale[2] *= act_scale.z;
      const float qd = qn.x * drot[0] + qn.y * drot[1] + qn.z * drot[2] + qn.w * drot[3];
      const float inv = 1.0f / raw_norm;
      drot[0] = (drot[0] - qn.x * qd) * inv; drot[1] = (drot[1] - qn.y * qd) * inv;
      drot[2] = (drot[2] - qn.z * qd) * inv; drot[3] = (drot[3] - qn.w * qd) * inv;
    }
    a.dL_dopacity[idx] = dopac;
    if (a.dL_dcov3D) {
#pragma unroll
      for (int k = 0; k < 6; k++) a.dL_dcov3D[(size_t)idx * 6 + k] = dcov[k];
    }
    a.dL_dscales[3 * idx] = dscale[0]; a.dL_dscales[3 * idx + 1] = dscale[1]; a.dL_dscales[3 * idx + 2] = dscale[2];
    *(reinterpret_cast<float4*>(a.dL_drotations) + idx) = make_float4(drot[0], drot[1], drot[2], drot[3]);
  }
  if (RAW && rest_block) {  // the block of d features_rest rows leaves with one bulk store
    fence_proxy_async_smem();
    __syncthreads();
    if (threadIdx.x == 0) {
      const int first = blockIdx.x * PB_THREADS;
      bulk_s2g(a.dL_dfeatures_rest + (size_t)first * K3, s_rest, (uint32_t)(min(PB_THREADS, a.P - first) * K3 * 4));
      bulk_commit();
      bulk_wait_read0();
    }
  }
  if (BULK) bulk_wait_read0();  // the row must stay valid until the TMA store has read it
  if (CAM) {
    // block partial sums -> cam_partial[block, CAM_STRIDE]; camera_reduce_kernel adds the blocks up (two stages instead
    // of 27 same-address atomics per block)
    __shared__ float s_cam[PB_THREADS / 32][CAM_STRIDE];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < CAM_N; i++) {
      float v = cg[i];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) s_cam[warp][i] = v;
    }
    __syncthreads();
    if (threadIdx.x < CAM_STRIDE) {
      float v = 0.f;
      if (threadIdx.x < CAM_N)
#pragma unroll
        for (int w = 0; w < PB_THREADS / 32; w++) v += s_cam[w][threadIdx.x];
      a.cam_partial[(size_t)blockIdx.x * CAM_STRIDE + threadIdx.x] = v;
    }
  }
}

// sums the per-block partials and scatters the compact layout into dL/dviewmatrix[16], dL/dprojmatrix[16], dL/dcampos[3]
__global__ void __launch_bounds__(1024) camera_reduce_kernel(const float* __restrict__ partial, int nblocks, float* __restrict__ dview,
                                                             float* __restrict__ dproj, float* __restrict__ dcampos) {
  __shared__ float s[32][CAM_STRIDE + 1];
  const int c = threadIdx.x & 31, r = threadIdx.x >> 5;
  float v = 0.f;
  for (int b = r; b < nblocks; b += 32) v += partial[(size_t)b * CAM_STRIDE + c];
  s[r][c] = v;
  __syncthreads();
  if (threadIdx.x < 16) { dview[threadIdx.x] = 0.f; dproj[threadIdx.x] = 0.f; }
  __syncthreads();
  if (r == 0 && c < CAM_N) {
    float t = 0.f;
    for (int k = 0; k < 32; k++) t += s[k][c];
    if (c < 12) dview[(c >> 2) + 4 * (c & 3)] = t;
    else if (c < 24) { const int rr = (c - 12) >> 2, j = (c - 12) & 3; dproj[(rr == 2 ? 3 : rr) + 4 * j] = t; }
    else dcampos[c - 24] = t;
  }
}

}  // namespace

size_t camera_scratch_bytes(int P) { return align_up((size_t)((P + PB_THREADS - 1) / PB_THREADS + 1) * CAM_STRIDE * sizeof(float)); }

int launch_preprocess_bwd(const gsr_settings& s, const gsr_cloud& c, const GeometryWS& g, const int32_t* radii,
                          const float* acc, const gsr_grads& gr, cudaStream_t st, const RawBackward* raw,
                          const CameraBackward* cam, bool depth) {
  PbArgs a;
  a.depth = depth ? 1 : 0;
  a.cam_partial = cam ? cam->scratch : nullptr;
  a.opacities = c.opacities;
  a.features_rest = raw ? raw->features_rest : nullptr;
  a.dL_dfeatures_rest = raw ? raw->dL_dfeatures_rest : nullptr;
  a.P = c.P; a.D = s.sh_degree; a.M = s.sh_coeffs; a.W = s.image_width; a.H = s.image_height;
  a.tan_fovx = s.tanfovx; a.tan_fovy = s.tanfovy;
  a.h_y = a.H / (2.0f * s.tanfovy);
  a.h_x = a.W / (2.0f * s.tanfovx);
  a.scale_modifier = s.scale_modifier;
  a.means3D = c.means3D; a.shs = c.shs; a.scales = c.scales; a.rotations = c.rotations;
  a.cov3D_precomp = c.cov3D_precomp; a.view = s.viewmatrix; a.proj = s.projmatrix; a.campos = s.campos;
  a.radii = radii; a.clamped = g.clamped; a.acc = acc;
  a.dL_dmeans3D = gr.dL_dmeans3D; a.dL_dmeans2D = gr.dL_dmeans2D; a.dL_dcolors = gr.dL_dcolors;
  a.dL_dopacity = gr.dL_dopacity; a.dL_dcov3D = gr.dL_dcov3D; a.dL_dsh = gr.dL_dsh;
  a.dL_dscales = gr.dL_dscales; a.dL_drotations = gr.dL_drotations;
  const int grid = (c.P + PB_THREADS - 1) / PB_THREADS;
  const bool bulk = g_opt.preprocess_variant >= 1 && c.shs != nullptr && gr.dL_dsh != nullptr &&
                    (s.sh_coeffs * 12) % 16 == 0 && s.sh_coeffs * 12 <= 192 &&
                    (reinterpret_cast<uintptr_t>(c.shs) % 16) == 0 && (reinterpret_cast<uintptr_t>(gr.dL_dsh) % 16) == 0;
  if (cam) {  // opt-in camera gradients (never together with the RAW entry point)
    if (raw) { set_error("camera gradients are not available on the fused-activation entry point"); return GSR_ERR_INVALID; }
    if (bulk)
      preprocess_bwd_kernel<true, false, true><<<grid, PB_THREADS, 0, st>>>(a);
    else
      preprocess_bwd_kernel<false, false, true><<<grid, PB_THREADS, 0, st>>>(a);
    camera_reduce_kernel<<<1, 1024, 0, st>>>(cam->scratch, grid, cam->dL_dviewmatrix, cam->dL_dprojmatrix, cam->dL_dcampos);
    g_launches += 2;
    return check_launch("preprocess_bwd (camera)", s.debug != 0, st);
  }
  if (raw)
    preprocess_bwd_kernel<false, true><<<grid, PB_THREADS, 0, st>>>(a);
  else if (bulk)
    preprocess_bwd_kernel<true><<<grid, PB_THREADS, 0, st>>>(a);
  else
    preprocess_bwd_kernel<false><<<grid, PB_THREADS, 0, st>>>(a);
  g_launches++;
  return check_launch("preprocess_bwd", s.debug != 0, st);
}

}  // namespace gsr
