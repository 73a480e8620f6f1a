// C ABI of libgsr_b200.so (include/gsr_b200.h): argument checks, workspace carving, stage orchestration.
// Orchestration mirrors CudaRasterizer::Rasterizer::{forward,backward,markVisible,apply_weights}
// (cuda_rasterizer/rasterizer_impl.cu:128-133,179-285,289-341,343-446) with the forward split in two halves
// around the single host read of num_rendered.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <vector>

#include "common.cuh"

namespace gsr {

Options g_opt;
unsigned long long* g_stats_dev = nullptr;
std::atomic<long long> g_launches{0};
static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int check_cuda(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return GSR_OK;
  set_error("CUDA error in %s: %s", what, cudaGetErrorString(e));
  return GSR_ERR_CUDA;
}
int check_launch(const char* what, bool debug, cudaStream_t st) {
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess && debug) e = cudaStreamSynchronize(st);
  return check_cuda(e, what);
}

struct ProfRec { int stage; cudaEvent_t a, b; };
static std::vector<ProfRec*> g_prof;
static std::mutex g_prof_mu;  // autograd runs the backward on its own thread while the main thread may be in a forward
StageScope::StageScope(int stage_, cudaStream_t st_) : stage(stage_), st(st_), rec(nullptr) {
  if (!g_opt.profile) return;
  ProfRec* r = new ProfRec();
  r->stage = stage;
  cudaEventCreate(&r->a);
  cudaEventCreate(&r->b);
  cudaEventRecord(r->a, st);
  rec = r;
}
StageScope::~StageScope() {
  if (!rec) return;
  ProfRec* r = (ProfRec*)rec;
  cudaEventRecord(r->b, st);
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof.push_back(r);
}

int validate_cloud(const gsr_settings* s, const gsr_cloud* c) {
  if (!s || !c) { set_error("null settings/cloud"); return GSR_ERR_INVALID; }
  if (c->P < 0 || s->image_width < 0 || s->image_height < 0) { set_error("negative size"); return GSR_ERR_INVALID; }
  if (c->P == 0) return GSR_OK;  // nothing to read; rasterize_points.cu:72,130 short-circuit the same way
  if (!c->means3D || !c->opacities) { set_error("means3D / opacities must not be null"); return GSR_ERR_INVALID; }
  // diff_gaussian_rasterization/__init__.py:271-283
  if ((c->shs == nullptr) == (c->colors_precomp == nullptr)) {
    set_error("Please provide excatly one of either SHs or precomputed colors!");
    return GSR_ERR_INVALID;
  }
  const bool sr = c->scales != nullptr && c->rotations != nullptr;
  if (((c->scales == nullptr || c->rotations == nullptr) && c->cov3D_precomp == nullptr) ||
      ((c->scales != nullptr || c->rotations != nullptr) && c->cov3D_precomp != nullptr)) {
    set_error("Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!");
    return GSR_ERR_INVALID;
  }
  if (sr && (reinterpret_cast<uintptr_t>(c->rotations) & 15)) { set_error("rotations must be 16-byte aligned"); return GSR_ERR_INVALID; }
  if (c->shs) {
    if (s->sh_degree < 0 || s->sh_degree > 3 || (s->sh_degree + 1) * (s->sh_degree + 1) > s->sh_coeffs || s->sh_coeffs > 16) {
      set_error("sh_degree %d needs %d <= sh_coeffs %d <= 16", s->sh_degree, (s->sh_degree + 1) * (s->sh_degree + 1), s->sh_coeffs);
      return GSR_ERR_INVALID;
    }
  }
  if (!s->bg || !s->viewmatrix || !s->projmatrix || !s->campos) { set_error("camera pointers must not be null"); return GSR_ERR_INVALID; }
  return GSR_OK;
}

}  // namespace gsr

using namespace gsr;

extern "C" {

int gsr_abi_version(void) { return GSR_ABI_VERSION; }
const char* gsr_last_error(void) { return g_err; }

size_t gsr_geometry_bytes(int32_t P) {
  GeometryWS ws;
  if (!carve_geometry(nullptr, P, ws)) return 0;
  return ws.total;
}
size_t gsr_image_bytes(int32_t W, int32_t H) {
  ImageWS ws;
  carve_image(nullptr, W, H, ws);
  return ws.total;
}
size_t gsr_binning_bytes(int32_t P, int64_t R, int32_t W, int32_t H) {
  BinningWS ws;
  if (!carve_binning(nullptr, P, R, W, H, ws)) return 0;
  return ws.total;
}
size_t gsr_backward_scratch_bytes(int32_t P) { return align_up((size_t)(P > 0 ? P : 1) * ACC_STRIDE * sizeof(float)); }

// First forward half on a carved workspace: preprocess, depth order, tile-count scan, and the copy of num_rendered to
// the host. With the tile-binning path (tile_binning.cu) the preprocess kernel accumulates the count itself, so the copy
// is issued right behind it and the host learns R while the GPU is still sorting.
static int first_half(const gsr_settings& s, const gsr_cloud& c, const GeometryWS& g, int32_t* radii,
                      int32_t* num_rendered_host, cudaStream_t st, bool raw, const float* features_rest) {
  const int gx = (s.image_width + TILE - 1) / TILE, gy = (s.image_height + TILE - 1) / TILE;
  const bool v2 = tile_binning_supported(gx, gy);
  int rc;
  {
    StageScope t(ST_PRE_FWD, st);
    if (v2 && (rc = clear_tile_counts(g, gx, gy, st))) return rc;
    rc = launch_preprocess_fwd(s, c, g, radii, st, nullptr, 0, raw, features_rest, v2);
    if (rc) return rc;
    if (v2) {
      if ((rc = launch_tile_count(g, gx, gy, TileOwner(), st))) return rc;
      cudaError_t e = cudaMemcpyAsync(num_rendered_host, g.R_dev, sizeof(int32_t), cudaMemcpyDeviceToHost, st);
      if (e != cudaSuccess) return check_cuda(e, "num_rendered readback");
    }
  }
  StageScope t(ST_DEPTH_SCAN, st);
  return run_depth_order_and_scan(c, g, v2 ? nullptr : num_rendered_host, st, s.debug != 0);
}

int gsr_forward_preprocess(const gsr_settings* s, const gsr_cloud* c, void* geometry, size_t geometry_bytes,
                           int32_t* radii, int32_t* num_rendered_host, void* stream) {
  int rc = validate_cloud(s, c);
  if (rc) return rc;
  if (!num_rendered_host) { set_error("num_rendered_host is null"); return GSR_ERR_INVALID; }
  cudaStream_t st = (cudaStream_t)stream;
  if (c->P == 0) { *num_rendered_host = 0; return GSR_OK; }
  if (!radii || !geometry) { set_error("radii / geometry workspace is null"); return GSR_ERR_INVALID; }
  GeometryWS g;
  if (!carve_geometry(geometry, c->P, g)) return GSR_ERR_CUDA;
  if (g.total > geometry_bytes) { set_error("geometry workspace too small: %zu < %zu", geometry_bytes, g.total); return GSR_ERR_WORKSPACE; }
  return first_half(*s, *c, g, radii, num_rendered_host, st, false, nullptr);
}

static int carve_all(const gsr_settings* s, const gsr_cloud* c, int64_t R, void* geometry, size_t gb, void* binning,
                     size_t bb, void* image, size_t ib, GeometryWS& g, BinningWS& b, ImageWS& im) {
  if (!carve_geometry(geometry, c->P, g)) return GSR_ERR_CUDA;
  if (g.total > gb) { set_error("geometry workspace too small: %zu < %zu", gb, g.total); return GSR_ERR_WORKSPACE; }
  if (!carve_binning(binning, c->P, R, s->image_width, s->image_height, b)) return GSR_ERR_CUDA;
  if (R > 0 && (b.total > bb || !binning)) { set_error("binning workspace too small: %zu < %zu", bb, b.total); return GSR_ERR_WORKSPACE; }
  carve_image(image, s->image_width, s->image_height, im);
  if (im.total > ib || !image) { set_error("image workspace too small: %zu < %zu", ib, im.total); return GSR_ERR_WORKSPACE; }
  return GSR_OK;
}

static int forward_render_impl(const gsr_settings* s, const gsr_cloud* c, int32_t R, bool speculative, void* geometry,
                               size_t geometry_bytes, void* binning, size_t binning_bytes, void* image,
                               size_t image_bytes, const int32_t* radii, float* out_color, float* out_depth,
                               void* stream) {
  int rc = validate_cloud(s, c);
  if (rc) return rc;
  if (!out_color || !out_depth) { set_error("output images are null"); return GSR_ERR_INVALID; }
  cudaStream_t st = (cudaStream_t)stream;
  const size_t npix = (size_t)s->image_width * s->image_height;
  if (c->P == 0) {  // rasterize_points.cu:72 -- outputs stay zero
    cudaError_t e = cudaMemsetAsync(out_color, 0, 3 * npix * sizeof(float), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(out_depth, 0, npix * sizeof(float), st);
    return check_cuda(e, "zero outputs");
  }
  GeometryWS g; BinningWS b; ImageWS im;
  rc = carve_all(s, c, R, geometry, geometry_bytes, binning, binning_bytes, image, image_bytes, g, b, im);
  if (rc) return rc;
  rc = run_binning(*s, *c, R, speculative, g, b, im, radii, st);
  if (rc) return rc;
  StageScope t(ST_RENDER_FWD, st);
  return launch_render_fwd(*s, g, b, im, out_color, out_depth, st);
}

int gsr_forward_render(const gsr_settings* s, const gsr_cloud* c, int32_t R, void* geometry, size_t geometry_bytes,
                       void* binning, size_t binning_bytes, void* image, size_t image_bytes, const int32_t* radii,
                       float* out_color, float* out_depth, void* stream) {
  return forward_render_impl(s, c, R, false, geometry, geometry_bytes, binning, binning_bytes, image, image_bytes, radii,
                             out_color, out_depth, stream);
}

int gsr_forward_render_speculative(const gsr_settings* s, const gsr_cloud* c, int32_t capacity, void* geometry,
                                   size_t geometry_bytes, void* binning, size_t binning_bytes, void* image,
                                   size_t image_bytes, const int32_t* radii, float* out_color, float* out_depth,
                                   void* stream) {
  if (capacity <= 0) { set_error("speculative capacity must be positive"); return GSR_ERR_INVALID; }
  return forward_render_impl(s, c, capacity, true, geometry, geometry_bytes, binning, binning_bytes, image, image_bytes,
                             radii, out_color, out_depth, stream);
}

static int backward_impl(const gsr_settings* s, const gsr_cloud* c, int32_t R, const void* geometry, size_t geometry_bytes,
                         const void* binning, size_t binning_bytes, const void* image, size_t image_bytes,
                         const int32_t* radii, const float* dL_dout_color, const float* dL_dout_alpha, void* scratch,
                         size_t scratch_bytes, const gsr_grads* gr, void* stream, const gsr_camera_grads* cam = nullptr,
                         const float* dL_dout_depth = nullptr) {
  int rc = validate_cloud(s, c);
  if (rc) return rc;
  if (!gr || !dL_dout_color) { set_error("grads / dL_dout_color is null"); return GSR_ERR_INVALID; }
  if (c->P == 0) return GSR_OK;
  if (!gr->dL_dmeans3D || !gr->dL_dmeans2D || !gr->dL_dcolors || !gr->dL_dopacity || !gr->dL_dcov3D ||
      !gr->dL_dscales || !gr->dL_drotations || (c->shs && !gr->dL_dsh)) {
    set_error("a gradient output pointer is null");
    return GSR_ERR_INVALID;
  }
  if (reinterpret_cast<uintptr_t>(gr->dL_drotations) & 15) { set_error("dL_drotations must be 16-byte aligned"); return GSR_ERR_INVALID; }
  cudaStream_t st = (cudaStream_t)stream;
  GeometryWS g; BinningWS b; ImageWS im;
  rc = carve_all(s, c, R, const_cast<void*>(geometry), geometry_bytes, const_cast<void*>(binning), binning_bytes,
                 const_cast<void*>(image), image_bytes, g, b, im);
  if (rc) return rc;
  const size_t need = gsr_backward_scratch_bytes(c->P);
  if (!scratch || scratch_bytes < need) { set_error("backward scratch too small: %zu < %zu", scratch_bytes, need); return GSR_ERR_WORKSPACE; }
  {
    StageScope t(ST_RENDER_BWD, st);  // includes zeroing the accumulators
    cudaError_t e = cudaMemsetAsync(scratch, 0, (size_t)c->P * ACC_STRIDE * sizeof(float), st);
    if (e != cudaSuccess) return check_cuda(e, "scratch memset");
    if (R > 0) {
      rc = launch_render_bwd(*s, g, b, im, dL_dout_color, (float*)scratch, st, TileOwner(), dL_dout_alpha, dL_dout_depth);
      if (rc) return rc;
    }
  }
  StageScope t(ST_PRE_BWD, st);
  if (cam) {
    if (!cam->dL_dviewmatrix || !cam->dL_dprojmatrix || !cam->dL_dcampos || !cam->scratch ||
        cam->scratch_bytes < camera_scratch_bytes(c->P)) {
      set_error("camera gradients: null output or scratch smaller than gsr_camera_scratch_bytes(P)");
      return GSR_ERR_INVALID;
    }
    CameraBackward cb{cam->dL_dviewmatrix, cam->dL_dprojmatrix, cam->dL_dcampos, (float*)cam->scratch};
    return launch_preprocess_bwd(*s, *c, g, radii, (const float*)scratch, *gr, st, nullptr, &cb, dL_dout_depth != nullptr);
  }
  return launch_preprocess_bwd(*s, *c, g, radii, (const float*)scratch, *gr, st, nullptr, nullptr, dL_dout_depth != nullptr);
}

size_t gsr_camera_scratch_bytes(int32_t P) { return camera_scratch_bytes(P > 0 ? P : 1); }

// P == 0: nothing contributes, the camera gradients are zero (the backward itself returns before any launch)
static int zero_camera_grads(const gsr_camera_grads* cam, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaSuccess;
  if (cam->dL_dviewmatrix) e = cudaMemsetAsync(cam->dL_dviewmatrix, 0, 64, st);
  if (e == cudaSuccess && cam->dL_dprojmatrix) e = cudaMemsetAsync(cam->dL_dprojmatrix, 0, 64, st);
  if (e == cudaSuccess && cam->dL_dcampos) e = cudaMemsetAsync(cam->dL_dcampos, 0, 12, st);
  return e == cudaSuccess ? GSR_OK : check_cuda(e, "camera gradient memset");
}

int gsr_backward_camera(const gsr_settings* s, const gsr_cloud* c, int32_t R, const void* geometry, size_t geometry_bytes,
                        const void* binning, size_t binning_bytes, const void* image, size_t image_bytes,
                        const int32_t* radii, const float* dL_dout_color, const float* dL_dout_alpha, void* scratch,
                        size_t scratch_bytes, const gsr_grads* gr, const gsr_camera_grads* cam, void* stream) {
  if (!cam) { set_error("camera gradients: null struct"); return GSR_ERR_INVALID; }
  if (c && c->P == 0) {
    int rc = zero_camera_grads(cam, stream);
    if (rc) return rc;
  }
  return backward_impl(s, c, R, geometry, geometry_bytes, binning, binning_bytes, image, image_bytes, radii,
                       dL_dout_color, dL_dout_alpha, scratch, scratch_bytes, gr, stream, cam);
}

int gsr_backward_depth(const gsr_settings* s, const gsr_cloud* c, int32_t R, const void* geometry, size_t geometry_bytes,
                       const void* binning, size_t binning_bytes, const void* image, size_t image_bytes,
                       const int32_t* radii, const float* dL_dout_color, const float* dL_dout_alpha,
                       const float* dL_dout_depth, void* scratch, size_t scratch_bytes, const gsr_grads* gr,
                       const gsr_camera_grads* cam, void* stream) {
  if (!dL_dout_depth) { set_error("depth gradients: dL_dout_depth is null"); return GSR_ERR_INVALID; }
  if (cam && c && c->P == 0) {
    int rc = zero_camera_grads(cam, stream);
    if (rc) return rc;
  }
  return backward_impl(s, c, R, geometry, geometry_bytes, binning, binning_bytes, image, image_bytes, radii,
                       dL_dout_color, dL_dout_alpha, scratch, scratch_bytes, gr, stream, cam, dL_dout_depth);
}

int gsr_backward(const gsr_settings* s, const gsr_cloud* c, int32_t R, const void* geometry, size_t geometry_bytes,
                 const void* binning, size_t binning_bytes, const void* image, size_t image_bytes,
                 const int32_t* radii, const float* dL_dout_color, void* scratch, size_t scratch_bytes,
                 const gsr_grads* gr, void* stream) {
  return backward_impl(s, c, R, geometry, geometry_bytes, binning, binning_bytes, image, image_bytes, radii,
                       dL_dout_color, nullptr, scratch, scratch_bytes, gr, stream);
}

int gsr_backward_alpha(const gsr_settings* s, const gsr_cloud* c, int32_t R, const void* geometry, size_t geometry_bytes,
                       const void* binning, size_t binning_bytes, const void* image, size_t image_bytes,
                       const int32_t* radii, const float* dL_dout_color, const float* dL_dout_alpha, void* scratch,
                       size_t scratch_bytes, const gsr_grads* gr, void* stream) {
  return backward_impl(s, c, R, geometry, geometry_bytes, binning, binning_bytes, image, image_bytes, radii,
                       dL_dout_color, dL_dout_alpha, scratch, scratch_bytes, gr, stream);
}

int gsr_alpha_image(const void* image, size_t image_bytes, int32_t W, int32_t H, float* out_alpha, void* stream) {
  if (W < 0 || H < 0 || !out_alpha || !image) { set_error("alpha_image: bad arguments"); return GSR_ERR_INVALID; }
  ImageWS im;
  carve_image(const_cast<void*>(image), W, H, im);
  if (im.total > image_bytes) { set_error("image workspace too small: %zu < %zu", image_bytes, im.total); return GSR_ERR_WORKSPACE; }
  const size_t n = (size_t)W * H;
  if (n == 0) return GSR_OK;
  return launch_alpha_image(im.final_T, n, out_alpha, (cudaStream_t)stream);
}

int gsr_mark_visible(int32_t P, const float* means3D, const float* viewmatrix, const float* projmatrix,
                     uint8_t* present, void* stream) {
  (void)projmatrix;
  if (P < 0 || (P > 0 && (!means3D || !viewmatrix || !present))) { set_error("mark_visible: bad arguments"); return GSR_ERR_INVALID; }
  if (P == 0) return GSR_OK;
  return launch_mark_visible(P, means3D, viewmatrix, present, (cudaStream_t)stream);
}

int gsr_apply_weights(const gsr_settings* s, const gsr_cloud* c, int32_t R, void* geometry, size_t geometry_bytes,
                      void* binning, size_t binning_bytes, void* image, size_t image_bytes, const int32_t* radii,
                      const float* image_weights, int32_t CH, float* weights, int32_t* cnt, void* stream) {
  int rc = validate_cloud(s, c);
  if (rc) return rc;
  if (!image_weights || !weights || !cnt) { set_error("apply_weights: null buffer"); return GSR_ERR_INVALID; }
  if (c->P == 0 || R <= 0) return GSR_OK;
  cudaStream_t st = (cudaStream_t)stream;
  GeometryWS g; BinningWS b; ImageWS im;
  rc = carve_all(s, c, R, geometry, geometry_bytes, binning, binning_bytes, image, image_bytes, g, b, im);
  if (rc) return rc;
  rc = run_binning(*s, *c, R, false, g, b, im, radii, st);
  if (rc) return rc;
  StageScope t(ST_APPLY_W, st);
  return launch_apply_weights(*s, g, b, im, image_weights, CH, weights, cnt, st);
}

// ---- fused activations (raw parameters) --------------------------------------------------------------------
static int raw_to_cloud(const gsr_settings* s, const gsr_raw_cloud* r, gsr_cloud& c) {
  if (!s || !r) { set_error("null settings/cloud"); return GSR_ERR_INVALID; }
  c = gsr_cloud{};
  c.P = r->P; c.means3D = r->means3D; c.opacities = r->opacity_logits; c.shs = r->features_dc;
  c.scales = r->log_scales; c.rotations = r->raw_rotations;
  int rc = validate_cloud(s, &c);
  if (rc) return rc;
  if (r->P > 0 && s->sh_coeffs > 1 && !r->features_rest) { set_error("features_rest is null but sh_coeffs = %d", s->sh_coeffs); return GSR_ERR_INVALID; }
  if (r->features_rest && (reinterpret_cast<uintptr_t>(r->features_rest) & 15)) { set_error("features_rest must be 16-byte aligned"); return GSR_ERR_INVALID; }
  return GSR_OK;
}

int gsr_forward_preprocess_raw(const gsr_settings* s, const gsr_raw_cloud* r, void* geometry, size_t geometry_bytes,
                               int32_t* radii, int32_t* num_rendered_host, void* stream) {
  gsr_cloud c;
  int rc = raw_to_cloud(s, r, c);
  if (rc) return rc;
  if (!num_rendered_host) { set_error("num_rendered_host is null"); return GSR_ERR_INVALID; }
  cudaStream_t st = (cudaStream_t)stream;
  if (c.P == 0) { *num_rendered_host = 0; return GSR_OK; }
  if (!radii || !geometry) { set_error("radii / geometry workspace is null"); return GSR_ERR_INVALID; }
  GeometryWS g;
  if (!carve_geometry(geometry, c.P, g)) return GSR_ERR_CUDA;
  if (g.total > geometry_bytes) { set_error("geometry workspace too small: %zu < %zu", geometry_bytes, g.total); return GSR_ERR_WORKSPACE; }
  return first_half(*s, c, g, radii, num_rendered_host, st, true, r->features_rest);
}

static int backward_raw_impl(const gsr_settings* s, const gsr_raw_cloud* r, int32_t R, const void* geometry,
                             size_t geometry_bytes, const void* binning, size_t binning_bytes, const void* image,
                             size_t image_bytes, const int32_t* radii, const float* dL_dout_color, void* scratch,
                             size_t scratch_bytes, const gsr_raw_grads* gr, void* stream,
                             const float* dL_dout_depth = nullptr) {
  gsr_cloud c;
  int rc = raw_to_cloud(s, r, c);
  if (rc) return rc;
  if (!gr || !dL_dout_color) { set_error("grads / dL_dout_color is null"); return GSR_ERR_INVALID; }
  if (c.P == 0) return GSR_OK;
  if (!gr->dL_dmeans3D || !gr->dL_dmeans2D || !gr->dL_dopacity_logits || !gr->dL_dfeatures_dc || !gr->dL_dlog_scales ||
      !gr->dL_draw_rotations || (s->sh_coeffs > 1 && !gr->dL_dfeatures_rest)) {
    set_error("a gradient output pointer is null");
    return GSR_ERR_INVALID;
  }
  if ((reinterpret_cast<uintptr_t>(gr->dL_draw_rotations) & 15) || (reinterpret_cast<uintptr_t>(gr->dL_dfeatures_rest) & 15)) {
    set_error("dL_draw_rotations / dL_dfeatures_rest must be 16-byte aligned");
    return GSR_ERR_INVALID;
  }
  cudaStream_t st = (cudaStream_t)stream;
  GeometryWS g; BinningWS b; ImageWS im;
  rc = carve_all(s, &c, R, const_cast<void*>(geometry), geometry_bytes, const_cast<void*>(binning), binning_bytes,
                 const_cast<void*>(image), image_bytes, g, b, im);
  if (rc) return rc;
  const size_t need = gsr_backward_scratch_bytes(c.P);
  if (!scratch || scratch_bytes < need) { set_error("backward scratch too small: %zu < %zu", scratch_bytes, need); return GSR_ERR_WORKSPACE; }
  {
    StageScope t(ST_RENDER_BWD, st);
    cudaError_t e = cudaMemsetAsync(scratch, 0, (size_t)c.P * ACC_STRIDE * sizeof(float), st);
    if (e != cudaSuccess) return check_cuda(e, "scratch memset");
    if (R > 0) {
      rc = launch_render_bwd(*s, g, b, im, dL_dout_color, (float*)scratch, st, TileOwner(), nullptr, dL_dout_depth);
      if (rc) return rc;
    }
  }
  gsr_grads full{};
  full.dL_dmeans3D = gr->dL_dmeans3D; full.dL_dmeans2D = gr->dL_dmeans2D; full.dL_dopacity = gr->dL_dopacity_logits;
  full.dL_dsh = gr->dL_dfeatures_dc; full.dL_dscales = gr->dL_dlog_scales; full.dL_drotations = gr->dL_draw_rotations;
  RawBackward raw{r->features_rest, gr->dL_dfeatures_rest};
  StageScope t(ST_PRE_BWD, st);
  return launch_preprocess_bwd(*s, c, g, radii, (const float*)scratch, full, st, &raw, nullptr, dL_dout_depth != nullptr);
}

int gsr_backward_raw(const gsr_settings* s, const gsr_raw_cloud* r, int32_t R, const void* geometry,
                     size_t geometry_bytes, const void* binning, size_t binning_bytes, const void* image,
                     size_t image_bytes, const int32_t* radii, const float* dL_dout_color, void* scratch,
                     size_t scratch_bytes, const gsr_raw_grads* gr, void* stream) {
  return backward_raw_impl(s, r, R, geometry, geometry_bytes, binning, binning_bytes, image, image_bytes, radii,
                           dL_dout_color, scratch, scratch_bytes, gr, stream);
}

int gsr_backward_raw_depth(const gsr_settings* s, const gsr_raw_cloud* r, int32_t R, const void* geometry,
                           size_t geometry_bytes, const void* binning, size_t binning_bytes, const void* image,
                           size_t image_bytes, const int32_t* radii, const float* dL_dout_color,
                           const float* dL_dout_depth, void* scratch, size_t scratch_bytes, const gsr_raw_grads* gr,
                           void* stream) {
  if (!dL_dout_depth) { set_error("depth gradients: dL_dout_depth is null"); return GSR_ERR_INVALID; }
  return backward_raw_impl(s, r, R, geometry, geometry_bytes, binning, binning_bytes, image, image_bytes, radii,
                           dL_dout_color, scratch, scratch_bytes, gr, stream, dL_dout_depth);
}

// ---- Gaussian-sharded multi-GPU path ---------------------------------------------------------------------
static int check_owner(const gsr_tile_owner* o, TileOwner& own) {
  if (!o || o->row_stride < 1 || o->row_phase < 0 || o->row_phase >= o->row_stride) {
    set_error("tile owner: need row_stride >= 1 and 0 <= row_phase < row_stride");
    return GSR_ERR_INVALID;
  }
  own.stride = o->row_stride; own.phase = o->row_phase;
  return GSR_OK;
}
static int check_settings(const gsr_settings* s) {
  if (!s) { set_error("null settings"); return GSR_ERR_INVALID; }
  if (s->image_width < 0 || s->image_height < 0) { set_error("negative size"); return GSR_ERR_INVALID; }
  if (!s->bg || !s->viewmatrix || !s->projmatrix || !s->campos) { set_error("camera pointers must not be null"); return GSR_ERR_INVALID; }
  return GSR_OK;
}
// the slice [base, base+n) of the per-Gaussian arrays of a P_total-sized geometry workspace
static GeometryWS slice_geometry(const GeometryWS& g, int base) {
  GeometryWS l = g;
  l.records += base; l.tiles_touched += base; l.clamped += base; l.depth_keys += base; l.ident += base;
  return l;
}

int gsr_view_exchange(void* geometry, int32_t P_total, gsr_exchange_view* out) {
  GeometryWS g;
  if (!out || P_total < 0 || !carve_geometry(geometry, P_total, g)) return GSR_ERR_INVALID;
  out->records = g.records;
  return GSR_OK;
}

int gsr_shard_preprocess(const gsr_settings* s, const gsr_cloud* shard, int32_t P_total, int32_t index_base,
                         int32_t slice_len, void* geometry, size_t geometry_bytes, int32_t* radii_total, void* stream) {
  int rc = validate_cloud(s, shard);
  if (rc) return rc;
  if (P_total <= 0 || index_base < 0 || slice_len < shard->P || (int64_t)index_base + slice_len > P_total) {
    set_error("shard [%d, %d+%d) (P=%d) does not fit P_total=%d", index_base, index_base, slice_len, shard->P, P_total);
    return GSR_ERR_INVALID;
  }
  if (!radii_total || !geometry) { set_error("radii / geometry workspace is null"); return GSR_ERR_INVALID; }
  cudaStream_t st = (cudaStream_t)stream;
  GeometryWS g;
  if (!carve_geometry(geometry, P_total, g)) return GSR_ERR_CUDA;
  if (g.total > geometry_bytes) { set_error("geometry workspace too small: %zu < %zu", geometry_bytes, g.total); return GSR_ERR_WORKSPACE; }
  StageScope t(ST_PRE_FWD, st);
  if (shard->P > 0) {
    rc = launch_preprocess_fwd(*s, *shard, slice_geometry(g, index_base), radii_total + index_base, st);
    if (rc) return rc;
  }
  const int pad = slice_len - shard->P;  // slots of the slice behind the shard: culled (radius 0 in the record)
  if (pad > 0) {
    cudaError_t e = cudaMemsetAsync(g.records + index_base + shard->P, 0, (size_t)pad * sizeof(SplatRecord), st);
    if (e != cudaSuccess) return check_cuda(e, "slice padding");
  }
  return GSR_OK;
}

int gsr_peer_alloc(size_t bytes, void** ptr_out, void* handle_out) {
  if (!ptr_out || !handle_out || bytes == 0) { set_error("peer_alloc: bad arguments"); return GSR_ERR_INVALID; }
  static_assert(sizeof(cudaIpcMemHandle_t) <= GSR_PEER_HANDLE_BYTES, "IPC handle size");
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e != cudaSuccess) return check_cuda(e, "peer_alloc cudaMalloc");
  cudaIpcMemHandle_t h;
  e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) { cudaFree(p); return check_cuda(e, "cudaIpcGetMemHandle"); }
  memset(handle_out, 0, GSR_PEER_HANDLE_BYTES);
  memcpy(handle_out, &h, sizeof(h));
  *ptr_out = p;
  return GSR_OK;
}
int gsr_peer_open(const void* handle, void** ptr_out) {
  if (!handle || !ptr_out) { set_error("peer_open: bad arguments"); return GSR_ERR_INVALID; }
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  void* p = nullptr;
  cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) return check_cuda(e, "cudaIpcOpenMemHandle");
  *ptr_out = p;
  return GSR_OK;
}
int gsr_peer_close(void* ptr) { return ptr ? check_cuda(cudaIpcCloseMemHandle(ptr), "cudaIpcCloseMemHandle") : GSR_OK; }
int gsr_peer_free(void* ptr) { return ptr ? check_cuda(cudaFree(ptr), "peer_free") : GSR_OK; }

int gsr_shard_preprocess_p2p(const gsr_settings* s, const gsr_cloud* shard, int32_t P_total, int32_t index_base,
                             int32_t slice_len, void* const* peer_geometry, int32_t world, int32_t rank,
                             size_t geometry_bytes, int32_t* radii_total, void* stream) {
  int rc = validate_cloud(s, shard);
  if (rc) return rc;
  if (world < 1 || world > GSR_MAX_PEERS || rank < 0 || rank >= world || !peer_geometry) {
    set_error("p2p preprocess: need 1 <= world <= %d, 0 <= rank < world", GSR_MAX_PEERS);
    return GSR_ERR_INVALID;
  }
  if (P_total <= 0 || index_base < 0 || slice_len < shard->P || (int64_t)index_base + slice_len > P_total) {
    set_error("shard [%d, %d+%d) (P=%d) does not fit P_total=%d", index_base, index_base, slice_len, shard->P, P_total);
    return GSR_ERR_INVALID;
  }
  if (!radii_total) { set_error("radii is null"); return GSR_ERR_INVALID; }
  cudaStream_t st = (cudaStream_t)stream;
  GeometryWS g;  // own workspace: everything but the records is local
  if (!peer_geometry[rank] || !carve_geometry(peer_geometry[rank], P_total, g)) return GSR_ERR_CUDA;
  if (g.total > geometry_bytes) { set_error("geometry workspace too small: %zu < %zu", geometry_bytes, g.total); return GSR_ERR_WORKSPACE; }
  SplatRecord* dst[GSR_MAX_PEERS];
  for (int r = 0; r < world; r++) {
    GeometryWS gr;
    if (!peer_geometry[r] || !carve_geometry(peer_geometry[r], P_total, gr)) { set_error("peer workspace %d is null", r); return GSR_ERR_INVALID; }
    dst[r] = gr.records + index_base;
  }
  StageScope t(ST_PRE_FWD, st);
  if (shard->P > 0) {
    rc = launch_preprocess_fwd(*s, *shard, slice_geometry(g, index_base), radii_total + index_base, st, dst, world);
    if (rc) return rc;
  }
  const int pad = slice_len - shard->P;
  for (int r = 0; pad > 0 && r < world; r++) {
    cudaError_t e = cudaMemsetAsync(dst[r] + shard->P, 0, (size_t)pad * sizeof(SplatRecord), st);
    if (e != cudaSuccess) return check_cuda(e, "slice padding");
  }
  return GSR_OK;
}

int gsr_shard_order(const gsr_settings* s, const gsr_tile_owner* owner, int32_t P_total, void* geometry,
                    size_t geometry_bytes, int32_t* radii_total, int32_t* num_rendered_host, void* stream) {
  int rc = check_settings(s);
  if (rc) return rc;
  TileOwner own;
  rc = check_owner(owner, own);
  if (rc) return rc;
  if (P_total <= 0 || !geometry || !radii_total || !num_rendered_host) { set_error("shard_order: bad arguments"); return GSR_ERR_INVALID; }
  cudaStream_t st = (cudaStream_t)stream;
  GeometryWS g;
  if (!carve_geometry(geometry, P_total, g)) return GSR_ERR_CUDA;
  if (g.total > geometry_bytes) { set_error("geometry workspace too small: %zu < %zu", geometry_bytes, g.total); return GSR_ERR_WORKSPACE; }
  StageScope t(ST_DEPTH_SCAN, st);
  rc = launch_retouch(*s, P_total, g, radii_total, own, st);
  if (rc) return rc;
  gsr_cloud c{};
  c.P = P_total;
  const bool v2 = tile_binning_supported((s->image_width + TILE - 1) / TILE, (s->image_height + TILE - 1) / TILE);
  if (v2) {
    if ((rc = launch_tile_count(g, (s->image_width + TILE - 1) / TILE, (s->image_height + TILE - 1) / TILE, own, st))) return rc;
    cudaError_t e = cudaMemcpyAsync(num_rendered_host, g.R_dev, sizeof(int32_t), cudaMemcpyDeviceToHost, st);
    if (e != cudaSuccess) return check_cuda(e, "num_rendered readback");
  }
  return run_depth_order_and_scan(c, g, v2 ? nullptr : num_rendered_host, st, s->debug != 0);
}

int gsr_shard_render(const gsr_settings* s, const gsr_tile_owner* owner, int32_t P_total, int32_t R, void* geometry,
                     size_t geometry_bytes, void* binning, size_t binning_bytes, void* image, size_t image_bytes,
                     const int32_t* radii_total, float* out_color, float* out_depth, void* stream) {
  int rc = check_settings(s);
  if (rc) return rc;
  TileOwner own;
  rc = check_owner(owner, own);
  if (rc) return rc;
  if (P_total <= 0 || R < 0 || !out_color || !out_depth || !radii_total) { set_error("shard_render: bad arguments"); return GSR_ERR_INVALID; }
  cudaStream_t st = (cudaStream_t)stream;
  gsr_cloud c{};
  c.P = P_total;
  GeometryWS g; BinningWS b; ImageWS im;
  rc = carve_all(s, &c, R, geometry, geometry_bytes, binning, binning_bytes, image, image_bytes, g, b, im);
  if (rc) return rc;
  rc = run_binning(*s, c, R, false, g, b, im, radii_total, st, own);
  if (rc) return rc;
  StageScope t(ST_RENDER_FWD, st);
  return launch_render_fwd(*s, g, b, im, out_color, out_depth, st, own);
}

int gsr_shard_backward_render(const gsr_settings* s, const gsr_tile_owner* owner, int32_t P_total, int32_t R,
                              const void* geometry, size_t geometry_bytes, const void* binning, size_t binning_bytes,
                              const void* image, size_t image_bytes, const float* dL_dout_color, void* acc_total,
                              size_t acc_bytes, void* stream) {
  int rc = check_settings(s);
  if (rc) return rc;
  TileOwner own;
  rc = check_owner(owner, own);
  if (rc) return rc;
  if (P_total <= 0 || R < 0 || !dL_dout_color) { set_error("shard_backward_render: bad arguments"); return GSR_ERR_INVALID; }
  const size_t need = (size_t)P_total * ACC_STRIDE * sizeof(float);
  if (!acc_total || acc_bytes < need) { set_error("accumulators too small: %zu < %zu", acc_bytes, need); return GSR_ERR_WORKSPACE; }
  cudaStream_t st = (cudaStream_t)stream;
  gsr_cloud c{};
  c.P = P_total;
  GeometryWS g; BinningWS b; ImageWS im;
  rc = carve_all(s, &c, R, const_cast<void*>(geometry), geometry_bytes, const_cast<void*>(binning), binning_bytes,
                 const_cast<void*>(image), image_bytes, g, b, im);
  if (rc) return rc;
  StageScope t(ST_RENDER_BWD, st);
  cudaError_t e = cudaMemsetAsync(acc_total, 0, need, st);
  if (e != cudaSuccess) return check_cuda(e, "accumulator memset");
  if (R == 0) return GSR_OK;
  return launch_render_bwd(*s, g, b, im, dL_dout_color, (float*)acc_total, st, own);
}

int gsr_shard_backward_preprocess(const gsr_settings* s, const gsr_cloud* shard, int32_t P_total, int32_t index_base,
                                  const void* geometry, size_t geometry_bytes, const int32_t* radii_total,
                                  const void* acc_slice, const gsr_grads* gr, void* stream) {
  int rc = validate_cloud(s, shard);
  if (rc) return rc;
  if (P_total <= 0 || index_base < 0 || (int64_t)index_base + shard->P > P_total) { set_error("shard does not fit P_total"); return GSR_ERR_INVALID; }
  if (shard->P == 0) return GSR_OK;
  if (!gr || !acc_slice || !radii_total) { set_error("grads / accumulators / radii is null"); return GSR_ERR_INVALID; }
  if (!gr->dL_dmeans3D || !gr->dL_dmeans2D || !gr->dL_dcolors || !gr->dL_dopacity || !gr->dL_dcov3D ||
      !gr->dL_dscales || !gr->dL_drotations || (shard->shs && !gr->dL_dsh)) {
    set_error("a gradient output pointer is null");
    return GSR_ERR_INVALID;
  }
  if (reinterpret_cast<uintptr_t>(gr->dL_drotations) & 15) { set_error("dL_drotations must be 16-byte aligned"); return GSR_ERR_INVALID; }
  if (reinterpret_cast<uintptr_t>(acc_slice) & 15) { set_error("acc_slice must be 16-byte aligned"); return GSR_ERR_INVALID; }
  cudaStream_t st = (cudaStream_t)stream;
  GeometryWS g;
  if (!carve_geometry(const_cast<void*>(geometry), P_total, g)) return GSR_ERR_CUDA;
  if (g.total > geometry_bytes) { set_error("geometry workspace too small: %zu < %zu", geometry_bytes, g.total); return GSR_ERR_WORKSPACE; }
  StageScope t(ST_PRE_BWD, st);
  return launch_preprocess_bwd(*s, *shard, slice_geometry(g, index_base), radii_total + index_base,
                               (const float*)acc_slice, *gr, st);
}

int gsr_view_geometry(const void* geometry, int32_t P, gsr_geometry_view* out) {
  GeometryWS g;
  if (!out || !carve_geometry(const_cast<void*>(geometry), P, g)) return GSR_ERR_INVALID;
  out->records = (const float*)g.records; out->tiles_touched = g.tiles_touched; out->clamped = g.clamped;
  out->depth_order = g.depth_order;
  return GSR_OK;
}
int gsr_view_binning(const void* binning, int32_t P, int64_t R, int32_t W, int32_t H, gsr_binning_view* out) {
  BinningWS b;
  if (!out || !carve_binning(const_cast<void*>(binning), P, R, W, H, b)) return GSR_ERR_INVALID;
  out->point_list = b.point_list; out->tile_keys = b.keys_sorted;
  out->tile_key_bytes = ((int64_t)((W + TILE - 1) / TILE) * ((H + TILE - 1) / TILE) < 65536 && g_opt.tile_key_bits == 16) ? 2 : 4;
  return GSR_OK;
}
int gsr_view_image(const void* image, int32_t W, int32_t H, gsr_image_view* out) {
  ImageWS im;
  if (!out) return GSR_ERR_INVALID;
  carve_image(const_cast<void*>(image), W, H, im);
  out->final_T = im.final_T; out->n_contrib = im.n_contrib; out->ranges = (const uint32_t*)im.ranges;
  return GSR_OK;
}

int gsr_set_option(const char* name, int64_t value) {
  if (!name) return GSR_ERR_INVALID;
  if (!strcmp(name, "render_fwd_variant")) g_opt.render_fwd_variant = (int)value;
  else if (!strcmp(name, "render_bwd_variant")) g_opt.render_bwd_variant = (int)value;
  else if (!strcmp(name, "preprocess_variant")) g_opt.preprocess_variant = (int)value;
  else if (!strcmp(name, "profile")) g_opt.profile = (int)value;
  else if (!strcmp(name, "tile_key_bits")) g_opt.tile_key_bits = (int)value;
  else if (!strcmp(name, "binning_variant")) g_opt.binning_variant = (int)value;
  else if (!strcmp(name, "depth_sort_variant")) g_opt.depth_sort_variant = (int)value;
  else if (!strcmp(name, "stats")) {
    if (value && !g_stats_dev) {
      if (cudaMalloc((void**)&g_stats_dev, 16 * sizeof(unsigned long long)) != cudaSuccess) return check_cuda(cudaGetLastError(), "stats alloc");
      cudaMemset(g_stats_dev, 0, 16 * sizeof(unsigned long long));
    } else if (!value && g_stats_dev) {
      cudaFree(g_stats_dev);
      g_stats_dev = nullptr;
    }
  }
  else { set_error("unknown option %s", name); return GSR_ERR_INVALID; }
  return GSR_OK;
}
int64_t gsr_get_option(const char* name) {
  if (!name) return -1;
  if (!strncmp(name, "stat", 4) && name[4] >= '0' && name[4] <= '9') {  // "stat0".."stat9": read + clear a counter
    if (!g_stats_dev) return -1;
    unsigned long long v = 0, z = 0;
    const int i = name[4] - '0';
    cudaDeviceSynchronize();
    cudaMemcpy(&v, g_stats_dev + i, sizeof(v), cudaMemcpyDeviceToHost);
    cudaMemcpy(g_stats_dev + i, &z, sizeof(z), cudaMemcpyHostToDevice);
    return (int64_t)v;
  }
  if (!strcmp(name, "render_fwd_variant")) return g_opt.render_fwd_variant;
  if (!strcmp(name, "render_bwd_variant")) return g_opt.render_bwd_variant;
  if (!strcmp(name, "preprocess_variant")) return g_opt.preprocess_variant;
  if (!strcmp(name, "profile")) return g_opt.profile;
  if (!strcmp(name, "tile_key_bits")) return g_opt.tile_key_bits;
  if (!strcmp(name, "binning_variant")) return g_opt.binning_variant;
  if (!strcmp(name, "depth_sort_variant")) return g_opt.depth_sort_variant;
  return -1;
}
int64_t gsr_launch_count(void) { return g_launches; }

int gsr_profile_read(double* ms_out, int64_t* calls_out) {
  if (!ms_out || !calls_out) return GSR_ERR_INVALID;
  for (int i = 0; i < GSR_NUM_STAGES; i++) { ms_out[i] = 0.0; calls_out[i] = 0; }
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return check_cuda(e, "profile_read");
  std::lock_guard<std::mutex> lk(g_prof_mu);
  for (ProfRec* r : g_prof) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, r->a, r->b) == cudaSuccess && r->stage >= 0 && r->stage < GSR_NUM_STAGES) {
      ms_out[r->stage] += ms;
      calls_out[r->stage]++;
    }
    cudaEventDestroy(r->a);
    cudaEventDestroy(r->b);
    delete r;
  }
  g_prof.clear();
  return GSR_OK;
}

}  // extern "C"

// ---- host-buffer convenience API -----------------------------------------------------------------------
struct gsr_host_ctx {
  int P = 0, M = 0;
  float *means3D = nullptr, *opac = nullptr, *shs = nullptr, *scales = nullptr, *rots = nullptr;
  float* cam = nullptr;  // bg[3] pad, view[16], proj[16], campos[3]: 40 floats
  void *geom = nullptr, *bin = nullptr, *img = nullptr, *scratch = nullptr;
  size_t geom_b = 0, bin_b = 0, img_b = 0, scratch_b = 0;
  int32_t* radii = nullptr;
  float *out_color = nullptr, *out_depth = nullptr, *dL = nullptr;
  size_t img_cap = 0;
  float* grads = nullptr;  // all gradient tensors, contiguous
  size_t grads_cap = 0;
  double* sums = nullptr;
  int32_t* R_pinned = nullptr;
  float* cam_pinned = nullptr;
  cudaStream_t st = nullptr;
};

namespace {
__global__ void checksum_kernel(const float* __restrict__ x, size_t n, double* out) {
  double acc = 0.0;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) acc += x[i];
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(out, acc);
}
template <typename T> int dev_alloc(T** p, size_t n) {
  if (*p) cudaFree(*p);
  *p = nullptr;
  return check_cuda(cudaMalloc((void**)p, n ? n : 1), "cudaMalloc");
}
}  // namespace

extern "C" {

gsr_host_ctx* gsr_host_create(void) {
  gsr_host_ctx* c = new gsr_host_ctx();
  if (cudaStreamCreateWithFlags(&c->st, cudaStreamNonBlocking) != cudaSuccess ||
      cudaMallocHost((void**)&c->R_pinned, sizeof(int32_t)) != cudaSuccess ||
      cudaMallocHost((void**)&c->cam_pinned, 40 * sizeof(float)) != cudaSuccess ||
      cudaMalloc((void**)&c->cam, 40 * sizeof(float)) != cudaSuccess ||
      cudaMalloc((void**)&c->sums, 8 * sizeof(double)) != cudaSuccess) {
    check_cuda(cudaGetLastError(), "gsr_host_create");
    delete c;
    return nullptr;
  }
  return c;
}
void gsr_host_destroy(gsr_host_ctx* c) {
  if (!c) return;
  void* ptrs[] = {c->means3D, c->opac, c->shs, c->scales, c->rots, c->cam, c->geom, c->bin, c->img, c->scratch,
                  c->radii, c->out_color, c->out_depth, c->dL, c->grads, c->sums};
  for (void* p : ptrs) if (p) cudaFree(p);
  if (c->R_pinned) cudaFreeHost(c->R_pinned);
  if (c->cam_pinned) cudaFreeHost(c->cam_pinned);
  if (c->st) cudaStreamDestroy(c->st);
  delete c;
}
int gsr_host_upload_cloud(gsr_host_ctx* c, int32_t P, int32_t M, const float* means3D, const float* opacities,
                          const float* shs, const float* scales, const float* rotations) {
  if (!c || P <= 0 || M <= 0 || !means3D || !opacities || !shs || !scales || !rotations) { set_error("upload_cloud: bad arguments"); return GSR_ERR_INVALID; }
  c->P = P; c->M = M;
  int rc;
  if ((rc = dev_alloc(&c->means3D, (size_t)P * 12))) return rc;
  if ((rc = dev_alloc(&c->opac, (size_t)P * 4))) return rc;
  if ((rc = dev_alloc(&c->shs, (size_t)P * M * 12))) return rc;
  if ((rc = dev_alloc(&c->scales, (size_t)P * 12))) return rc;
  if ((rc = dev_alloc(&c->rots, (size_t)P * 16))) return rc;
  if ((rc = dev_alloc(&c->radii, (size_t)P * 4))) return rc;
  cudaMemcpyAsync(c->means3D, means3D, (size_t)P * 12, cudaMemcpyHostToDevice, c->st);
  cudaMemcpyAsync(c->opac, opacities, (size_t)P * 4, cudaMemcpyHostToDevice, c->st);
  cudaMemcpyAsync(c->shs, shs, (size_t)P * M * 12, cudaMemcpyHostToDevice, c->st);
  cudaMemcpyAsync(c->scales, scales, (size_t)P * 12, cudaMemcpyHostToDevice, c->st);
  cudaMemcpyAsync(c->rots, rotations, (size_t)P * 16, cudaMemcpyHostToDevice, c->st);
  c->geom_b = gsr_geometry_bytes(P);
  if ((rc = dev_alloc((char**)&c->geom, c->geom_b))) return rc;
  c->scratch_b = gsr_backward_scratch_bytes(P);
  if ((rc = dev_alloc((char**)&c->scratch, c->scratch_b))) return rc;
  const size_t gn = (size_t)P * (3 + 3 + 3 + 1 + 6 + 3 * (size_t)M + 3 + 4);
  if ((rc = dev_alloc(&c->grads, gn * 4 + 256))) return rc;
  c->grads_cap = gn;
  return check_cuda(cudaStreamSynchronize(c->st), "upload_cloud");
}

int64_t gsr_host_step(gsr_host_ctx* c, const gsr_settings* sh, const float* dL_host, float* out_color_host,
                      int32_t* out_radii_host, double* sums_host) {
  if (!c || !sh || c->P <= 0) { set_error("host_step: no cloud uploaded"); return GSR_ERR_INVALID; }
  const int W = sh->image_width, H = sh->image_height, P = c->P, M = c->M;
  const size_t npix = (size_t)W * H;
  int rc;
  if (npix > c->img_cap) {
    if ((rc = dev_alloc(&c->out_color, npix * 12))) return rc;
    if ((rc = dev_alloc(&c->out_depth, npix * 4))) return rc;
    if ((rc = dev_alloc(&c->dL, npix * 12))) return rc;
    c->img_b = gsr_image_bytes(W, H);
    if ((rc = dev_alloc((char**)&c->img, c->img_b))) return rc;
    c->img_cap = npix;
  }
  // camera: host -> pinned -> device
  memcpy(c->cam_pinned, sh->bg, 12);
  memcpy(c->cam_pinned + 4, sh->viewmatrix, 64);
  memcpy(c->cam_pinned + 20, sh->projmatrix, 64);
  memcpy(c->cam_pinned + 36, sh->campos, 12);
  cudaMemcpyAsync(c->cam, c->cam_pinned, 160, cudaMemcpyHostToDevice, c->st);
  gsr_settings s = *sh;
  s.bg = c->cam; s.viewmatrix = c->cam + 4; s.projmatrix = c->cam + 20; s.campos = c->cam + 36;
  s.sh_coeffs = M;
  gsr_cloud cl;
  cl.P = P; cl.means3D = c->means3D; cl.opacities = c->opac; cl.shs = c->shs; cl.colors_precomp = nullptr;
  cl.scales = c->scales; cl.rotations = c->rots; cl.cov3D_precomp = nullptr;
  if (dL_host) cudaMemcpyAsync(c->dL, dL_host, npix * 12, cudaMemcpyHostToDevice, c->st);
  rc = gsr_forward_preprocess(&s, &cl, c->geom, c->geom_b, c->radii, c->R_pinned, c->st);
  if (rc) return rc;
  if ((rc = check_cuda(cudaStreamSynchronize(c->st), "host_step sync"))) return rc;
  const int R = *c->R_pinned;
  const size_t need = gsr_binning_bytes(P, R, W, H);
  if (need > c->bin_b) {
    c->bin_b = need + need / 4;
    if ((rc = dev_alloc((char**)&c->bin, c->bin_b))) return rc;
  }
  rc = gsr_forward_render(&s, &cl, R, c->geom, c->geom_b, c->bin, c->bin_b, c->img, c->img_b, c->radii, c->out_color,
                          c->out_depth, c->st);
  if (rc) return rc;
  if (out_color_host) cudaMemcpyAsync(out_color_host, c->out_color, npix * 12, cudaMemcpyDeviceToHost, c->st);
  if (out_radii_host) cudaMemcpyAsync(out_radii_host, c->radii, (size_t)P * 4, cudaMemcpyDeviceToHost, c->st);
  if (dL_host) {
    float* p = c->grads;
    gsr_grads gr;
    gr.dL_drotations = p; p += (size_t)P * 4;  // first: keeps 16-byte alignment
    gr.dL_dsh = p; p += (size_t)P * M * 3;
    gr.dL_dmeans3D = p; p += (size_t)P * 3;
    gr.dL_dmeans2D = p; p += (size_t)P * 3;
    gr.dL_dcolors = p; p += (size_t)P * 3;
    gr.dL_dopacity = p; p += (size_t)P;
    gr.dL_dcov3D = p; p += (size_t)P * 6;
    gr.dL_dscales = p; p += (size_t)P * 3;
    rc = gsr_backward(&s, &cl, R, c->geom, c->geom_b, c->bin, c->bin_b, c->img, c->img_b, c->radii, c->dL, c->scratch,
                      c->scratch_b, &gr, c->st);
    if (rc) return rc;
    if (sums_host) {
      cudaMemsetAsync(c->sums, 0, 8 * sizeof(double), c->st);
      const float* ptrs[8] = {gr.dL_dmeans3D, gr.dL_dmeans2D, gr.dL_dcolors, gr.dL_dopacity,
                              gr.dL_dcov3D, gr.dL_dsh, gr.dL_dscales, gr.dL_drotations};
      const size_t ns[8] = {(size_t)P * 3, (size_t)P * 3, (size_t)P * 3, (size_t)P, (size_t)P * 6, (size_t)P * M * 3, (size_t)P * 3, (size_t)P * 4};
      for (int i = 0; i < 8; i++) {
        checksum_kernel<<<296, 256, 0, c->st>>>(ptrs[i], ns[i], c->sums + i);
        g_launches++;
      }
      cudaMemcpyAsync(sums_host, c->sums, 8 * sizeof(double), cudaMemcpyDeviceToHost, c->st);
    }
  }
  if ((rc = check_cuda(cudaStreamSynchronize(c->st), "host_step end"))) return rc;
  return R;
}

}  // extern "C"
