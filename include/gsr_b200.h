/* gsr_b200.h -- C ABI of the B200-native (sm_100a) differentiable 3D-Gaussian-splatting rasterizer.
 *
 * This is the drop-in boundary for the ONE hot path of buaacyw/GaussianEditor this repo rebuilds:
 * the `diff_gaussian_rasterization._C` extension behind gaussiansplatting/gaussian_renderer.render().
 * Every entry point replaces one binding of the reference's private pybind module
 * (all paths relative to /root/reference/gaussiansplatting/submodules/diff-gaussian-rasterization/):
 *
 *   gsr_forward_preprocess + gsr_forward_render   <- _C.rasterize_gaussians          ext.cpp:16, rasterize_points.cu:35-95,
 *                                                                                     cuda_rasterizer/rasterizer_impl.cu:179-285
 *   gsr_backward                                  <- _C.rasterize_gaussians_backward ext.cpp:17, rasterize_points.cu:97-157,
 *                                                                                     cuda_rasterizer/rasterizer_impl.cu:289-341
 *   gsr_mark_visible                              <- _C.mark_visible                 ext.cpp:18, rasterize_points.cu:159-175
 *   gsr_apply_weights                             <- _C.apply_weights                ext.cpp:19, rasterize_points.cu:177-234
 *
 * Conventions
 *   - plain C: pointers + sizes, no torch / C++ types.  Unless a parameter says "host", every pointer is a
 *     DEVICE pointer on the current CUDA device; the caller (PyTorch's caching allocator in the Python
 *     binding, cudaMalloc in a C host) owns all memory.  "Optional" pointers may be NULL; the reference
 *     encodes the same thing as empty tensors (rasterizer_impl.cu:205,241,275).
 *   - every call takes the cudaStream_t to run on (as void*); the reference always ran on the legacy
 *     default stream and blocked on a cudaMemcpy (rasterizer_impl.cu:237) -- here the only host
 *     synchronisation is the caller waiting for `num_rendered` between the two forward halves.
 *   - return value: 0 = ok, <0 = error (see gsr_last_error()).  There is NO CPU fallback: without a usable
 *     sm_100 device every compute entry point fails with GSR_ERR_CUDA.
 *   - all floating-point data is IEEE binary32, exactly as in the reference.
 */
#ifndef GSR_B200_H_
#define GSR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSR_OK 0
#define GSR_ERR_INVALID (-1) /* bad argument combination (mirrors the reference's Python/C++ argument checks) */
#define GSR_ERR_CUDA (-2)    /* CUDA runtime error; message in gsr_last_error() */
#define GSR_ERR_WORKSPACE (-3) /* a workspace is smaller than the matching gsr_*_bytes() query */

#define GSR_ABI_VERSION 2

#if defined(__GNUC__)
#define GSR_API __attribute__((visibility("default")))
#else
#define GSR_API
#endif

/* Per-call camera / configuration bundle: the fields of GaussianRasterizationSettings
 * (diff_gaussian_rasterization/__init__.py:228-240) plus the two SH sizes the glue derives
 * (rasterize_points.cu:73-76). */
typedef struct gsr_settings {
  int32_t image_height;
  int32_t image_width;
  float tanfovx;
  float tanfovy;
  float scale_modifier;
  int32_t sh_degree;   /* D: active degree, 0..3 */
  int32_t sh_coeffs;   /* M: coefficients ALLOCATED per Gaussian in `shs` (0 when colors_precomp is used) */
  int32_t prefiltered; /* kept for API parity; a culled point with prefiltered!=0 is simply skipped */
  int32_t debug;       /* !=0: synchronise and check for CUDA errors after every launch (auxiliary.h:166-173) */
  const float* bg;         /* [3]  */
  const float* viewmatrix; /* [16] transposed world->camera (scene/cameras.py:92)  */
  const float* projmatrix; /* [16] transposed full projection (scene/cameras.py:93-94) */
  const float* campos;     /* [3]  */
} gsr_settings;

/* The Gaussian cloud as the reference's forward takes it (diff_gaussian_rasterization/__init__.py:258-268).
 * Exactly one of {shs, colors_precomp} and exactly one of {(scales, rotations), cov3D_precomp} is non-NULL. */
typedef struct gsr_cloud {
  int32_t P;                   /* number of Gaussians */
  const float* means3D;        /* [P,3] */
  const float* opacities;      /* [P,1] already sigmoid-ed */
  const float* shs;            /* [P,M,3] optional */
  const float* colors_precomp; /* [P,3]   optional */
  const float* scales;         /* [P,3]   optional, already exp-ed */
  const float* rotations;      /* [P,4]   optional, (r,x,y,z), normalised by the caller */
  const float* cov3D_precomp;  /* [P,6]   optional */
} gsr_cloud;

/* Gradient outputs of the backward pass, shapes as rasterize_points.cu:120-128. The kernels write EVERY
 * element (zeros for invisible Gaussians and for SH coefficients above the active degree), so the
 * buffers may be uninitialised on entry. */
typedef struct gsr_grads {
  float* dL_dmeans3D;   /* [P,3] */
  float* dL_dmeans2D;   /* [P,3] (z is always 0; x,y carry the 0.5*W / 0.5*H NDC scaling, backward.cu:460-461) */
  float* dL_dcolors;    /* [P,3] */
  float* dL_dopacity;   /* [P,1] */
  float* dL_dcov3D;     /* [P,6] */
  float* dL_dsh;        /* [P,M,3] (NULL when M == 0) */
  float* dL_dscales;    /* [P,3] */
  float* dL_drotations; /* [P,4] */
} gsr_grads;

GSR_API int gsr_abi_version(void);
GSR_API const char* gsr_last_error(void); /* thread-local, valid until the next failing call on this thread */
/* Threading: every entry point only touches the buffers it is handed and enqueues on the stream it is handed, so calls
 * from several host threads are safe as long as they do not share a workspace. The library-global pieces are the option
 * table (gsr_set_option: set before the threads start), the launch counter (atomic) and the stage profile (mutex). */

/* ---- workspace sizing (the three opaque buffers of rasterize_points.cu:62-69) ------------------------ */
GSR_API size_t gsr_geometry_bytes(int32_t P);
GSR_API size_t gsr_image_bytes(int32_t image_width, int32_t image_height);
GSR_API size_t gsr_binning_bytes(int32_t P, int64_t num_rendered, int32_t image_width, int32_t image_height);
/* scratch for the backward pass (2-D gradient accumulators) */
GSR_API size_t gsr_backward_scratch_bytes(int32_t P);

/* ---- forward, first half: per-Gaussian preprocess + depth order + tile-count scan --------------------
 * Writes `radii` [P] int32 (0 = culled) and fills `geometry`. The total number of (Gaussian, tile)
 * instances is copied asynchronously into *num_rendered_host (PINNED host memory, int32); the caller must
 * synchronise `stream` (or an event recorded after this call) before reading it. */
GSR_API int gsr_forward_preprocess(const gsr_settings* s, const gsr_cloud* c, void* geometry, size_t geometry_bytes,
                           int32_t* radii, int32_t* num_rendered_host, void* stream);

/* ---- forward, second half: instance emission, per-tile ordering, tile ranges, alpha blending ----------
 * out_color [3,H,W], out_depth [1,H,W] (depth = sum view_z*alpha*T, no background, forward.cu:359,377). */
GSR_API int gsr_forward_render(const gsr_settings* s, const gsr_cloud* c, int32_t num_rendered, void* geometry,
                       size_t geometry_bytes, void* binning, size_t binning_bytes, void* image, size_t image_bytes,
                       const int32_t* radii, float* out_color, float* out_depth, void* stream);

/* ---- forward, second half, without waiting for num_rendered ------------------------------------------------
 * Same as gsr_forward_render, but launched BEFORE the host knows num_rendered: `capacity` is the caller's guess
 * (e.g. 1.25x the previous frame's value) and sizes the binning workspace and the launches; the real count is read
 * from the scan result on the device and the slots [num_rendered, capacity) are padding that sorts behind every
 * tile. The caller must afterwards read *num_rendered_host (after the stream reaches the copy issued by
 * gsr_forward_preprocess) and, if it exceeds `capacity`, discard the outputs and call gsr_forward_render with the
 * exact count. gsr_backward then takes `capacity` as its num_rendered argument (it only sizes the workspace).
 * This keeps the GPU busy while the host waits for the count (the reference blocks in cudaMemcpy with an idle
 * GPU, rasterizer_impl.cu:237). */
GSR_API int gsr_forward_render_speculative(const gsr_settings* s, const gsr_cloud* c, int32_t capacity, void* geometry,
                       size_t geometry_bytes, void* binning, size_t binning_bytes, void* image, size_t image_bytes,
                       const int32_t* radii, float* out_color, float* out_depth, void* stream);

/* ---- backward ------------------------------------------------------------------------------------------
 * dL_dout_color [3,H,W]; the three workspaces and `radii` are the ones the forward produced. */
GSR_API int gsr_backward(const gsr_settings* s, const gsr_cloud* c, int32_t num_rendered, const void* geometry,
                 size_t geometry_bytes, const void* binning, size_t binning_bytes, const void* image,
                 size_t image_bytes, const int32_t* radii, const float* dL_dout_color, void* scratch,
                 size_t scratch_bytes, const gsr_grads* grads, void* stream);

/* ---- alpha image (north-star output "RGB / depth / alpha"; opt-in, not in the reference's return tuple) ----
 * out_alpha [H*W] = 1 - final_T, where final_T is what the reference keeps as ImageState::accum_alpha
 * (cuda_rasterizer/rasterizer_impl.h:50, written at forward.cu:371-378). Call after gsr_forward_render on the same
 * `image` workspace. gsr_backward_alpha is gsr_backward with the additional upstream gradient dL_dout_alpha [H*W]
 * (NULL = none): d(1 - T_final)/d(alpha_i) = T_final / (1 - alpha_i) enters dL/dalpha_i next to the background term
 * of backward.cu:505-511. */
GSR_API int gsr_alpha_image(const void* image, size_t image_bytes, int32_t image_width, int32_t image_height,
                    float* out_alpha, void* stream);
GSR_API int gsr_backward_alpha(const gsr_settings* s, const gsr_cloud* c, int32_t num_rendered, const void* geometry,
                       size_t geometry_bytes, const void* binning, size_t binning_bytes, const void* image,
                       size_t image_bytes, const int32_t* radii, const float* dL_dout_color,
                       const float* dL_dout_alpha, void* scratch, size_t scratch_bytes, const gsr_grads* grads,
                       void* stream);

/* ---- camera gradients (north star: backward over {..., viewmatrix}; opt-in, the reference has none) -------------
 * The reference's autograd returns None for the raster settings (diff_gaussian_rasterization/__init__.py:213-223), so
 * there is nothing to be drop-in for; this entry point extends gsr_backward_alpha with
 *   dL/dviewmatrix [16], dL/dprojmatrix [16], dL/dcampos [3]
 * for the three camera arrays of gsr_settings treated as INDEPENDENT inputs, exactly as the forward reads them (the
 * view matrix through t = view*mean and the rotation W of the EWA Jacobian product, cuda_rasterizer/forward.cu:74-113;
 * the full projection through p_hom, :196-200; the camera centre through the SH view direction, :20-71). The same
 * conventions as the mean gradient apply (clamped t.x / t.y pass no gradient, backward.cu:205-212). A caller that
 * derives projmatrix and campos from the view matrix (scene/cameras.py:92-95) chains the three in its own autograd.
 * Checked against central finite differences of the fp64 CPU oracle (tests/test_parity_gpu.py). */
typedef struct gsr_camera_grads {
  float* dL_dviewmatrix; /* [16] same layout as gsr_settings.viewmatrix; entries the forward never reads stay 0 */
  float* dL_dprojmatrix; /* [16] */
  float* dL_dcampos;     /* [3]  */
  void* scratch;         /* gsr_camera_scratch_bytes(P) bytes of device memory */
  size_t scratch_bytes;
} gsr_camera_grads;
GSR_API size_t gsr_camera_scratch_bytes(int32_t P);
GSR_API int gsr_backward_camera(const gsr_settings* s, const gsr_cloud* c, int32_t num_rendered, const void* geometry,
                        size_t geometry_bytes, const void* binning, size_t binning_bytes, const void* image,
                        size_t image_bytes, const int32_t* radii, const float* dL_dout_color,
                        const float* dL_dout_alpha /* may be NULL */, void* scratch, size_t scratch_bytes,
                        const gsr_grads* grads, const gsr_camera_grads* camera, void* stream);

/* ---- depth gradients (opt-in; the reference's backward ignores the gradient of its depth output) -----------------
 * The forward's depth image D = sum_i d_i*alpha_i*T_i (d_i = view-space z of Gaussian i, no background term) is blended
 * exactly like a colour channel. gsr_backward_depth is gsr_backward_camera with the additional upstream gradient
 * dL_dout_depth [H*W] (REQUIRED: NULL is GSR_ERR_INVALID; pass zeros for "none") and with dL_dout_alpha and camera both
 * optional (NULL = no alpha gradient / no camera gradients), so it covers every combination of the three extras. It adds
 *   dL/dalpha_i += T_i * (d_i - depth blended behind i) * dL/dD   (-> mean2D, conic, opacity, and so on down the chain)
 *   dL/dmean3D_i += (sum over pixels of alpha_i*T_i*dL/dD) * (view[2], view[6], view[10])
 * and, with camera gradients, dL/dview[2 + 4r] += that sum * mean_r, dL/dview[14] += that sum. d_i is the unclamped
 * view depth, so no clamp applies; projmatrix and campos receive nothing from the depth image.
 * gsr_backward_raw_depth is gsr_backward_raw with the same additional dL_dout_depth. */
GSR_API int gsr_backward_depth(const gsr_settings* s, const gsr_cloud* c, int32_t num_rendered, const void* geometry,
                       size_t geometry_bytes, const void* binning, size_t binning_bytes, const void* image,
                       size_t image_bytes, const int32_t* radii, const float* dL_dout_color,
                       const float* dL_dout_alpha /* may be NULL */, const float* dL_dout_depth /* [H*W] */,
                       void* scratch, size_t scratch_bytes, const gsr_grads* grads,
                       const gsr_camera_grads* camera /* may be NULL */, void* stream);

/* ---- markVisible: present[i] = view-space z > 0.2 (auxiliary.h:139-164) ------------------------------- */
GSR_API int gsr_mark_visible(int32_t P, const float* means3D, const float* viewmatrix, const float* projmatrix,
                     uint8_t* present, void* stream);

/* ---- apply_weights (semantic tracing, cuda_rasterizer/apply_weights.cu:240-356) ------------------------
 * Second half of a forward whose colours are ignored: for every (pixel, splat) pair the forward would blend,
 * weights[id*CH+ch] += image_weights[ch,pixel] and cnt[id] += 1 once per channel. Call
 * gsr_forward_preprocess first (with colors_precomp = weights, as the reference does,
 * rasterize_points.cu:223). CH = 1..3. */
GSR_API int gsr_apply_weights(const gsr_settings* s, const gsr_cloud* c, int32_t num_rendered, void* geometry,
                      size_t geometry_bytes, void* binning, size_t binning_bytes, void* image, size_t image_bytes,
                      const int32_t* radii, const float* image_weights, int32_t num_channels, float* weights,
                      int32_t* cnt, void* stream);

/* ---- introspection for parity tests: device pointers into the opaque workspaces ----------------------- */
typedef struct gsr_geometry_view {
  const float* records;          /* [P,12]: x,y,conicA,conicB | conicC,opacity,depth,_ | r,g,b,_  (visible only) */
  const uint32_t* tiles_touched; /* [P] */
  const uint8_t* clamped;        /* [P] bit ch set = SH colour channel ch was clamped at 0 */
  const uint32_t* depth_order;   /* [P] Gaussian indices ascending in (depth bits, index); culled ones last */
} gsr_geometry_view;
typedef struct gsr_binning_view {
  const uint32_t* point_list; /* [R] == the reference's sorted point_list (rasterizer_impl.cu:256-261) */
  const void* tile_keys;      /* [R] sorted tile id of each instance, uint16 or uint32 (tile_key_bytes) */
  int32_t tile_key_bytes;
} gsr_binning_view;
typedef struct gsr_image_view {
  const float* final_T;       /* [H*W] */
  const uint32_t* n_contrib;  /* [H*W] */
  const uint32_t* ranges;     /* [Ntile,2] */
} gsr_image_view;
GSR_API int gsr_view_geometry(const void* geometry, int32_t P, gsr_geometry_view* out);
GSR_API int gsr_view_binning(const void* binning, int32_t P, int64_t num_rendered, int32_t image_width,
                     int32_t image_height, gsr_binning_view* out);
GSR_API int gsr_view_image(const void* image, int32_t image_width, int32_t image_height, gsr_image_view* out);

/* ---- fused activations (SURVEY.md 8(f-3)) -----------------------------------------------------------------------
 * Opt-in variant that takes the scene model's RAW parameters and applies the activations of
 * scene/gaussian_model.py:221-258 inside the preprocess kernels instead of in PyTorch before every render:
 *   opacity = sigmoid(logit), scale = exp(log_scale), rotation = raw / max(|raw|, 1e-12),
 *   SH row  = [features_dc | features_rest]   (read from the two arrays; no torch.cat, no [P,M,3] copy).
 * gsr_forward_preprocess_raw replaces gsr_forward_preprocess; the second forward half is the ordinary
 * gsr_forward_render (pass a gsr_cloud with P and any non-null pointers); gsr_backward_raw replaces gsr_backward and
 * returns gradients w.r.t. the raw parameters (chain rule through the activations included). settings.sh_coeffs is
 * M = 1 + K, the coefficients allocated over both arrays. Results agree with the PyTorch-activated path to rounding
 * (not bit-for-bit: torch's normalize reduces in a different order); the default entry points keep exact parity. */
typedef struct gsr_raw_cloud {
  int32_t P;
  const float* means3D;        /* [P,3] */
  const float* opacity_logits; /* [P,1] */
  const float* features_dc;    /* [P,1,3] */
  const float* features_rest;  /* [P,K,3], K = sh_coeffs - 1 (NULL when K == 0) */
  const float* log_scales;     /* [P,3] */
  const float* raw_rotations;  /* [P,4], 16-byte aligned */
} gsr_raw_cloud;
typedef struct gsr_raw_grads {
  float* dL_dmeans3D;        /* [P,3] */
  float* dL_dmeans2D;        /* [P,3] */
  float* dL_dopacity_logits; /* [P,1] */
  float* dL_dfeatures_dc;    /* [P,1,3] */
  float* dL_dfeatures_rest;  /* [P,K,3] (NULL when K == 0) */
  float* dL_dlog_scales;     /* [P,3] */
  float* dL_draw_rotations;  /* [P,4], 16-byte aligned */
} gsr_raw_grads;
GSR_API int gsr_forward_preprocess_raw(const gsr_settings* s, const gsr_raw_cloud* c, void* geometry,
                               size_t geometry_bytes, int32_t* radii, int32_t* num_rendered_host, void* stream);
GSR_API int gsr_backward_raw(const gsr_settings* s, const gsr_raw_cloud* c, int32_t num_rendered, const void* geometry,
                     size_t geometry_bytes, const void* binning, size_t binning_bytes, const void* image,
                     size_t image_bytes, const int32_t* radii, const float* dL_dout_color, void* scratch,
                     size_t scratch_bytes, const gsr_raw_grads* grads, void* stream);
/* gsr_backward_raw plus the gradient of the depth image, dL_dout_depth [H*W] (required; see gsr_backward_depth) */
GSR_API int gsr_backward_raw_depth(const gsr_settings* s, const gsr_raw_cloud* c, int32_t num_rendered,
                           const void* geometry, size_t geometry_bytes, const void* binning, size_t binning_bytes,
                           const void* image, size_t image_bytes, const int32_t* radii, const float* dL_dout_color,
                           const float* dL_dout_depth, void* scratch, size_t scratch_bytes, const gsr_raw_grads* grads,
                           void* stream);

/* ---- Gaussian-sharded multi-GPU path (BASELINE config 4; SURVEY.md 8(e)) ----------------------------------
 * The reference has no multi-GPU rasterizer; these entry points split the single-GPU pipeline at the two places
 * where the Gaussian-index decomposition (preprocess, fused preprocess backward) meets the tile decomposition
 * (binning, blending), so that a host can put one collective in each gap:
 *
 *   rank g owns Gaussians [index_base, index_base + shard.P) of P_total and the tile rows ty % row_stride == row_phase.
 *   forward : gsr_shard_preprocess  -> ALL-GATHER of the 48-byte splat records (gsr_view_exchange gives the array;
 *                                      a record carries its radius and depth key, so it is the whole exchange)
 *             gsr_shard_order       -> radii of all Gaussians, owned-tile counts, depth order, scan, num_rendered
 *                                      (this rank's instances)
 *             gsr_shard_render      -> binning + blending of the owned tiles into zero-initialised full frames
 *                                      -> ALL-REDUCE(sum) of the frames (every pixel has exactly one non-zero
 *                                         contributor, so the sum is a bit-exact concatenation)
 *   backward: gsr_shard_backward_render     -> partial 2-D gradient accumulators [P_total, 12]
 *                                              -> REDUCE-SCATTER(sum) to the index owners
 *             gsr_shard_backward_preprocess -> gradients of this rank's Gaussians
 * All P_total-sized arrays (geometry workspace, radii, accumulators) are indexed by GLOBAL Gaussian index, so
 * the gathered state is exactly the single-GPU state and the images are bit-identical to gsr_forward_render's.
 * Every rank must pass the same P_total and slice_len (= ceil(P_total / world)); slots of a slice beyond
 * shard.P are marked culled. */
typedef struct gsr_tile_owner {
  int32_t row_stride; /* >= 1 */
  int32_t row_phase;  /* 0 .. row_stride-1 */
} gsr_tile_owner;
typedef struct gsr_exchange_view {
  void* records; /* [P_total] 48-byte splat records; rank g writes [g*slice_len, (g+1)*slice_len) */
} gsr_exchange_view;
GSR_API int gsr_view_exchange(void* geometry, int32_t P_total, gsr_exchange_view* out);
GSR_API int gsr_shard_preprocess(const gsr_settings* s, const gsr_cloud* shard, int32_t P_total, int32_t index_base,
                         int32_t slice_len, void* geometry, size_t geometry_bytes, int32_t* radii_total, void* stream);
/* radii_total [P_total] is (re)written here for ALL Gaussians from the gathered records. */
GSR_API int gsr_shard_order(const gsr_settings* s, const gsr_tile_owner* owner, int32_t P_total, void* geometry,
                    size_t geometry_bytes, int32_t* radii_total, int32_t* num_rendered_host, void* stream);
GSR_API int gsr_shard_render(const gsr_settings* s, const gsr_tile_owner* owner, int32_t P_total, int32_t num_rendered,
                     void* geometry, size_t geometry_bytes, void* binning, size_t binning_bytes, void* image,
                     size_t image_bytes, const int32_t* radii_total, float* out_color, float* out_depth, void* stream);
GSR_API int gsr_shard_backward_render(const gsr_settings* s, const gsr_tile_owner* owner, int32_t P_total,
                              int32_t num_rendered, const void* geometry, size_t geometry_bytes, const void* binning,
                              size_t binning_bytes, const void* image, size_t image_bytes, const float* dL_dout_color,
                              void* acc_total, size_t acc_bytes, void* stream);
/* acc_slice: this rank's [shard.P, 12] rows of the reduced accumulators (gsr_backward_scratch_bytes(shard.P)). */
GSR_API int gsr_shard_backward_preprocess(const gsr_settings* s, const gsr_cloud* shard, int32_t P_total,
                                  int32_t index_base, const void* geometry, size_t geometry_bytes,
                                  const int32_t* radii_total, const void* acc_slice, const gsr_grads* grads,
                                  void* stream);

/* ---- fused preprocess + all-gather over NVLink peer memory ---------------------------------------------------
 * Instead of gsr_shard_preprocess followed by an all-gather, every rank's preprocess kernel pushes its block of
 * records into the geometry workspace of EVERY rank (TMA bulk stores from shared memory to peer-mapped global
 * memory). The workspaces must come from gsr_peer_alloc and be opened on the other ranks with gsr_peer_open:
 * peer_geometry[r] is rank r's workspace as mapped in THIS process (own entry = the local pointer), all of the same
 * size and therefore the same layout. The caller must run a cross-rank barrier on `stream` (e.g. a 4-byte
 * all-reduce) between this call and gsr_shard_order, and between a rank's last read of a workspace and the next
 * gsr_shard_preprocess_p2p that targets it (any collective of the step does). */
#define GSR_MAX_PEERS 8
#define GSR_PEER_HANDLE_BYTES 64
GSR_API int gsr_peer_alloc(size_t bytes, void** ptr_out, void* handle_out /* [GSR_PEER_HANDLE_BYTES] host */);
GSR_API int gsr_peer_open(const void* handle /* [GSR_PEER_HANDLE_BYTES] host */, void** ptr_out);
GSR_API int gsr_peer_close(void* ptr);
GSR_API int gsr_peer_free(void* ptr);
GSR_API int gsr_shard_preprocess_p2p(const gsr_settings* s, const gsr_cloud* shard, int32_t P_total, int32_t index_base,
                             int32_t slice_len, void* const* peer_geometry /* [world] host array */, int32_t world,
                             int32_t rank, size_t geometry_bytes, int32_t* radii_total, void* stream);

/* ---- sparse exchange for the Gaussian-sharded path -------------------------------------------------------------
 * The dense scheme above moves, sorts and reduces P_total-sized arrays on every rank. Here a splat record travels only
 * to the ranks whose tile rows (ty % world == d) its tile rectangle touches, into slot  rank*seg_cap + j  of that
 * rank's CANDIDATE array, where j is the record's position among this rank's Gaussians bound for d, in index order.
 * The candidate array (world segments of capacity seg_cap; unused slots are holes with the "culled" sort key) is in
 * global-index order, so the existing stable depth sort / scan / binning / blending stages run on it unchanged as a
 * cloud of world*seg_cap Gaussians (gsr_shard_render / gsr_shard_backward_render with P_total = world*seg_cap and the
 * candidate workspace as `geometry`) and produce the single-GPU lists of the owned tiles bit for bit. The backward
 * returns each candidate's 12-float accumulator row to slot  d*seg_cap + j  of the OWNER's `ret` array, where the
 * owner adds the <= world partial rows of each Gaussian in ascending rank order (deterministic).
 *
 *   forward : gsr_sparse_preprocess   preprocess + destination masks + ordered slots + peer stores of the records;
 *                                     writes counts_row[d] = n[rank -> d]
 *             -- host: all-reduce(sum) of the [world, GSR_MAX_PEERS] count matrix (row = source, written by its rank). It is also the barrier that
 *                orders the peer stores before the readers. --
 *             gsr_sparse_order        candidates -> radii / owned-tile counts / depth order / scan; host_out[0] =
 *                                     num_rendered of this rank, host_out[1] = max over the matrix (a value > seg_cap
 *                                     means some segment overflowed on some rank: redo the step with a larger seg_cap)
 *             gsr_shard_render        (existing)   -> gsr_frame_broadcast or an all-reduce of the frames
 *   backward: gsr_shard_backward_render (existing) -> gsr_sparse_return (peer stores) -- barrier --
 *             gsr_sparse_backward_preprocess       gather of the returned rows + fused preprocess backward
 * peer_cand[r] is rank r's candidate workspace (gsr_sparse_candidate_bytes, from gsr_peer_alloc / gsr_peer_open) as
 * mapped in this process; with virtual ranks on one device they are simply different buffers. */
typedef struct gsr_sparse_plan {
  int32_t world, rank;
  int32_t slice_len; /* ceil(P_total / world): Gaussians per rank (the last rank may hold fewer) */
  int32_t seg_cap;   /* capacity of one (source -> destination) segment; the same on every rank */
} gsr_sparse_plan;
typedef struct gsr_sparse_view_t {
  void* records;         /* [world*seg_cap] 48-byte candidate records */
  float* ret;            /* [world*seg_cap, 12] accumulator rows returned by the tile owners */
  size_t geometry_bytes; /* size of the leading part that is laid out like gsr_geometry_bytes(world*seg_cap) */
} gsr_sparse_view_t;
GSR_API size_t gsr_sparse_local_bytes(int32_t slice_len);
GSR_API size_t gsr_sparse_candidate_bytes(int32_t world, int32_t seg_cap);
GSR_API int gsr_sparse_view(void* cand_ws, int32_t world, int32_t seg_cap, gsr_sparse_view_t* out);
GSR_API int gsr_sparse_preprocess(const gsr_settings* s, const gsr_cloud* shard, const gsr_sparse_plan* plan, void* local_ws,
                          size_t local_bytes, int32_t* radii_local /* [shard.P] */, void* const* peer_cand /* [world] host */,
                          size_t cand_bytes, int32_t* counts_row /* [GSR_MAX_PEERS] device */, void* stream);
GSR_API int gsr_sparse_order(const gsr_settings* s, const gsr_sparse_plan* plan, void* cand_ws, size_t cand_bytes,
                     const int32_t* counts_matrix /* [world, GSR_MAX_PEERS] device, row = source */,
                     int32_t* radii_cand /* [world*seg_cap] */, int32_t* host_out /* [2] pinned host */, void* stream);
GSR_API int gsr_sparse_return(const gsr_sparse_plan* plan, const void* acc_cand /* [world*seg_cap, 12] */,
                      const int32_t* counts_matrix, void* const* peer_cand, void* stream);
GSR_API int gsr_sparse_backward_preprocess(const gsr_settings* s, const gsr_cloud* shard, const gsr_sparse_plan* plan,
                                   const void* local_ws, size_t local_bytes, const int32_t* radii_local,
                                   const void* cand_ws, size_t cand_bytes, void* acc_slice /* [shard.P,12] scratch */,
                                   size_t acc_bytes, const gsr_grads* grads, void* stream);
/* Cross-rank barrier over peer memory (replaces the 4-byte NCCL all-reduces of the dense scheme: ~5 us instead of
 * ~25 us at 8 GPUs). Every rank's peer-visible block starts with GSR_PEER_CTRL_BYTES of control words, zeroed once at
 * creation: flags[rank] = number of the last barrier that rank reached, and the [GSR_MAX_PEERS, GSR_MAX_PEERS] int32
 * count matrix at byte GSR_PEER_CTRL_MATRIX_OFFSET (row s = n[s -> d], written by rank s: gsr_sparse_preprocess takes
 * counts_row = own row of the OWN block). peer_ctrl[r] is rank r's block as mapped here. `epoch` must increase by one per
 * barrier on this block, identically on every rank. with_matrix_row != 0 first copies this rank's row into every
 * peer's matrix, so that after the barrier every rank holds the complete matrix. Work queued on `stream` behind this
 * call starts only after every rank has reached the same barrier (a rank that never arrives costs ~2 s and sets the
 * int32 error word at byte GSR_PEER_CTRL_ERROR_OFFSET of the OWN block to 1 instead of hanging the GPU; the word is
 * sticky -- the host binding copies it out once per step and raises, gaussianeditor_b200/sparse_sharded.py). */
#define GSR_PEER_CTRL_BYTES 512
#define GSR_PEER_CTRL_ERROR_OFFSET 32
#define GSR_PEER_CTRL_MATRIX_OFFSET 64
GSR_API int gsr_peer_barrier(int32_t world, int32_t rank, void* const* peer_ctrl /* [world] host */, uint32_t epoch,
                     int32_t with_matrix_row, void* stream);
/* Copies the tile rows this rank owns of its [4,H,W] frame (colour + depth) into the frames of all other ranks
 * (128-bit peer stores): with one writer per pixel this replaces the all-reduce of the frames. A cross-rank barrier
 * must follow before the frames are read. */
GSR_API int gsr_frame_broadcast(const gsr_tile_owner* owner, int32_t image_width, int32_t image_height, const float* frame,
                        void* const* peer_frames /* [world] host */, void* stream);

/* ---- tuning / instrumentation ---------------------------------------------------------------------------
 * gsr_set_option("render_variant", v) etc.; unknown names return GSR_ERR_INVALID.
 * gsr_launch_count(): number of this library's kernel launches (CUB's included) since process start. */
GSR_API int gsr_set_option(const char* name, int64_t value);
GSR_API int64_t gsr_get_option(const char* name);
GSR_API int64_t gsr_launch_count(void);

/* Per-stage device timing (CUDA events recorded on the launching stream around each stage while the option
 * "profile" is 1). gsr_profile_read synchronises the device, adds up the elapsed times recorded since the last
 * read, writes GSR_NUM_STAGES milliseconds / call counts, and clears the records. */
#define GSR_NUM_STAGES 9
#define GSR_STAGE_NAMES "preprocess_fwd,depth_order_scan,emit_instances,tile_sort,tile_ranges,render_fwd,render_bwd,preprocess_bwd,apply_weights"
GSR_API int gsr_profile_read(double* ms_out, int64_t* calls_out);

/* ---- host-buffer convenience entry points (what a non-PyTorch host binds; used by bench.py's e2e leg) ---
 * One persistent device context; all pointers below are HOST pointers. The cloud is uploaded once with
 * gsr_host_upload_cloud; each gsr_host_step copies the camera + dL/dcolor image in (H2D) and the rendered
 * image + a few gradient checksums out (D2H) inside the call. */
typedef struct gsr_host_ctx gsr_host_ctx;
GSR_API gsr_host_ctx* gsr_host_create(void);
GSR_API void gsr_host_destroy(gsr_host_ctx* ctx);
GSR_API int gsr_host_upload_cloud(gsr_host_ctx* ctx, int32_t P, int32_t M, const float* means3D, const float* opacities,
                          const float* shs, const float* scales, const float* rotations);
/* settings pointers (bg, viewmatrix, projmatrix, campos) are HOST here. dL_dcolor_host may be NULL (forward only).
 * out_color_host [3,H,W] optional, out_radii_host [P] optional, grad_checksum_host[8] optional (sum of each
 * gradient tensor, computed on the device). Returns num_rendered (>=0) or an error (<0). */
GSR_API int64_t gsr_host_step(gsr_host_ctx* ctx, const gsr_settings* s_host, const float* dL_dcolor_host,
                      float* out_color_host, int32_t* out_radii_host, double* grad_checksum_host);

#ifdef __cplusplus
}
#endif
#endif /* GSR_B200_H_ */
