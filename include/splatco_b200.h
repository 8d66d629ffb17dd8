/*
 * splatco_b200.h — C ABI of libsplatco_b200.so, the B200 (sm_100a) implementation of SplatCo's
 * differentiable render hot path.
 *
 * What this boundary replaces.  The reference reaches its native rasterizer through the pybind
 * module `diff_gaussian_rasterization._C` (package shipped in the reference's submodules.zip;
 * call sites pinned at /root/reference gaussian_renderer/__init__.py:15, :145-171 (forward),
 * :208-242 (visible_filter); SURVEY.md §8b).  Upstream entry points [SURVEY Appendix A.1]:
 *     _C.rasterize_gaussians            -> splatco_preprocess_fwd + splatco_binning + splatco_blend_fwd
 *     _C.rasterize_gaussians_backward   -> splatco_blend_bwd + splatco_preprocess_bwd
 *     _C.rasterize_aussians_filter      -> splatco_visible_filter            (Scaffold-GS fork)
 * and the PyTorch decode in generate_neural_gaussians (gaussian_renderer/__init__.py:18-116,
 * scene/gaussian_model.py:149-169, scene/grids.py:146-201) -> splatco_decode_*.
 *
 * Conventions
 *  - every function returns 0 on success, <0 on error; splatco_last_error() gives the message
 *    (thread-local).  Nothing throws, nothing allocates device memory: the caller owns every buffer
 *    (inputs, outputs and the three opaque workspaces, sized by splatco_*_bytes) and the library
 *    only borrows pointers for the duration of the call on `stream` (a cudaStream_t).
 *  - all array pointers are DEVICE pointers unless the name ends in _host.
 *  - matrices are the reference's transposed (row-vector) 4x4 tensors, read flat:
 *    out.x = m[0]x + m[4]y + m[8]z + m[12]  (scene/cameras.py:54-56).
 *  - no thread-affine state: forward runs on the Python main thread, backward on the autograd thread.
 */
#ifndef SPLATCO_B200_H
#define SPLATCO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPLATCO_ABI_VERSION 1
#define SPLATCO_TILE 16              /* BLOCK_X = BLOCK_Y = 16 (SURVEY Appendix A) */

int splatco_abi_version(void);
const char *splatco_last_error(void);
/* Number of CUDA kernels this library has launched in this process (for bench.py's gpu_launches). */
uint64_t splatco_launch_count(void);

/* ---- workspace sizing (bytes; every internal chunk is 256-byte aligned) ---------------------- */
size_t splatco_geom_bytes(int P);                 /* per-Gaussian projected state               */
size_t splatco_binning_bytes(int64_t R);          /* key/value ping-pong buffers + histograms   */
size_t splatco_image_bytes(int H, int W);         /* tile ranges, final_T, n_contrib            */

/* Byte offsets of the chunks inside each workspace, for tests and debuggers.
 * geom   : [0] rec float4[3P] (x,y,conA,conB | conC,opacity,r,g | b,depth,radius,0)  [1] depths f32[P]
 *          [2] tiles_touched u32[P]  [3] block_sums u32[nb]  [4] block_offsets u32[nb]  [5] total u32
 * binning: [0] keys0 u64[R] [1] keys1 u64[R] [2] vals0 u32[R] [3] vals1 u32[R] [4] hist u32[256*nsb]
 *          [5] bin_totals u32[256]
 * image  : [0] ranges int2[T] [1] final_T f32[HW] [2] n_contrib i32[HW]
 * Returns the number of chunks written (<= max_chunks). */
int splatco_geom_layout(int P, size_t *offsets, int max_chunks);
int splatco_binning_layout(int64_t R, size_t *offsets, int max_chunks);
int splatco_image_layout(int H, int W, size_t *offsets, int max_chunks);
/* 0/1: which of the ping-pong buffers (keys0/vals0 or keys1/vals1) holds the sorted list. */
int splatco_sorted_buffer_index(int H, int W);

/* ---- anchor prefilter: replaces GaussianRasterizer.visible_filter ----------------------------
 * (gaussian_renderer/__init__.py:239-242).  scales is read with a row stride (in floats) because
 * the reference passes the strided view get_scaling[:, :3] of an [N,6] tensor. */
int splatco_visible_filter(int N, const float *means3D, const float *scales, int scale_stride,
                           const float *rots, float scale_mod, const float *view, const float *proj,
                           float tanfovx, float tanfovy, int H, int W, int32_t *radii_out,
                           void *stream);

/* Same filter, plus what render() derives from it next: mask_out[N] (uint8 0/1 = radii > 0, the bool tensor
 * prefilter_voxel returns, gaussian_renderer/__init__.py:243-244), the ascending list idx_out[<= N] of the visible
 * anchors (what the boolean indexing at :21-29 computes) and their count (device, in ws; copied to count_host
 * (pinned) asynchronously if not NULL).  ws: splatco_visible_compact_ws_bytes(N). */
size_t splatco_visible_compact_ws_bytes(int N);
/* Device address (inside ws) of the visible-anchor count splatco_visible_filter_compact leaves behind. */
const int32_t *splatco_visible_compact_count_ptr(const void *ws, int N);
int splatco_visible_filter_compact(int N, const float *means3D, const float *scales, int scale_stride,
                                   const float *rots, float scale_mod, const float *view, const float *proj,
                                   float tanfovx, float tanfovy, int H, int W, int32_t *radii_out, uint8_t *mask_out,
                                   int32_t *idx_out, void *ws, int32_t *count_host, void *stream);

/* ---- forward, stage 1: preprocess + tile counts + scan --------------------------------------
 * Fills geom, radii_out[P]; leaves the instance count R in geom (device) and, if
 * num_rendered_host != NULL (pinned host memory), copies it there asynchronously on `stream`. */
int splatco_preprocess_fwd(int P, const float *means3D, const float *scales, int scale_stride,
                           const float *rots, const float *opacities, const float *colors,
                           float scale_mod, const float *view, const float *proj, float tanfovx,
                           float tanfovy, int H, int W, int32_t *radii_out, void *geom,
                           int32_t *num_rendered_host, void *stream);
/* Same, for callers whose live row count is still on the device: the input arrays (and geom, radii_out)
 * are sized for P_max rows, *P_dev (device, e.g. splatco_decode_count_ptr) holds the number of valid
 * rows; rows beyond it get radii 0 / no tiles.  Every later stage is then called with P = P_max.  Lets
 * render() read the decode's survivor count M and the instance count R with ONE host sync. */
int splatco_preprocess_fwd_counted(int P_max, const int32_t *P_dev, const float *means3D,
                                   const float *scales, int scale_stride, const float *rots,
                                   const float *opacities, const float *colors, float scale_mod,
                                   const float *view, const float *proj, float tanfovx, float tanfovy,
                                   int H, int W, int32_t *radii_out, void *geom,
                                   int32_t *num_rendered_host, void *stream);

/* 1 when splatco_binning(P, R, H, W) will take the tile-segmented path, for which R may be an upper bound on the
 * instance count (a capacity: all writes are clamped to it).  0: the call falls back to the radix composition
 * (splatco_binning_radix), which needs the exact R -- do not pass a guessed capacity then. */
int splatco_binning_accepts_capacity(int P, int64_t R, int H, int W);
/* ---- forward, stage 2: the sorted per-tile instance lists ------------------------------------
 * Produces what upstream's duplicateWithKeys + stable 64-bit SortPairs + identifyTileRanges produce:
 * sorted keys (tile << 32 | depth bits), the sorted Gaussian-id list and the per-tile ranges, bit for
 * bit.  splatco_binning is tile-segmented (count per tile, scan, scatter into segments, per-tile sort
 * in shared memory; see csrc/binning.cu); R is the capacity of the binning buffers and must be >= the
 * value produced by stage 1.  splatco_binning_radix is the literal composition of the three upstream
 * stages (global LSD radix sort), which are also exported individually so parity tests can check
 * keys, permutation and ranges one by one. */
int splatco_binning(int P, int64_t R, int H, int W, const int32_t *radii, const void *geom,
                    void *binning, void *image, void *stream);
int splatco_binning_radix(int P, int64_t R, int H, int W, const int32_t *radii, const void *geom,
                          void *binning, void *image, void *stream);
int splatco_duplicate_with_keys(int P, int64_t R, int H, int W, const int32_t *radii,
                                const void *geom, void *binning, void *stream);
int splatco_sort_pairs(int64_t R, int H, int W, void *binning, void *stream);
int splatco_identify_tile_ranges(int64_t R, int H, int W, const void *binning, void *image,
                                 void *stream);

/* ---- forward, stage 3: per-tile front-to-back alpha blend ------------------------------------ */
int splatco_blend_fwd(int64_t R, int H, int W, const float *bg, const void *geom, const void *binning,
                      void *image, float *out_color /* [3,H,W] */, void *stream);

/* ---- backward --------------------------------------------------------------------------------
 * blend_bwd ACCUMULATES into the four gradient arrays (caller zero-fills them):
 * dL_dmean2D[P,3] (x,y scaled by 0.5W / 0.5H, z untouched), dL_dconic[P,3], dL_dopacity[P],
 * dL_dcolor[P,3].  preprocess_bwd OVERWRITES dL_dmeans3D[P,3], dL_dscales[P,3], dL_drots[P,4]. */
int splatco_blend_bwd(int P, int64_t R, int H, int W, const float *bg, const void *geom,
                      const void *binning, const void *image, const float *dL_dpix /* [3,H,W] */,
                      float *dL_dmean2D, float *dL_dconic, float *dL_dopacity, float *dL_dcolor,
                      void *stream);

/* Same-GPU comparator (NOT used by the product path): the upstream rasterizer's blend STRUCTURE restated -- 256-instance
 * batches, every pixel evaluates every staged instance, nine global atomicAdds per (pixel, instance) in the backward
 * (SURVEY.md Appendix A.4 / A.5; builder-authored, the reference's own source is absent).  Same arguments, workspaces
 * and results as splatco_blend_fwd / splatco_blend_bwd; bench.py times both (`gpu_baseline`). */
int splatco_blend_fwd_upstream(int64_t R, int H, int W, const float *bg, const void *geom, const void *binning,
                               void *image, float *out_color, void *stream);
int splatco_blend_bwd_upstream(int P, int64_t R, int H, int W, const float *bg, const void *geom, const void *binning,
                               const void *image, const float *dL_dpix, float *dL_dmean2D, float *dL_dconic,
                               float *dL_dopacity, float *dL_dcolor, void *stream);

/* A/B switch of the blend kernels (process-wide; timing and debugging only; 0 keeps the current choice).
 *   fwd: 1 = warp-synchronous walk of the patch masks (one splat per warp step), 2 = per-pixel candidate lists from
 *        per-row alpha >= 1/255 spans, every lane walks its own list (default)
 *   bwd: 1 = per-visit nine-sum transposition buffer, 2 = two-value matrix-form reduction with constant-weight FMAs (default),
 *        3 = the same with 256-splat batches
 * Environment: SPLATCO_BLEND_FWD, SPLATCO_BLEND_BWD. */
int splatco_blend_set_impl(int fwd, int bwd);
/* Work census of a view's blend (measurement aid, bench.py's issue-slot roofline): out2[0] = (pixel, instance) pairs
 * the front-to-back walk visits before each pixel terminates, out2[1] = LIVE pairs among them (alpha >= 1/255: the pairs
 * that contribute colour and receive gradients).  out2: two device uint64. */
int splatco_blend_census(int64_t R, int H, int W, const void *geom, const void *binning, const void *image,
                         unsigned long long *out2, void *stream);
int splatco_preprocess_bwd(int P, const float *means3D, const float *scales, int scale_stride,
                           const float *rots, float scale_mod, const float *view, const float *proj,
                           float tanfovx, float tanfovy, int H, int W, const int32_t *radii,
                           const float *dL_dmean2D, const float *dL_dconic, float *dL_dmeans3D,
                           float *dL_dscales, float *dL_drots, void *stream);

/* ---- depth and alpha maps (opt-in; the colour-only entry points above are unchanged) ----------
 * Same walk and contributor set as the colour: for each pixel
 *   depth[p] = sum_i z_i alpha_i T_i   (view-space z of each Gaussian, background 0: ACCUMULATED depth;
 *                                       the expected depth is depth / alpha, which the caller forms)
 *   alpha[p] = 1 - T_final[p]
 * These entry points always run the v2 blend kernels; splatco_blend_set_impl does not apply to them.
 *
 * blend_fwd_depth_alpha: what splatco_blend_fwd computes (out_color, and final_T / n_contrib in the image workspace,
 * bit for bit), plus the caller-owned maps out_depth[H,W] and out_alpha[H,W]. */
int splatco_blend_fwd_depth_alpha(int64_t R, int H, int W, const float *bg, const void *geom, const void *binning,
                                  void *image, float *out_color /* [3,H,W] */, float *out_depth /* [H,W] */,
                                  float *out_alpha /* [H,W] */, void *stream);
/* blend_bwd_depth_alpha: the backward of the three maps.  Any of dL_dpix [3,H,W], dL_ddepth_map [H,W] and
 * dL_dalpha_map [H,W] may be NULL (= zero), but not all three.  Like splatco_blend_bwd it ACCUMULATES into
 * caller-zeroed dL_dmean2D, dL_dconic, dL_dopacity, dL_dcolor, and into dL_ddepth[P] (dL / d view-space z), which
 * splatco_preprocess_bwd_depth takes on to dL_dmeans3D. */
int splatco_blend_bwd_depth_alpha(int P, int64_t R, int H, int W, const float *bg, const void *geom,
                                  const void *binning, const void *image, const float *dL_dpix,
                                  const float *dL_ddepth_map, const float *dL_dalpha_map, float *dL_dmean2D,
                                  float *dL_dconic, float *dL_dopacity, float *dL_dcolor, float *dL_ddepth,
                                  void *stream);
/* preprocess_bwd_depth: splatco_preprocess_bwd plus dL_ddepth[P] . (dz_view / dmean3D) in dL_dmeans3D. */
int splatco_preprocess_bwd_depth(int P, const float *means3D, const float *scales, int scale_stride,
                                 const float *rots, float scale_mod, const float *view, const float *proj,
                                 float tanfovx, float tanfovy, int H, int W, const int32_t *radii,
                                 const float *dL_dmean2D, const float *dL_dconic, float *dL_dmeans3D,
                                 float *dL_dscales, float *dL_drots, const float *dL_ddepth, void *stream);

/* ---- camera gradients ---------------------------------------------------------------------------
 * Both camera entry points WRITE (do not accumulate) their camera gradient, reduced in a fixed order: the same inputs
 * give bitwise the same result.  ws: caller-owned scratch of splatco_camera_grad_ws_bytes(n) bytes, n = P Gaussians
 * for the preprocess backward, n = V visible anchors for the decode backward.  Neither needs it zeroed. */
size_t splatco_camera_grad_ws_bytes(int n);
/* preprocess_bwd_camera: the per-Gaussian outputs of splatco_preprocess_bwd (dL_ddepth NULL) or of
 * splatco_preprocess_bwd_depth (dL_ddepth given), computed by the same kernels, plus dL_dview[16] and dL_dproj[16]:
 * the gradients with respect to the 16 floats of view and proj as the kernels read them.  The forward never reads
 * view[3,7,11,15] or proj[2,6,10,14]; their gradients are 0.  Clamped t.x / t.y (beyond 1.3 tanfov) count as
 * constants, as in the per-Gaussian backward. */
int splatco_preprocess_bwd_camera(int P, const float *means3D, const float *scales, int scale_stride,
                                  const float *rots, float scale_mod, const float *view, const float *proj,
                                  float tanfovx, float tanfovy, int H, int W, const int32_t *radii,
                                  const float *dL_dmean2D, const float *dL_dconic, float *dL_dmeans3D,
                                  float *dL_dscales, float *dL_drots, const float *dL_ddepth, void *ws,
                                  float *dL_dview, float *dL_dproj, void *stream);

/* ---- antialiasing (opt-in; the entry points above are unchanged) ------------------------------------
 * The screen-space mip filter with opacity compensation.  With (a0, b, c0) the projected 2D covariance before the
 * 0.3 px^2 dilation and (a, b, c) = (a0 + 0.3, b, c0 + 0.3) after it, each Gaussian's opacity is scaled by
 *     rho = sqrt(max(2.5e-5, (a0 c0 - b^2) / (a c - b^2)))
 * so that a Gaussian smaller than a pixel keeps its integrated weight instead of being drawn as a full-opacity blob.
 *
 * preprocess_fwd_aa / preprocess_fwd_aa_counted: splatco_preprocess_fwd / splatco_preprocess_fwd_counted with the
 * record's opacity opacities[i] * rho.  radii, tiles, depths, the conic and the rest of the record are bit for bit
 * those of the plain calls; the binning and blend entry points take the geometry workspace unchanged. */
int splatco_preprocess_fwd_aa(int P, const float *means3D, const float *scales, int scale_stride,
                              const float *rots, const float *opacities, const float *colors,
                              float scale_mod, const float *view, const float *proj, float tanfovx,
                              float tanfovy, int H, int W, int32_t *radii_out, void *geom,
                              int32_t *num_rendered_host, void *stream);
int splatco_preprocess_fwd_aa_counted(int P_max, const int32_t *P_dev, const float *means3D,
                                      const float *scales, int scale_stride, const float *rots,
                                      const float *opacities, const float *colors, float scale_mod,
                                      const float *view, const float *proj, float tanfovx, float tanfovy,
                                      int H, int W, int32_t *radii_out, void *geom,
                                      int32_t *num_rendered_host, void *stream);
/* preprocess_bwd_aa: the preprocess backward of an antialiased forward.  On entry dL_dopacity[P] holds what the blend
 * backward accumulated (dL / d record opacity); it is rewritten IN PLACE to dL/dopacities = that * rho, and
 * dL/drho = that * opacities[i] is taken on through (a, b, c) to dL_dmeans3D, dL_dscales and dL_drots.
 * dL_ddepth [P] may be NULL (as splatco_preprocess_bwd) or given (as splatco_preprocess_bwd_depth).  ws, dL_dview and
 * dL_dproj are either all NULL or all given (as splatco_preprocess_bwd_camera, including the rho term). */
int splatco_preprocess_bwd_aa(int P, const float *means3D, const float *scales, int scale_stride,
                              const float *rots, float scale_mod, const float *view, const float *proj,
                              float tanfovx, float tanfovy, int H, int W, const int32_t *radii,
                              const float *dL_dmean2D, const float *dL_dconic, float *dL_dmeans3D,
                              float *dL_dscales, float *dL_drots, const float *opacities, float *dL_dopacity,
                              const float *dL_ddepth, void *ws, float *dL_dview, float *dL_dproj, void *stream);

/* ---- anchor decode: replaces generate_neural_gaussians -----------------------------------------
 * (gaussian_renderer/__init__.py:18-116; FeaturePlanes.forward scene/gaussian_model.py:149-169;
 * PlaneGrid scene/grids.py:146-201; heads scene/gaussian_model.py:316-337).
 * The kernels are specialised for feat_dim = 32 and n_offsets = 10 (the reference's defaults,
 * arguments/__init__.py:50-51); other values are rejected with an error.
 * All pointers are device pointers; arrays indexed [3] run over activate levels / heads
 * (heads: 0 opacity, 1 cov, 2 colour).  Entries of levels > `level` may be NULL. */
typedef struct splatco_decode_desc {
    int32_t N, V, K, rc, level, app_dim;   /* anchors, visible anchors, n_offsets, channels per plane
                                              (num_channels // 3), activate_level 0..2, appearance dim */
    int32_t E[3];                          /* plane edge of k0s[0] (TA level), k0s[1], k0s[2]           */
    int32_t use_dist[3];                   /* add_opacity_dist, add_cov_dist, add_color_dist            */
    int32_t update_running;                /* 1: update BatchNorm running stats in place (train mode)   */
    const float *xyz_min, *xyz_max, *cam;  /* DEVICE pointers to 3 floats each: plane bbox (PlaneGrid.xyz_min/max)
                                              and camera_center — read on the device, no host sync needed  */
    float bn_eps, bn_momentum;
    const float *anchor_feat, *anchor, *offset, *scaling;   /* [N,32] [N,3] [N,K,3] [N,6] (activated)   */
    const int32_t *vis;                    /* [V] ascending indices of the visible anchors              */
    const float *plane[9];                 /* [level*3 + {xy,xz,yz}] each [rc,E,E]                       */
    const float *att[3];                   /* TriPlaneAttention output planes of level 0, [rc,E0,E0]     */
    const float *bn_w[3], *bn_b[3], *lin_w[3], *lin_b[3];       /* FeaturePlanes.models[l]      */
    const float *cbn_w[3], *cbn_b[3], *clin_w[3], *clin_b[3];   /* FeaturePlanes.CTX_models[l]  */
    float *bn_rm[3], *bn_rv[3], *cbn_rm[3], *cbn_rv[3];         /* running_mean / running_var   */
    int64_t *bn_nbt[3], *cbn_nbt[3];                            /* num_batches_tracked          */
    const float *w1[3], *b1[3], *w2[3], *b2[3];                 /* head Linear layers (torch [out,in]) */
    const float *app_vec;                  /* [app_dim] embedding row of this camera, or NULL           */
    const float *noise;                    /* [V, DP - 6*rc] additive plane-feature noise U(-.5,.5)*Q for
                                              levels >= 1 (scene/grids.py:159-164), or NULL (Q = 0)     */
    float noise_q;                         /* used when noise == NULL: != 0 adds U(-.5,.5) * noise_q to the same
                                              features, generated in the kernel from noise_seed             */
    uint64_t noise_seed;
    int32_t plane_layout;                  /* 0: plane[] / att[] (and their gradients) are [rc,E,E] as the
                                              reference stores them; 1: [E,E,8] channel-last copies made by
                                              splatco_pack_planes (rc <= 8)                              */
    const int32_t *V_dev;                  /* NULL: V is the exact number of visible anchors.  Else (forward of the two-stage
                                              implementation only): DEVICE pointer to the count -- e.g.
                                              splatco_visible_compact_count_ptr -- read by the kernels; V is then only an
                                              upper bound (grids, buffer rows), `vis` has at least V entries, and the host
                                              need not wait for the prefilter before it queues the decode             */
    int32_t V_layout;                      /* rows the workspaces were sized / laid out for (the V passed to
                                              splatco_decode_*_ws_bytes); 0 = V.  A forward queued with V_dev uses
                                              V = V_layout = capacity; its backward passes the exact V and the same V_layout */
} splatco_decode_desc;

/* Gradient destinations (same shapes as the inputs).  EVERY destination is ACCUMULATED into (+=):
 * the caller zero-fills a buffer once and may hand the same buffer to the decode backward of every
 * view of an iteration (train.py:171-240 sums the mv views' losses before one backward), which
 * removes the per-view N-row / plane-sized temporaries and the autograd additions between them.
 * anchor_feat/anchor/offset/scaling are [N,*] (only visible rows are touched); plane/att receive
 * bilinear scatter atomics.  NULL plane/att/parameter entries are skipped. */
typedef struct splatco_decode_grads {
    float *anchor_feat, *anchor, *offset, *scaling;
    float *plane[9];
    float *att[3];
    float *bn_w[3], *bn_b[3], *lin_w[3], *lin_b[3];
    float *cbn_w[3], *cbn_b[3], *clin_w[3], *clin_b[3];
    float *w1[3], *b1[3], *w2[3], *b2[3];
    float *app_vec;
} splatco_decode_grads;

/* Channel-last copies of three [rc,E,E] planes: out[(y*E + x)*8 + ch] (ch >= rc zero).  The gather reads 4 sectors
 * per plane sample instead of 4 per channel, and the backward's bilinear scatter issues one request per texel.
 * splatco_unpack_planes_add adds channel-last gradients back into [rc,E,E] gradients (+=). */
int splatco_pack_planes(int rc, int E, const float *xy, const float *xz, const float *yz, float *pxy, float *pxz,
                        float *pyz, void *stream);
int splatco_unpack_planes_add(int rc, int E, const float *gpxy, const float *gpxz, const float *gpyz, float *gxy,
                              float *gxz, float *gyz, void *stream);

size_t splatco_decode_fwd_ws_bytes(int V, int rc, int level);
size_t splatco_decode_bwd_ws_bytes(int V, int rc, int level);
/* Stage 1: gather + BN statistics + MLP heads + opacity mask.  Writes neural_opacity[V*K] (tanh
 * output), mask[V*K] (uint8 0/1) and the survivor count M (device, inside ws; copied to
 * M_host (pinned) asynchronously if not NULL). */
int splatco_decode_fwd(const splatco_decode_desc *d, void *ws, float *neural_opacity, uint8_t *mask,
                       int32_t *M_host, void *stream);
/* Two implementations sit behind the decode entry points: 1 = the three-stage chain (geo -> hidden -> heads), 2 = the
 * collapsed two-stage pipeline (default for plane grids with <= 5 channels per plane; csrc/decode2.cuh).  The choice
 * is process-wide, must not change between a forward and its backward, and is meant for A/B timing and debugging
 * (environment: SPLATCO_DECODE_IMPL=1|2). */
int splatco_decode_set_impl(int impl);
/* Measurement aid: with profiling enabled the library brackets the tensor-core MLP kernel of every splatco_decode_fwd /
 * splatco_decode_bwd with CUDA events on the caller's stream; splatco_decode_profile_read returns the device time (ms)
 * of the most recent forward / backward MLP kernel once the stream has been synchronised. */
int splatco_decode_profile(int enable);      /* 0 off, 1 event timing of the MLP kernels, 2 phase trace (below) */
/* With splatco_decode_profile(2): clock64 stamps of CTA 0 at the phase boundaries of its first tiles, [0..63] forward
 * MLP kernel (8 per tile), [64..127] backward MLP kernel (16 per tile); read after synchronising.  tools/decode_trace.py. */
int splatco_decode_trace_read(unsigned long long *out128);
int splatco_decode_profile_read(float *fwd_mlp_ms, float *bwd_mlp_ms);
int splatco_decode_get_impl(void);
/* Introspection for the tests: the gathered rows [V, LDX] of a finished splatco_decode_fwd (LDX = round_up4(DP + 71),
 * columns [plane features DP | anchor_feat 32 | anchor 3 | offsets 30 | scaling 6 | zero padding]), whatever the
 * implementation's internal layout. */
int splatco_decode_gathered_rows(const void *ws, int V, int rc, int level, float *out, void *stream);
/* Device address (inside ws) of the survivor count M that splatco_decode_fwd leaves behind. */
const int32_t *splatco_decode_count_ptr(const void *ws, int V, int rc, int level);
/* Stage 2: stable compaction + post-processing into the M surviving Gaussians.  M is only tested for
 * zero: a caller that has not read M back yet passes output arrays with V*K rows and M = V*K. */
int splatco_decode_emit(const splatco_decode_desc *d, const void *ws, int M, float *xyz, float *color,
                        float *opacity, float *scaling, float *rot, void *stream);
/* Backward of both stages.  d_neural_opacity ([V*K]) may be NULL. */
int splatco_decode_bwd(const splatco_decode_desc *d, const void *fwd_ws, void *bwd_ws, int M,
                       const float *d_xyz, const float *d_color, const float *d_opacity,
                       const float *d_scaling, const float *d_rot, const float *d_neural_opacity,
                       const splatco_decode_grads *g, void *stream);
/* splatco_decode_bwd (which accumulates into g) plus d_cam[3] = dL / d camera_center (written): minus the sum, over
 * the visible anchors, of the gradient of the view direction and distance (anchor - camera_center).  ws:
 * splatco_camera_grad_ws_bytes(V). */
int splatco_decode_bwd_camera(const splatco_decode_desc *d, const void *fwd_ws, void *bwd_ws, int M,
                              const float *d_xyz, const float *d_color, const float *d_opacity,
                              const float *d_scaling, const float *d_rot, const float *d_neural_opacity,
                              const splatco_decode_grads *g, void *ws, float *d_cam, void *stream);

/* ---- TriPlaneAttention over the TA-level planes (SURVEY.md §8 row f2) ---------------------------
 * Replaces TriPlaneAttention.forward (scene/grids.py:22-64) as applied at scene/grids.py:166-169 to
 * cat(xy_plane, xz_plane, yz_plane) of k0s[0]: channel attention (global avg + max pool -> 1x1 conv
 * C -> hidden -> ReLU -> 1x1 conv -> sigmoid) then spatial attention (channel mean / max -> ksize x ksize
 * conv, zero padding, no bias -> sigmoid).  Planes are [rc, E, E] each, C = 3*rc <= 32, hidden <= 8,
 * ksize must be 7 (what the reference constructs).  w_ca1 [hidden, C], w_ca2 [C, hidden],
 * w_sa [1, 2, 7, 7] are the Conv2d weights in torch layout.  fwd_ws keeps what the backward needs.
 * splatco_ta_bwd ACCUMULATES (+=) into g_xy/g_xz/g_yz and the three weight gradients (NULL weight
 * gradients are skipped), like splatco_decode_bwd. */
size_t splatco_ta_fwd_ws_bytes(int rc, int E);
size_t splatco_ta_bwd_ws_bytes(int rc, int E);
int splatco_ta_fwd(int rc, int E, int hidden, int ksize, const float *xy, const float *xz, const float *yz,
                   const float *w_ca1, const float *w_ca2, const float *w_sa, void *fwd_ws, float *out_xy,
                   float *out_xz, float *out_yz, void *stream);
int splatco_ta_bwd(int rc, int E, int hidden, int ksize, const float *xy, const float *xz, const float *yz,
                   const float *w_ca1, const float *w_ca2, const float *w_sa, void *fwd_ws, void *bwd_ws,
                   const float *g_out_xy, const float *g_out_xz, const float *g_out_yz, float *g_xy,
                   float *g_xz, float *g_yz, float *g_w_ca1, float *g_w_ca2, float *g_w_sa, void *stream);

/* ---- densification statistics of one view (SURVEY.md §8 row f1) --------------------------------
 * Replaces GaussianModel.training_statis (scene/gaussian_model.py:761-782; called at train.py:264-266 with the
 * last view's outputs).  vis_idx [V]: ascending indices of the anchors in voxel_visible_mask; neural_opacity
 * [V*K]; selection_mask [V*K] (uint8, the decode's opacity mask) with selection_excl [V*K] its exclusive prefix
 * sum (= index of the offset among the M rendered Gaussians); update_filter [M] (uint8, radii > 0);
 * viewspace_grad [M,3] (.grad of viewspace_points; may be NULL if M == 0).  Updates in place opacity_accum [N],
 * anchor_demon [N], offset_gradient_accum [N*K], offset_denom [N*K]. */
int splatco_training_statis(int V, int K, const int32_t *vis_idx, const float *neural_opacity,
                            const uint8_t *selection_mask, const int32_t *selection_excl,
                            const uint8_t *update_filter, const float *viewspace_grad, float *opacity_accum,
                            float *anchor_demon, float *offset_gradient_accum, float *offset_denom, void *stream);

/* ---- fused L1 + SSIM image loss (SURVEY.md §8 row f3) ------------------------------------------
 * Replaces l1_loss + ssim of utils/loss_utils.py:17-18,33-63 as combined at train.py:192-196:
 *   loss = (1 - lambda_dssim) * mean|img - gt| + lambda_dssim * (1 - mean(ssim_map(img, gt)))
 * img, gt: [C,H,W] fp32.  fwd writes out3[0..2] = (loss, l1, ssim) on the device and keeps the three
 * partial-derivative maps in ws (splatco_loss_ws_bytes); bwd writes dL/dimg = *grad_loss * dloss/dimg. */
size_t splatco_loss_ws_bytes(int C, int H, int W);
int splatco_l1_ssim_fwd(int C, int H, int W, const float *img, const float *gt, float lambda_dssim, void *ws,
                        float *out3, void *stream);
int splatco_l1_ssim_bwd(int C, int H, int W, const float *img, const float *gt, float lambda_dssim, const void *ws,
                        const float *grad_loss, float *dL_dimg, void *stream);

/* Scaling regulariser of the per-view loss (train.py:195): out[0] = mean_i (scaling[i,0] * scaling[i,1] * scaling[i,2]),
 * scaling [M,3] contiguous fp32, M >= 1; ws: 16 bytes.  bwd writes d_scaling = *grad_loss * d out / d scaling.  Unlike
 * torch's prod backward (which counts zeros with a device-to-host read) neither call waits for the GPU. */
int splatco_scaling_reg_fwd(int M, const float *scaling, void *ws, float *out, void *stream);
int splatco_scaling_reg_bwd(int M, const float *scaling, const float *grad_loss, float *d_scaling, void *stream);

/* ---- cross-view consistency term of the multi-view batch (SURVEY.md §8 rows a12 / f3) ----------------
 * Replaces the pair loop of train.py:199-216 (+ align_images, train.py:79-96; summed in at train.py:237-239):
 *   for i < j:  s = ssim(real_i, real_j);  loss_ij = s * |l1_loss(real_i - real_j, gen_i - gen_j)| if s > gate else 0
 * The crop is per pair (align_images crops the pair's four images to their common top-left region).
 * gen[i], real[i]: host arrays of n_views device pointers to contiguous [C, img_h[i], img_w[i]] fp32 images (a view's
 * rendered and ground-truth image have the same size).  pair_ssim [n(n-1)/2] (device): ssim(real_i, real_j) on the pair's
 * crop, in (0,1),(0,2),...,(n-2,n-1) order (splatco_l1_ssim_fwd with lambda 1 gives it).  fwd writes out[0] = sum_ij loss_ij
 * and out[1 + p] = loss of pair p; bwd writes every view's full dL/dgen_i = *grad_loss * d out[0] / d gen_i. */
#define SPLATCO_MVC_MAX_VIEWS 8
size_t splatco_mv_consistency_ws_bytes(int n_views);
int splatco_mv_consistency_fwd(int n_views, int C, const float *const *gen, const float *const *real, const int *img_h,
                               const int *img_w, const float *pair_ssim, float ssim_gate, void *ws, float *out,
                               void *stream);
int splatco_mv_consistency_bwd(int n_views, int C, const float *const *gen, const float *const *real, float *const *dgen,
                               const int *img_h, const int *img_w, const void *ws, const float *grad_loss, void *stream);

/* ---- plane total-variation regulariser (SURVEY.md §8 row f2) -----------------------------------------
 * Replaces PlaneGrid.total_variation_add_grad (scene/grids.py:240-250; GaussianLearner.tv_loss,
 * scene/gaussian_model.py:217-220; train.py:242-243) for ONE plane [C,H,W]:
 *   grad += d/dplane [ w/6 * (smooth_l1(p[:,1:,:], p[:,:-1,:], sum) + smooth_l1(p[:,:,1:], p[:,:,:-1], sum)) ]
 * (the reference's six terms are these two for each of the three planes).  grad is the plane's .grad, updated in place. */
int splatco_tv_add_grad(int C, int H, int W, const float *plane, float *grad, float w, void *stream);

/* ---- anchor growing (SURVEY.md §8 row f4) -------------------------------------------------------------
 * Replaces one pass of the loop of GaussianModel.anchor_growing (scene/gaussian_model.py:832-925).
 * Offset slot t = anchor * K + k, t < n_stat (= rows of the statistics; anchors grown by an earlier pass have none).
 * A slot is a candidate if cand_mask[t] (when cand_mask != NULL) or else if
 *   grads[t] >= threshold && offset_mask[t] && rand[t] > rand_cut            (gaussian_model.py:839-846).
 * Its position anchor + offset * scaling[:, :3] is rounded to the voxel grid of size cur_size (div_mode 0: multiply by
 * the fp32 reciprocal like torch's CUDA `tensor / scalar`; 1: true division like torch's CPU kernel); voxels that already
 * hold one of the N anchors are dropped; the new anchors are the remaining distinct voxels in torch.unique(dim=0)'s
 * row order (x, y, z signed-lexicographic) times cur_size, and new_feat is the per-voxel channel-wise maximum of the
 * candidates' anchor features (torch_scatter.scatter_max).  Three calls with two 4-byte read-backs in between:
 *   splatco_grow_count  -> counts[0] = number of candidates                 (host reads it, allocates ws)
 *   splatco_grow_unique -> counts[2] = number of new anchors                (host reads it, allocates outputs)
 *   splatco_grow_emit   -> new_anchor [n_new,3], new_feat [n_new,F]
 * counts: 4 x uint32 on the device.  scaling: activated (exp), row stride scale_stride floats. */
size_t splatco_grow_ws_bytes(int64_t n_cand);
int splatco_grow_count(int64_t n_stat, const uint8_t *cand_mask, const float *grads, float threshold,
                       const uint8_t *offset_mask, const float *rand, float rand_cut, uint32_t *counts, void *stream);
int splatco_grow_unique(int N, int K, int64_t n_stat, const float *anchors, const float *offsets, const float *scaling,
                        int scale_stride, const uint8_t *cand_mask, const float *grads, float threshold,
                        const uint8_t *offset_mask, const float *rand, float rand_cut, float cur_size, int div_mode,
                        int64_t n_cand, void *ws, uint32_t *counts, void *stream);
int splatco_grow_emit(int K, int F, float cur_size, int64_t n_cand, int64_t n_new, void *ws, const float *anchor_feat,
                      float *new_anchor, float *new_feat, void *stream);

/* ---- CVPM pruning mask (SURVEY.md §8 row a13) ---------------------------------------------------------
 * Replaces the point-cloud half of GaussianModel.compute_fast_loss_with_key_points (scene/gaussian_model.py:1163-1165,
 * 1178-1216; train.py:218-234): mask[i] = anchor i lies within distance_threshold of the line through t1 and t2 AND
 * (is closer than min_cam_distance to t1 or t2, OR is a sigma_threshold-sigma outlier of the cloud on some axis).
 * points [N,3]; t1, t2: 3 floats each and ssim: 1 float (ssim(real_1, real_2); NULL = no gate), all on the DEVICE —
 * the mask is all-false when *ssim < ssim_threshold, without a host sync.  mask [N] uint8, count [1] = its sum. */
size_t splatco_cvpm_ws_bytes(void);
int splatco_cvpm_mask(int N, const float *points, const float *t1, const float *t2, const float *ssim,
                      float ssim_threshold, float distance_threshold, float sigma_threshold, float min_cam_distance,
                      void *ws, uint8_t *mask, int32_t *count, void *stream);

/* ---- fused multi-tensor Adam step (SURVEY.md §8 row f2) ------------------------------------------------
 * Replaces `gaussians.optimizer.step()` (train.py:310-312; optimizer of scene/gaussian_model.py:519-572:
 * torch.optim.Adam, eps 1e-15, betas (0.9, 0.999), no weight decay / amsgrad, per-group lr) for fp32 tensors:
 *   m += (g - m)(1 - beta1);  v = v beta2 + (1 - beta2) g^2;  p -= lr / (1 - beta1^step) * m / (sqrt(v) / sqrt(1 - beta2^step) + eps)
 * `tensors` is a HOST array; step is the value AFTER this update's increment (>= 1).  One pass, up to 64 tensors per launch. */
typedef struct splatco_adam_tensor {
    float *param;
    const float *grad;
    float *exp_avg;
    float *exp_avg_sq;
    int64_t numel;
    int64_t step;
    float lr;
    float reserved;
} splatco_adam_tensor;
int splatco_adam_step(int n_tensors, const splatco_adam_tensor *tensors, double beta1, double beta2, double eps, void *stream);

/* ---- diagnostics --------------------------------------------------------------------------------
 * Self-test of the tcgen05 3xTF32 tile-GEMM primitives the decode kernels are built on:
 * C[M,N] = A[M,K] * B[N,K]^T (row-major fp32, N <= 112, K <= 136).  variant bit0: swapped LBO/SBO
 * descriptor convention (expected to be wrong), bit1: single-pass TF32.  Used by tests/test_tc_gpu.py. */
int splatco_tc_gemm_selftest(int M, int N, int K, const float *A, const float *B, float *C, int variant,
                             void *stream);


/* Self-test of the MN-major (transposed-operand) tcgen05 path used by the decode backward's weight-gradient
 * products: C[m][n] = sum_k At[k][m] * Bt[k][n], At [128][128], Bt [128][N], C [128][N], N <= 96.
 * variant bits: 0 A read as an MN-major tile, 1 B read as an MN-major tile (otherwise transposed into K-major tiles by
 * the threads), 2 LBO/SBO roles swapped, 3 single-pass TF32, [4,7) descriptor layout type, 7 unused stride = 0. */
int splatco_tc_wgrad_selftest(int N, const float *At, const float *Bt, float *C, int variant, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* SPLATCO_B200_H */
