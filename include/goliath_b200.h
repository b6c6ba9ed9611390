/*
 * include/goliath_b200.h — C ABI of libgoliath_b200.so (hand-written sm_100a kernels).
 *
 * The drop-in boundary of the goliath render hot path (SURVEY.md §8b).  Every entry point
 *   - takes raw DEVICE pointers (fp32 / int32 / int64, contiguous, layouts exactly as the reference's
 *     tensors), plain sizes and a cudaStream_t passed as void*;
 *   - runs on the CURRENT device of the calling thread and only on the given stream (the reference's
 *     mvpraymarchlib/utilslib launch on stream 0 with no device guard, mvpraymarch.cpp:122,142,176 —
 *     this ABI is the superset behaviour needed for one-process-per-GPU operation);
 *   - never allocates or synchronises: the caller owns outputs, gradients and workspaces;
 *   - returns 0, or the cudaError_t value of the failing launch / argument check.
 * Each declaration names the reference binding it replaces.  The Python-side bindings that mirror the
 * reference's pybind modules live in goliath_b200/{sgutilslib,mvpraymarchlib,utilslib}.py and
 * goliath_b200/gsplat/; INTEGRATION.md shows the stub a goliath maintainer would add.
 */
#ifndef GOLIATH_B200_H_
#define GOLIATH_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* library/ABI version: major*1000 + minor */
int gb_version(void);
/* kernels launched by this library since load / last reset (host counter; bench.py gpu_launches) */
unsigned long long gb_launch_count(void);
void gb_launch_count_reset(void);

/* ---------------------------------------------------------------- sgutilslib (extensions/sgutils/sg.cu) */

/* replaces sgutilslib.evaluate_gaussian_fwd — sg.cu:177-224 (kernel :27-76).
 * lobe_dirs [N,D,3] (already normalised by sgutils.py:75), lobe_sigmas [N,D], light_values [N,L,3],
 * light_pts [N,L,3], prim_pts [N,D,3], n_lights [N] int32, integral [N,D,3] out. w_type in 0..3. */
int gb_sg_evaluate_fwd(const float* lobe_dirs, const float* lobe_sigmas, const float* light_values,
                       const float* light_pts, const float* prim_pts, const int32_t* n_lights, float* integral,
                       int N, int D, int L, int w_type, void* stream);

/* replaces sgutilslib.evaluate_gaussian_bwd — sg.cu:226-277 (kernel :78-175).
 * grad_dirs [N,D,3], grad_sigmas [N,D] are overwritten; grad_light_values [N,L,3] may be NULL, otherwise it
 * is accumulated into (the reference zero-fills it in sgutils.py:43-47). */
int gb_sg_evaluate_bwd(const float* lobe_dirs, const float* lobe_sigmas, const float* light_values,
                       const float* light_pts, const float* prim_pts, const int32_t* n_lights,
                       const float* grad_integral, float* grad_dirs, float* grad_sigmas, float* grad_light_values,
                       int N, int D, int L, int w_type, void* stream);

/* ---------------------------------------------------------------- gsplat 0.1.11 (third-party; call sites
 * ca_code/utils/render_gsplat.py:49-63, 65-78, 90-104) */

/* replaces gsplat._C.project_gaussians_forward.  means3d [G,3], scales [G,3], quats [G,4] (w,x,y,z),
 * viewmat: DEVICE pointer to >= 12 floats, row-major [R|t].  Outputs (all written for every Gaussian;
 * culled ones get zeros): cov3d [G,6], xys [G,2], depths [G], radii [G] i32, conics [G,3],
 * compensation [G], num_tiles_hit [G] i32. */
int gb_project_gaussians_fwd(int G, const float* means3d, const float* scales, float glob_scale,
                             const float* quats, const float* viewmat, float fx, float fy, float cx, float cy,
                             int img_h, int img_w, int block_width, float clip_thresh, float* cov3d, float* xys,
                             float* depths, int32_t* radii, float* conics, float* compensation,
                             int32_t* num_tiles_hit, void* stream);

/* replaces gsplat._C.project_gaussians_backward.  All five gradient outputs are overwritten. */
int gb_project_gaussians_bwd(int G, const float* means3d, const float* scales, float glob_scale,
                             const float* quats, const float* viewmat, float fx, float fy, const float* cov3d,
                             const int32_t* radii, const float* conics, const float* compensation,
                             const float* v_xy, const float* v_depth, const float* v_conic,
                             const float* v_compensation, float* v_cov2d, float* v_cov3d, float* v_mean3d,
                             float* v_scale, float* v_quat, void* stream);

/* replaces gsplat.utils.compute_cumulative_intersects (torch.cumsum int32): inclusive scan. */
size_t gb_cumsum_workspace_bytes(int n);
int gb_cumsum_i32(int n, const int32_t* in, int32_t* out, void* workspace, void* stream);

/* replaces gsplat._C.map_gaussian_to_intersects: isect_ids [I] int64 = (tile_id << 32) | bits(depth),
 * gaussian_ids [I] int32, emitted per Gaussian in row-major tile order. */
int gb_map_gaussian_to_intersects(int G, const float* xys, const float* depths, const int32_t* radii,
                                  const int32_t* cum_tiles_hit, int img_h, int img_w, int block_width,
                                  int64_t* isect_ids, int32_t* gaussian_ids, void* stream);

/* replaces torch.sort(isect_ids) + gather in gsplat.utils.bin_and_sort_gaussians: stable ascending radix
 * sort on the low key_bits bits (32 + ceil(log2(#tiles))). */
size_t gb_sort_workspace_bytes(int64_t n);
int gb_sort_intersects(int64_t n, const int64_t* isect_ids, const int32_t* gaussian_ids, int64_t* isect_sorted,
                       int32_t* gids_sorted, int key_bits, void* workspace, void* stream);

/* replaces gsplat._C.get_tile_bin_edges: tile_bins [T,2] int32, zeroed by the caller. */
int gb_get_tile_bin_edges(int64_t n, const int64_t* isect_sorted, int32_t* tile_bins, void* stream);

/* replaces gsplat._C.rasterize_forward (channels == 3); channels == 4 is the fused rgb+depth pass.
 * colors [G,C], opacities [G], background [C] (device).  out_img [H,W,C], final_Ts [H,W],
 * final_idx [H,W] i32 are fully overwritten. */
int gb_rasterize_fwd(int img_h, int img_w, int block_width, int channels, const int32_t* gids_sorted,
                     const int32_t* tile_bins, const float* xys, const float* conics, const float* colors,
                     const float* opacities, const float* background, float* out_img, float* final_Ts,
                     int32_t* final_idx, void* stream);

/* replaces gsplat._C.rasterize_backward.  v_xy [G,2], v_conic [G,3], v_colors [G,C], v_opacity [G] are
 * accumulated into (caller zeroes them).  v_output_alpha [H,W] may be NULL (no gradient through alpha) here and in every
 * gb_rasterize_*_bwd below. */
int gb_rasterize_bwd(int img_h, int img_w, int block_width, int channels, const int32_t* gids_sorted,
                     const int32_t* tile_bins, const float* xys, const float* conics, const float* colors,
                     const float* opacities, const float* background, const float* final_Ts,
                     const int32_t* final_idx, const float* v_output, const float* v_output_alpha, float* v_xy,
                     float* v_conic, float* v_colors, float* v_opacity, void* stream);

/* ---- B200 blend path (block_width == 16): same results as gb_rasterize_fwd/bwd, different work distribution.
 * These have no counterpart in gsplat's binding; they sit behind the same rasterize_gaussians call
 * (ca_code/utils/render_gsplat.py:65-78,90-104). */

/* gather (xy, conic, opacity, colours, cull box) of every intersection in sorted order: records [n,12] fp32 */
int gb_pack_records(int64_t n, int channels, const int32_t* gids_sorted, const float* xys, const float* conics,
                    const float* colors, const float* opacities, float* records, void* stream);

/* fused-render variant: record opacity = opacity*compensation (render_gsplat.py:72), 4th colour = depth (:97) */
int gb_pack_records_fused(int64_t n, const int32_t* gids_sorted, const float* xys, const float* conics,
                          const float* colors3, const float* depths, const float* opacity, const float* compensation,
                          float* records, void* stream);

/* multi-condition (OLAT) renders: the lighting conditions of a view share geometry, projection and tile lists
 * (ca_code/utils/light_decorator.py:167 feeds the same avatar under one light at a time); this rewrites only the colour
 * quarter of the fused-render records in place: records[i].c = (colors3[gids_sorted[i]], depths[gids_sorted[i]]).
 * n_dev: device int32 count of valid records (may be NULL: cap records). */
int gb_records_set_colors(int64_t cap, const int32_t* n_dev, const int32_t* gids_sorted, const float* colors3,
                          const float* depths, float* records, void* stream);

/* four lighting conditions per blend pass (OLAT, BASELINE config 3): the conditions of a view share every alpha and
 * transmittance, so one walk of the tile lists blends four colour sets (csrc/splat_blend_mom.cu).  "Wide" records [cap,20]
 * fp32 = the 32-byte geometry of the packed records + 4 x rgb; gb_records_widen copies the geometry once per view,
 * gb_records_set_colors4 rewrites the colour part per group of (up to 4) conditions from nk consecutive [G,3] tables. */
int gb_records_widen(int64_t cap, const int32_t* n_dev, const float* records, float* records_wide, void* stream);
int gb_records_set_colors4(int64_t cap, const int32_t* n_dev, const int32_t* gids_sorted, const float* colors, int nk,
                           int64_t G, float* records_wide, void* stream);
/* out_planes [4][H][W][3] (3-channel background added to each). */
int gb_rasterize_multi_fwd(int img_h, int img_w, const int32_t* tile_bins, const int32_t* tile_order, int sched,
                           const float* records_wide, const float* background, float* out_planes, void* stream);
/* v_planes [4][H][W][3]; final_Ts / final_idx from the view's single-condition pass; v_xy / v_conic / v_opacity accumulated;
 * v_colors12 [G,12] (zero-filled): the four colour gradients interleaved per Gaussian, split by gb_colors12_unpack (which
 * also clears it for the next group). */
int gb_rasterize_multi_bwd(int img_h, int img_w, const int32_t* gids_sorted, const int32_t* tile_bins,
                           const int32_t* tile_order, int sched, const float* records_wide, const float* background,
                           const float* final_Ts, const int32_t* final_idx, const float* v_planes, float* v_xy, float* v_conic,
                           float* v_colors12, float* v_opacity, void* stream);
int gb_colors12_unpack(int64_t G, int nk, float* v_colors12, float* v_colors, void* stream);

/* backward glue of the fused render: split v_colors4 / v_opacity_eff into v_colors3, v_opacity, v_comp, v_depth */
int gb_splat_grad_unpack(int G, const float* v_colors4, const float* v_opac_eff, const float* opacity,
                         const float* compensation, float* v_colors3, float* v_opacity, float* v_comp, float* v_depth,
                         void* stream);

/* ---- sync-free ("_dn": device-side n) variants: the intersection count stays on the device (n_dev = last element of
 * cum_tiles_hit), buffers hold `cap` intersections, *overflow is set when the true count exceeds cap.  They remove
 * the host synchronisation the reference performs (gsplat utils: cum_tiles_hit[-1].item()) and make the whole render
 * capturable in a CUDA graph. */
int gb_map_gaussian_to_intersects_dn(int G, const float* xys, const float* depths, const int32_t* radii,
                                     const int32_t* cum_tiles_hit, int img_h, int img_w, int block_width, int64_t cap,
                                     int64_t* isect_ids, int32_t* gaussian_ids, void* stream);
int gb_sort_intersects_dn(int64_t cap, const int32_t* n_dev, const int64_t* isect_ids, const int32_t* gaussian_ids,
                          int64_t* isect_sorted, int32_t* gids_sorted, int key_bits, void* workspace, void* stream);
int gb_get_tile_bin_edges_dn(int64_t cap, const int32_t* n_dev, const int64_t* isect_sorted, int32_t* tile_bins,
                             int32_t* overflow, void* stream);
int gb_pack_records_fused_dn(int64_t cap, const int32_t* n_dev, const int32_t* gids_sorted, const float* xys,
                             const float* conics, const float* colors3, const float* depths, const float* opacity,
                             const float* compensation, float* records, void* stream);

/* ordering inside gb_bin_tiles_pack / gb_bin_tiles_pack_ev: 0 = each tile's (depth key, id) pairs sorted in shared memory
 * by one CTA, no depth ranks (default); 1 = depth ranks of all Gaussians + per-tile rank ordering, the path the rank and
 * tile sort modes below select between (gb_bin_tiles_ranked always takes it).  Identical outputs.
 * GOLIATH_B200_BINSORT=tile|rank. */
int gb_get_bin_sort_mode(void);
void gb_set_bin_sort_mode(int mode);
/* depth ranks of the rank path: 0 = one cooperative LSD kernel over the key bits that vary (default), 1 = four
 * radix passes as separate launches (round 1), 2 = 2048 key buckets + in-bucket ranking of the visible Gaussians (a
 * device flag hands degenerate depth distributions to the cooperative sort; measured slower).  Identical outputs.
 * GOLIATH_B200_RANKSORT=coop|passes|buckets. */
int gb_get_rank_sort_mode(void);
/* per-tile rank ordering of the rank path: 0 = bitmap sort per tile + one grid-wide record gather (default), 1 = one
 * kernel per tile doing both (round 1).  Identical outputs.  GOLIATH_B200_TILESORT=split|fused. */
int gb_get_tile_sort_mode(void);
void gb_set_tile_sort_mode(int mode);
void gb_set_rank_sort_mode(int mode);

/* Bucket binning of the fused render (csrc/splat_bin_tiles.cu): replaces, for the fused path, the whole of gsplat
 * 0.1.11 bin_and_sort_gaussians (compute_cumulative_intersects, map_gaussian_to_intersects, torch.sort,
 * get_tile_bin_edges — call sites ca_code/utils/render_gsplat.py:65-78,90-104) plus the record packing, with the same
 * bit-exact outputs: intersections are bucketed per tile with atomics as (depth key, id) pairs, and each tile's bucket
 * is sorted by one CTA in shared memory (a tile too long for it sorts in its own slots of `records`, which the final
 * record gather overwrites).  Outputs: tile_bins [T,2], tile_order [T]
 * (tile_sched = 1: an SM-affine schedule of gb_tile_schedule_ints(T) int32 instead, see gb_tile_schedule),
 * gids_sorted [cap], records [cap,12]; n_out (device int32, may be NULL) = true intersection count; *overflow = 1
 * when it exceeds cap (the excess is dropped).  Sync-free, never allocates, capturable in a CUDA graph. */
int gb_bin_tiles_supported(int G); /* 1 if one tile's G-bit rank bitmap fits in shared memory */
size_t gb_bin_tiles_workspace_bytes(int G, int num_tiles, int64_t cap);
int gb_bin_tiles_pack(int G, const float* xys, const float* depths, const int32_t* radii, const float* conics,
                      const float* colors3, const float* opacity, const float* compensation, int img_h, int img_w,
                      int block_width, int64_t cap, int32_t* tile_bins, int32_t* tile_order, int tile_sched,
                      int32_t* gids_sorted, float* records, int32_t* n_out, int32_t* overflow, void* workspace,
                      void* stream);
/* Same, with colors3 allowed to arrive late: colors_ready (cudaEvent_t recorded on the stream that writes colors3, or
 * NULL) is waited for on `stream` just before the first kernel that reads colors3 (with the split tile sort: a small
 * kernel after the per-tile sort), so ranks, buckets and the per-tile sort run beside the caller's shade (rgca.py:557-575 precedes
 * render_gsplat.py:65 in the reference; only the colours depend on it). */
int gb_bin_tiles_pack_ev(int G, const float* xys, const float* depths, const int32_t* radii, const float* conics,
                         const float* colors3, const float* opacity, const float* compensation, int img_h, int img_w,
                         int block_width, int64_t cap, int32_t* tile_bins, int32_t* tile_order, int tile_sched,
                         int32_t* gids_sorted, float* records, int32_t* n_out, int32_t* overflow, void* workspace,
                         void* colors_ready, void* stream);

/* Binning WITHOUT the sorted-record gather, for gb_rasterize_ranked_fwd/bwd: ranks_sorted [cap] (per tile, the depth ranks
 * in blend order), rec_by_rank [G,12] (one 48-byte record per visible Gaussian, at its depth rank) and rank_to_gid [G] are
 * written to the CALLER's arrays (they must live until the backward).  Everything else as gb_bin_tiles_pack_ev.  No
 * counterpart in gsplat: it replaces the per-intersection sorted arrays of bin_and_sort_gaussians by per-Gaussian ones. */
int gb_bin_tiles_ranked(int G, const float* xys, const float* depths, const int32_t* radii, const float* conics,
                        const float* colors3, const float* opacity, const float* compensation, int img_h, int img_w,
                        int block_width, int64_t cap, int32_t* tile_bins, int32_t* tile_order, int tile_sched,
                        int32_t* ranks_sorted, float* rec_by_rank, int32_t* rank_to_gid, int32_t* n_out, int32_t* overflow,
                        void* workspace, void* colors_ready, void* stream);
/* Blend straight from the by-rank table (csrc/splat_blend_mom.cu, RANKED staging: 16-byte cp.async gathers by rank into
 * the stage ring instead of bulk copies of materialised sorted records).  Same results as gb_rasterize_packed_fwd/bwd;
 * final_idx indexes ranks_sorted.  channels 3 or 4; tile_order = launch order (gb_tile_order) or NULL. */
int gb_rasterize_ranked_fwd(int img_h, int img_w, int channels, const int32_t* tile_bins, const int32_t* tile_order,
                            const int32_t* ranks_sorted, const float* rec_by_rank, const float* background,
                            float* out_img, float* final_Ts, int32_t* final_idx, void* stream);
int gb_rasterize_ranked_bwd(int img_h, int img_w, int channels, const int32_t* rank_to_gid, const int32_t* ranks_sorted,
                            const int32_t* tile_bins, const int32_t* tile_order, const float* rec_by_rank,
                            const float* background, const float* final_Ts, const int32_t* final_idx,
                            const float* v_output, const float* v_output_alpha, float* v_xy, float* v_conic,
                            float* v_colors, float* v_opacity, void* stream);

/* launch order of the tiles, longest list first: order [T] int32 */
int gb_tile_order(int num_tiles, const int32_t* tile_bins, int32_t* order, void* stream);

/* blend formulation: 0 = CTA-synchronous double buffer (csrc/splat_blend_packed.cu), 1 = warp-decoupled mbarrier
 * pipeline (csrc/splat_blend_pipe.cu), 2 = the pipeline over an SM-affine tile schedule; environment
 * GOLIATH_B200_BLEND=batch|pipe|affine.  gb_rasterize_packed_fwd/bwd launch the CTA-synchronous kernels in mode 0 and
 * the pipeline otherwise; callers that build a schedule use gb_rasterize_sched_fwd/bwd in mode 2.  Outputs are
 * identical in every mode: pixels bit for bit, gradients to atomics order. */
int gb_get_blend_mode(void);
void gb_set_blend_mode(int mode);

/* SM-affine schedule of the tiles (one work queue per SM, near-equal sums of list lengths): sched holds
 * gb_tile_schedule_ints(num_tiles) int32; consumed by gb_rasterize_sched_fwd/bwd, which take the same arguments as
 * gb_rasterize_packed_fwd/bwd and give the same outputs. */
int gb_tile_schedule_ints(int num_tiles);
int gb_tile_schedule(int num_tiles, const int32_t* tile_bins, int32_t* sched, void* stream);
int gb_rasterize_sched_fwd(int img_h, int img_w, int channels, const int32_t* tile_bins, int32_t* sched,
                           const float* records, const float* background, float* out_img, float* final_Ts,
                           int32_t* final_idx, void* stream);
int gb_rasterize_sched_bwd(int img_h, int img_w, int channels, const int32_t* gids_sorted, const int32_t* tile_bins,
                           int32_t* sched, const float* records, const float* background, const float* final_Ts,
                           const int32_t* final_idx, const float* v_output, const float* v_output_alpha, float* v_xy,
                           float* v_conic, float* v_colors, float* v_opacity, void* stream);

/* blend forward over packed records streamed with cp.async.bulk; tile_order may be NULL */
int gb_rasterize_packed_fwd(int img_h, int img_w, int channels, const int32_t* tile_bins, const int32_t* tile_order,
                            const float* records, const float* background, float* out_img, float* final_Ts,
                            int32_t* final_idx, void* stream);

/* blend backward over packed records; gradients are accumulated into (caller zeroes them) */
int gb_rasterize_packed_bwd(int img_h, int img_w, int channels, const int32_t* gids_sorted,
                            const int32_t* tile_bins, const int32_t* tile_order, const float* records,
                            const float* background, const float* final_Ts, const int32_t* final_idx,
                            const float* v_output, const float* v_output_alpha, float* v_xy, float* v_conic,
                            float* v_colors, float* v_opacity, void* stream);

/* ---------------------------------------------------------------- utilslib (extensions/utils) */

/* replaces utilslib.compute_raydirs_forward — utils.cpp:46-82 (kernel utils_kernel.cu:11-51).
 * viewpos [N,3], viewrot [N,3,3], focal [N,2], princpt [N,2], pixelcoords [N,H,W,2] or NULL (integer grid),
 * outputs raypos/raydir [N,H,W,3], tminmax [N,H,W,2]. */
int gb_compute_raydirs_fwd(int N, int H, int W, const float* viewpos, const float* viewrot, const float* focal,
                           const float* princpt, const float* pixelcoords, float volradius, float* raypos,
                           float* raydir, float* tminmax, void* stream);
/* replaces utilslib.compute_raydirs_backward — utils.cpp:84-132: the reference kernel is an empty stub. */
int gb_compute_raydirs_bwd(void);

/* ---------------------------------------------------------------- mvpraymarchlib (extensions/mvpraymarch) */

/* replaces mvpraymarchlib.compute_aabb — mvpraymarch.cpp (compute_aabb) -> bvh.cu:157-201,249-294.
 * Tree arrays as built by mvpraymarch.py:44-82; nodeaabb [N,2K-1,2,3] out; workspace of
 * gb_mvp_aabb_workspace_bytes(N,K) bytes replaces the reference's per-call cudaMalloc. */
size_t gb_mvp_aabb_workspace_bytes(int N, int K);
int gb_mvp_compute_aabb(int N, int K, const float* primpos, const float* primrot, const float* primscale,
                        const int32_t* sortedobjid, const int32_t* nodechildren, const int32_t* nodeparent,
                        float* nodeaabb, void* workspace, void* stream);

/* march formulation for algo 0 without the shadow splat: bit 0 / bit 1 = lane-compacted sampling queue in the forward /
 * backward march (inside-the-box (ray, primitive) pairs are enqueued, sampled 32 at a time with every lane busy, applied in
 * the original order); default 2: the backward only (measured: backward 9.9 -> 8.3 ms at config 4, forward slower
 * with the queue).  GOLIATH_B200_RAYMARCH=legacy|queue-fwd|queue-bwd|queue. */
int gb_get_raymarch_mode(void);
void gb_set_raymarch_mode(int mode);

/* replaces mvpraymarchlib.raymarch_forward — mvpraymarch.cpp:179-283 -> mvpraymarch_kernel.cu:41-130.
 * template [N,K,TD,TH,TW,4] channels-last; warp [N,K,WD,WH,WW,3] or NULL (algo 0); rayrgba [N,H,W,4] out;
 * raysat [N,H,W,3] out or NULL; shadow [N,K,TD,TH,TW,2] accumulated or NULL.  The arguments the reference
 * accepts and ignores (sortboxes, maxhitboxes, synchitboxes, chlast, accum, termthresh, griddim, SURVEY.md §0.9)
 * are handled by the Python binding and are not part of the ABI. */
int gb_mvp_raymarch_fwd(int N, int H, int W, int K, const float* raypos, const float* raydir, float stepsize,
                        const float* tminmax, const float* nodeaabb, const float* primpos, const float* primrot,
                        const float* primscale, int TD, int TH, int TW, const float* tplate, int WD, int WH, int WW,
                        const float* warp, float* rayrgba, float* raysat, float* shadow, int algo, float fadescale,
                        float fadeexp, int blocksizex, int blocksizey, void* stream);

/* replaces mvpraymarchlib.raymarch_backward — mvpraymarch.cpp:285-399 -> mvpraymarch_kernel.cu:132-221.
 * Gradient buffers are accumulated into (the caller zero-fills them, mvpraymarch.py:256-263). */
int gb_mvp_raymarch_bwd(int N, int H, int W, int K, const float* raypos, const float* raydir, float stepsize,
                        const float* tminmax, const float* nodeaabb, const float* primpos, const float* primrot,
                        const float* primscale, int TD, int TH, int TW, const float* tplate, int WD, int WH, int WW,
                        const float* warp, const float* raysat, const float* grad_rayrgba, float* grad_primpos,
                        float* grad_primrot, float* grad_primscale, float* grad_tplate, float* grad_warp, int algo,
                        float fadescale, float fadeexp, int blocksizex, int blocksizey, void* stream);

/* ---------------------------------------------------------------- RGCA decoder heads (row R2) */

/* replaces the eager PyTorch block ca_code/models/rgca.py:506-546 (Gaussian heads, SH diffuse, reflection
 * direction); there is no native boundary in the reference, the Python mirror is goliath_b200.rgca_heads.
 * f_vnocond [B,125,G], f_vcond [B,4,G], postex / tn [B,3,G] planes (G = H*W), albedo [G,3], light_sh [B,3,81],
 * campos [B,3].  Outputs [B,G,3] except primqvec [B,G,4] and opacity / sigma / spec_vis [B,G]; shsum [B,G,3] is
 * saved for the backward. */
int gb_rgca_heads_fwd(int B, int G, const float* f_vnocond, const float* f_vcond, const float* postex, const float* tn,
                      const float* albedo, const float* light_sh, const float* campos, float scale_lo, float scale_hi,
                      float* primpos, float* primqvec, float* primscale, float* primscale_preclip, float* opacity,
                      float* sigma, float* spec_vis, float* spec_dnml, float* spec_nml, float* diff_color,
                      float* ref_dirs, float* primnmlbase, float* shsum, const float* light_sh2, float* shsum2,
                      void* stream);
/* light_sh2 [B,3,81] / shsum2 [B,G,3] (both NULL or both set): a second light-SH table evaluated in the same pass over the
 * 113 diffuse planes — the training-mode random back light `diff_color_rand` of rgca.py:590-616 (no albedo, unclamped). */

/* backward of the above; upstream gradients may be NULL; g_albedo is [B,G,3] (summed over B by the caller);
 * light_sh2 / g_shsum2: the second table and the upstream gradient of shsum2 (both NULL when unused). */
int gb_rgca_heads_bwd(int B, int G, const float* f_vnocond, const float* f_vcond, const float* postex, const float* tn,
                      const float* albedo, const float* light_sh, const float* campos, float scale_lo, float scale_hi,
                      const float* shsum, const float* g_primpos, const float* g_primqvec, const float* g_primscale,
                      const float* g_primscale_preclip, const float* g_opacity, const float* g_sigma,
                      const float* g_spec_vis, const float* g_spec_dnml, const float* g_spec_nml,
                      const float* g_diff_color, const float* g_ref_dirs, const float* g_primnmlbase, float* g_f_vnocond,
                      float* g_f_vcond, float* g_postex, float* g_tn, float* g_albedo, const float* light_sh2,
                      const float* g_shsum2, void* stream);

/* ---------------------------------------------------------------- mesh front end of the decoders (section 8f-4) */

/* replaces vert_normals (ca_code/utils/geom.py:327-346): v [B,V,3], vi [F,3] -> vn [B,V,3]; acc [B,V,3] = scratch
 * zero-filled by the caller (sum of the unit face normals per vertex), kept for the backward. */
int gb_vert_normals_fwd(int B, int V, int F, const float* v, const int32_t* vi, float eps, float* acc, float* vn, void* stream);
/* g_vn -> g_v [B,V,3] (zero-filled by the caller, accumulated); g_acc [B,V,3] scratch. */
int gb_vert_normals_bwd(int B, int V, int F, const float* v, const int32_t* vi, float eps, const float* acc, const float* g_vn,
                        float* g_acc, float* g_v, void* stream);
/* replaces values_to_uv (ca_code/utils/geom.py:308-324, GeometryModule.to_uv): values [B,V,C], index [T,3] int32 (-1 =
 * uncovered), bary [T,3] -> out [B,C,T] with T = uv_size^2. */
int gb_values_to_uv_fwd(int B, int V, int C, int64_t T, const float* values, const int32_t* index, const float* bary, float* out,
                        void* stream);
/* g_out [B,C,T] -> g_values [B,V,C] (zero-filled by the caller, accumulated). */
int gb_values_to_uv_bwd(int B, int V, int C, int64_t T, const int32_t* index, const float* bary, const float* g_out,
                        float* g_values, void* stream);

/* ---------------------------------------------------------------- gradient hygiene + clip + Adam (section 8f-3) */

/* replaces ca_code/utils/train.py:209-215 around the optimizer of config/*.yml (torch.optim.Adam / AdamW): zero the NaN /
 * Inf gradient entries, clip_grad_norm_(params, max_norm), optimizer.step().  rows: device array of 56-byte records
 * {float* p, g, m, v; int64 numel; float lr, wd; int32 missed, pad} (g == NULL: parameter skipped; missed = steps it sat out); chunks: device (tensor, chunk) int32
 * pairs covering every tensor in steps of gb_optim_chunk_elems() elements. */
int gb_optim_chunk_elems(void);
int gb_optim_row_bytes(void);
/* non-finite gradient entries -> 0 in place; *sqnorm (device fp64, zero-filled by the caller) += sum of squares. */
int gb_grad_sanitize_sqnorm(const void* rows, const int32_t* chunks, int n_chunks, double* sqnorm, void* stream);
/* Adam (adamw = 0, L2 weight decay) or AdamW (adamw = 1) step; gradients scaled by clamp(max_norm / (sqrt(*sqnorm) + 1e-6),
 * max = 1) when sqnorm != NULL and max_norm > 0; bias corrections 1 - beta^(step - row.missed); write_grads = 1 stores the clipped
 * gradients back (what clip_grad_norm_ leaves in p.grad). */
int gb_adam_step(const void* rows, const int32_t* chunks, int n_chunks, const double* sqnorm, float max_norm, float beta1,
                 float beta2, float eps, int step, int adamw, int write_grads, void* stream);

/* ---------------------------------------------------------------- post-render chain + photometric losses (section 8f-2) */

/* replaces CalV5.forward (ca_code/nn/color_cal.py:211-241), the background composite of rgca.AutoEncoder.forward
 * (ca_code/models/rgca.py:226-230) and LearnableBlur.forward (ca_code/nn/dof_cal.py:44-56; torchvision gaussian_blur 3x3 /
 * 7x7, reflect padding): pred = blur(cal(rgb) + (1 - alpha) * bg).  rgb / bg / pred [B,3,H,W], alpha [B,1,H,W], cal_w / cal_b /
 * blur_w [B,3] (blur_w = softmax-ed weights), grey [B] int32.  Stages with NULL tensors are skipped. */
int gb_post_render_fwd(int B, int H, int W, const float* rgb, const float* alpha, const float* bg, const float* cal_w,
                       const float* cal_b, const int32_t* grey, const float* blur_w, float* pred, void* stream);
/* g_pred -> g_rgb (overwritten); g_cal_w / g_cal_b / g_blur_w [B,3] accumulated (zero-filled by the caller, may be NULL). */
int gb_post_render_bwd(int B, int H, int W, const float* rgb, const float* alpha, const float* bg, const float* cal_w,
                       const float* cal_b, const int32_t* grey, const float* blur_w, const float* g_pred, float* g_rgb,
                       float* g_cal_w, float* g_cal_b, float* g_blur_w, void* stream);
/* replaces rgb_l1 and rgb_ssim (ca_code/loss/__init__.py:391-410, 479-494 over ca_code/utils/ssim.py:25-63): sums [3] fp64
 * (zero-filled by the caller) = sum |(pred - target) * mask|, sum ssim_map * mask, sum of the mask over 3 channels;
 * d_mu / d_pp / d_tp [B,3,H,W] are kept for the backward. */
int gb_ssim_l1_fwd(int B, int H, int W, const float* pred, const float* target, const float* mask, float* d_mu, float* d_pp,
                   float* d_tp, double* sums, void* stream);
/* gradient of l1_weight * rgb_l1 + ssim_weight * rgb_ssim w.r.t. pred, times *g_loss (device scalar, NULL = 1). */
int gb_ssim_l1_bwd(int B, int H, int W, const float* pred, const float* target, const float* mask, const float* d_mu,
                   const float* d_pp, const float* d_tp, const double* sums, const float* g_loss, float l1_weight,
                   float ssim_weight, float* g_pred, void* stream);

/* replaces the environment-map specular branch of rgca.PrimDecoder.forward (ca_code/models/rgca.py:548-556):
 * einsum("bxy,bny->bnx", lightrot, ref_dirs) -> dir2uv (ca_code/utils/envmap.py:284-292) -> mipmap_grid_sample of the
 * pre-convolved pyramid at level sigma * level_scale (ca_code/utils/mipmap_sampler.py:13-66: bilinear, border padding,
 * align_corners=False, two adjacent levels blended by the fractional level) -> clamp(max=1) * spec_vis.
 * levels: q (1..8) device pointers to [B,3,H_l,W_l] fp32 (the array itself in HOST memory); level_hw: q (H, W) pairs
 * (host).  ref_dirs [B,G,3], sigma [B,G], spec_vis [B,G], lightrot [B,3,3] -> spec [B,G,3]. */
int gb_envmap_spec_fwd(int B, int G, int q, const float* const* levels, const int32_t* level_hw, const float* ref_dirs,
                       const float* sigma, const float* spec_vis, const float* lightrot, float level_scale, float* spec,
                       void* stream);
/* g_spec [B,G,3] -> g_ref_dirs [B,G,3], g_spec_vis [B,G] (overwritten); no gradient for sigma (the level is picked
 * under no_grad upstream) nor for the environment map. */
int gb_envmap_spec_bwd(int B, int G, int q, const float* const* levels, const int32_t* level_hw, const float* ref_dirs,
                       const float* sigma, const float* spec_vis, const float* lightrot, float level_scale,
                       const float* g_spec, float* g_ref_dirs, float* g_spec_vis, void* stream);

/* replaces the per-view post-processing of rgca.AutoEncoder.render (ca_code/models/rgca.py:136-151, with
 * render_gsplat.py:79-108): colour HWC -> CHW, alpha = 1 - final_T (detached), depth / alpha.clamp(0.05, 1).
 * out4 [H,W,4] = rgb + depth-as-colour, alpha [H,W] -> rgb [3,H,W], alpha_img [1,H,W], depth [1,H,W]. */
int gb_render_finish_fwd(int img_h, int img_w, const float* out4, const float* alpha, float* rgb, float* alpha_img,
                         float* depth, void* stream);
/* g_rgb / g_depth may be NULL; g_out4 [H,W,4] is written. */
int gb_render_finish_bwd(int img_h, int img_w, const float* alpha, const float* g_rgb, const float* g_depth,
                         float* g_out4, void* stream);

/* fused shade + compose: replaces F.normalize (extensions/sgutils/sgutils.py:74-75) + evaluate_gaussian + the colour
 * composition of ca_code/models/rgca.py:557-575 (`spec * spec_vis`, `diff.clamp(0) + spec`, `.clamp(0)`) with one kernel
 * each way.  lobe_dirs are the UN-normalised reflection directions [N,D,3]; diff_color [N,D,3], spec_vis [N,D];
 * color [N,D,3] out (its sign bit keeps the pre-clamp sign for the backward); spec_color [N,D,3] out or NULL. */
int gb_sg_shade_compose_fwd(const float* lobe_dirs, const float* lobe_sigmas, const float* light_values,
                            const float* light_pts, const float* prim_pts, const int32_t* n_lights,
                            const float* diff_color, const float* spec_vis, float* color, float* spec_color, int N,
                            int D, int L, int w_type, void* stream);
/* backward: color = the forward's output; g_spec_color may be NULL; g_dirs / g_sigmas / g_diff / g_vis are written,
 * g_light_values (nullable) is accumulated into (caller zeroes it). */
int gb_sg_shade_compose_bwd(const float* lobe_dirs, const float* lobe_sigmas, const float* light_values,
                            const float* light_pts, const float* prim_pts, const int32_t* n_lights,
                            const float* diff_color, const float* spec_vis, const float* color, const float* g_color,
                            const float* g_spec_color, float* g_dirs, float* g_sigmas, float* g_diff, float* g_vis,
                            float* g_light_values, int N, int D, int L, int w_type, void* stream);

/* ---------------------------------------------------------------- decoder layers (rows R1 / R8) */

/* replaces conv_transpose2d + untied-bias add (ca_code/nn/layers.py:380-396) + the LeakyReLU that follows it in
 * make_conv_trans (layers.py:27-47) for k=4, s=2, p=1, with the weight-norm scale folded in:
 * out = act(scale[co] * convT(x, v) + bias).  x [B,Cin,Hi,Wi], v [Cin,Cout,4,4], scale [Cout] = g / ||v||_F,
 * bias [Cout,2Hi,2Wi] or NULL, out [B,Cout,2Hi,2Wi]; apply_act != 0 applies LeakyReLU(slope). */
int gb_deconv4x4s2_wnub_fwd(int B, int Cin, int Cout, int Hi, int Wi, const float* x, const float* v,
                            const float* scale, const float* bias, float slope, int apply_act, float* out,
                            void* stream);

/* backward of the above (replaces the cuDNN backward-data / backward-filter calls autograd makes for
 * layers.py:380-396).  gz [B,Cout,2Hi,2Wi] scratch; g_bias [Cout,2Hi,2Wi] or NULL; gx [B,Cin,Hi,Wi] or NULL;
 * gw [Cin,Cout,4,4] = dL/d(effective weight), ACCUMULATED (caller zeroes it and applies the weight-norm chain rule). */
int gb_deconv4x4s2_wnub_bwd(int B, int Cin, int Cout, int Hi, int Wi, const float* x, const float* v,
                            const float* scale, const float* out, const float* gout, float slope, int apply_act,
                            float* gz, float* g_bias, float* gx, float* gw, void* stream);

/* ---- tensor-core (tcgen05 + TMA + TMEM) forward of the same layer, inference path; Cin_pad % 32 == 0,
 * Cout % 16 == 0, 16 <= Cout <= 256.  Activations are NHWC split into a tf32 "hi" part and the fp32 remainder "lo"
 * (3xTF32 accumulation keeps the 1e-4 bar).  Same reference lines as gb_deconv4x4s2_wnub_fwd.
 * v may be NULL when w_scratch still holds the matrices prepared by an earlier call with the same weight_v
 * (inference with frozen parameters). */
size_t gb_deconv_tc_weight_bytes(int Cin_pad, int Cout);
int gb_nchw_to_nhwc_split(int B, int C, int Cpad, int H, int W, const float* x, float* hi, float* lo, void* stream);
int gb_deconv4x4s2_tc_fwd(int B, int Cin, int Cin_pad, int Cout, int Hi, int Wi, const float* x_hi, const float* x_lo,
                          const float* v, float* w_scratch, const float* scale, const float* bias, float slope,
                          int apply_act, float* out_hi, float* out_lo, int ldc, float* out_nchw, void* stream);

/* ---------------------------------------------------------------- hand-MVP decoders (row R8) */

/* replaces conv2d + bias add (+ LeakyReLU) of la.Conv2dWNUB / Conv2dWN (ca_code/nn/layers.py:276-327,468-472;
 * users: hand_mvp.py:297-321 TransDecoder, hand_mvp.py:269-294 PoseEncoder via blocks.py:232-280 ConvBlock), stride 1,
 * K = 1 or 3, padding (K-1)/2, with the weight-norm scale folded in: out = act(scale[co] * conv(x, v) + bias).
 * x [B,Cin,H,W], v [Cout,Cin,K,K], scale [Cout] = g / ||v||_F; bias_mode 0 none, 1 tied [Cout], 2 untied [Cout,H,W]. */
int gb_conv2d_wnub_fwd(int B, int Cin, int Cout, int H, int W, int K, const float* x, const float* v, const float* scale,
                       const float* bias, int bias_mode, float slope, int apply_act, float* out, void* stream);

/* backward of the above.  gz [B,Cout,H,W] scratch; g_bias: [Cout,H,W] written (mode 2) or [Cout] ACCUMULATED (mode 1,
 * caller zeroes) or NULL; gx [B,Cin,H,W] or NULL; gw [Cout,Cin,K,K] = dL/d(effective weight at unit scale),
 * ACCUMULATED (caller zeroes it and applies the weight-norm chain rule). */
int gb_conv2d_wnub_bwd(int B, int Cin, int Cout, int H, int W, int K, const float* x, const float* v, const float* scale,
                       const float* out, const float* gout, float slope, int apply_act, int bias_mode, float* gz,
                       float* g_bias, float* gx, float* gw, void* stream);

/* replaces the slab -> primitive-template sequence: relu(25*rgb+100) (hand_mvp.py:472), relu(alpha) (:434),
 * cat/view/permute/reshape (hand_mvp.py:172-185) and the valid-primitive gather (ca_code/utils/render_raymarcher.py:44-46)
 * with one pass.  rgb [B,PZ,3,U,U], alpha [B,PZ,1,U,U]; prim_slot [(U/PSY)*(U/PSX)] i32 (slot of a primitive in the
 * output, -1 = dropped) or NULL; tpl [B,Kout,PZ,PSY,PSX,4].  rgb_mul/rgb_add/apply_relu carry the output activation
 * (1, 0, 0 for a plain re-layout of already-activated slabs). */
int gb_mvp_slab_to_prims_fwd(int B, int PZ, int U, int PSX, int PSY, int Kout, const float* rgb, const float* alpha,
                             const int* prim_slot, float rgb_mul, float rgb_add, int apply_relu, float* tpl,
                             void* stream);
int gb_mvp_slab_to_prims_bwd(int B, int PZ, int U, int PSX, int PSY, int Kout, const float* rgb, const float* alpha,
                             const int* prim_slot, float rgb_mul, float rgb_add, int apply_relu, const float* g_tpl,
                             float* g_rgb, float* g_alpha, void* stream);

/* replaces TransDecoder's head scaling (hand_mvp.py:317-321) + GeomDecoder's transform composition
 * (hand_mvp.py:410-425, axisangle_to_matrix :477-510).  dec [B,9,K] (dec0 output viewed [B,9,64*64]);
 * posbase [B,K,3], rotbase [B,K,3,3]; zero_delta = the `iteration < primposstart` warm start (:412-415). */
int gb_mvp_prim_transform_fwd(int B, int K, const float* dec, const float* posbase, const float* rotbase,
                              float prim_scale, int zero_delta, float* primpos, float* primrot, float* primscale,
                              void* stream);
int gb_mvp_prim_transform_bwd(int B, int K, const float* dec, const float* posbase, const float* rotbase,
                              float prim_scale, int zero_delta, const float* g_primpos, const float* g_primrot,
                              const float* g_primscale, float* g_dec, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GOLIATH_B200_H_ */
