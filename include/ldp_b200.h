/*
 * ldp_b200.h -- C ABI of the B200-native post-matching densification hot path.
 *
 * The reference plugin (shadygm/Lichtfeld-Densification-Plugin v0.8.3) has NO FFI / operator ABI for
 * this path: it is a private Python function,
 *     core.pipeline._triangulate_ref(matched_ref, tri_ctx, collect_debug_matches)   core/pipeline.py:602-606
 * called once per reference view from run_dense_pipeline (core/pipeline.py:842-898).  This header is
 * therefore the boundary a maintainer would bind with ctypes (see INTEGRATION.md); every entry point
 * cites the reference code it replaces.  Plain pointers and sizes only; the caller (PyTorch on the
 * host side) owns every buffer; calls are stream-ordered and never synchronise unless stated.
 *
 * All functions return LDP_OK (0) or a negative ldp_error.  Per-reference outcomes that the
 * reference handles by *skipping the view* (core/pipeline.py:650-651,874-879) are reported in
 * ldp_outputs.status[r], not as call failures.
 */
#ifndef LDP_B200_H
#define LDP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LDP_ABI_VERSION 16
#define LDP_MAX_NN 16          /* neighbours per reference view (the panel clamps to 10) */
#define LDP_MAX_BINS 4096      /* coverage tiles per map: ceil(W/tile)*ceil(H/tile), tile = max(1, W/24) */

typedef enum ldp_error {
    LDP_OK = 0,
    LDP_ERR_INVALID = -1,      /* bad argument / unsupported shape */
    LDP_ERR_CUDA = -2,         /* a CUDA runtime call failed; see ldp_last_error_string() */
    LDP_ERR_WORKSPACE = -3,    /* workspace too small */
    LDP_ERR_NO_DEVICE = -4     /* no sm_100 device */
} ldp_error;

/* status[r]: why a reference view produced no samples (the reference returns None / raises and the
 * caller skips the view).  Bit flags >= 0x100 are informational and accompany LDP_REF_OK. */
typedef enum ldp_ref_status {
    LDP_REF_OK = 0,
    LDP_REF_EMPTY = 1,           /* weight sum s <= 0          -> core/sampling.py:27-28, pipeline.py:650-651 */
    LDP_REF_FEWER_NONZERO = 2,   /* np.random.choice ValueError "Fewer non-zero entries in p than size" */
    LDP_REF_BAD_WEIGHTS = 3,     /* NaN / negative probabilities -> ValueError in np.random.choice */
    LDP_REF_PSUM = 4,            /* "probabilities do not sum to 1" (only with a bad weight_sum_override) */
    LDP_REF_UNIFORMS_EXHAUSTED = 5, /* explicit uniform stream too short */
    LDP_REF_ROUNDS_EXCEEDED = 6,
    LDP_REF_NO_NEIGHBOURS = 7,
    LDP_REF_INEXACT_SCAN = 0x100 /* flag: f64 prefix sums not provably exact (tiny weights): sampled set is
                                    numpy's up to draws within ~1e-16 of a cdf step (DESIGN.md) */
} ldp_ref_status;

typedef enum ldp_rng_mode {
    LDP_RNG_PHILOX = 0,     /* production: Philox4x32-10, key = seed, stream = rng_stream[r], counter = draw index */
    LDP_RNG_EXPLICIT = 1    /* parity: uniforms[r*uniforms_per_ref + i] is the i-th double numpy's legacy
                               RandomState.random_sample would have produced (np.random.choice, core/sampling.py:32) */
} ldp_rng_mode;

/* Problem shape + the scalars of DensePipelineConfig (core/config.py:7-26) and _TriangulationContext
 * (core/pipeline.py:99-105) that the path reads. */
typedef struct ldp_params {
    int32_t n_refs;            /* reference views in this launch */
    int32_t H, W;              /* warp / certainty map resolution */
    int32_t w_match, h_match;  /* matcher resolution W_lr, H_lr (core/matcher.py:93-94) */
    int32_t matches_per_ref;   /* M */
    int32_t border;            /* 2   core/pipeline.py:646 */
    int32_t tiles;             /* 24  core/pipeline.py:647 */
    float sample_cap;          /* f32(0.9) core/matcher.py:92 */
    float reproj_thresh;       /* f32(config.reproj_thresh): compared in f32, core/pipeline.py:745 */
    float min_parallax_deg;    /* f32; <= 0 disables, core/pipeline.py:748 */
    double sampson_thresh;     /* f64; <= 0 disables, core/pipeline.py:708 */
    int32_t no_filter;         /* core/sampling.py:15-21 + core/pipeline.py:739-743 */
    int32_t collect_debug;     /* core/pipeline.py:761-769 */
    int32_t rng_mode;          /* ldp_rng_mode */
    int32_t scalar_loads;      /* 1: certainty planes are not 16-byte aligned -> scalar load path */
    int32_t nn_max;            /* largest ldp_ref_desc.nn of the launch (0 = unknown): selects the unrolled stream kernel */
    int32_t prologue;          /* 1: the certainty planes are RAW matcher outputs; the kernels apply the reference's
                                  post-processing on the fly (core/pipeline.py:405-430): clamp(min = certainty_floor),
                                  x mask_a (nearest-resized to the map), x mask_b[k] sampled at the warp's (xB, yB)
                                  (nearest, zeros outside, align_corners = False).  0: planes are already processed */
    float certainty_floor;     /* f32(config.certainty_thresh), core/pipeline.py:407; read only if prologue */
    int32_t no_warped_masks;   /* prologue only.  1: the caller guarantees that every ldp_ref_desc.mask_b[k] of the launch is NULL
                                  (no neighbour masks to sample through the warp): the first kernel's instantiation that reads
                                  no warp row runs, with the plain kernel's registers and occupancy (and the experimental fused
                                  front kernel may take raw planes); 0: unknown -- the instantiation that reads the warp planes */
    uint64_t seed;             /* Philox key */
    int64_t uniforms_per_ref;  /* explicit mode: doubles available per reference view */
    int32_t sm_reserve;        /* SMs the one-CTA-per-SM first draw kernel leaves to kernels of OTHER launches in flight on other
                                  streams (engine.DensifyRing passes 16) or to a collective; 0 = take every SM; -1 = the
                                  process-wide default of ldp_set_sm_reserve.  Per call: no shared state between engines */
    int32_t lens;              /* 1: some camera of the launch has a lens model (ldp_ref_desc.lens_a / lens_b[k] not PINHOLE): the geometry
                                  kernels' lens instantiation runs.  0: the caller guarantees that every camera is pinhole; the lens
                                  fields of the descriptors are not read */
    int32_t multiview;         /* 1: multi-view refinement of the kept points (see below); needs no_filter = 0 */
    float multiview_min_cert;  /* multiview: a neighbour's certainty at the sample must be >= this to join, in (0, 1] */
} ldp_params;

/* Multi-view refinement (ldp_params.multiview = 1).  Not in the reference, which triangulates every sampled pixel from the
 * reference view and its winning neighbour k alone.  It changes WHERE a kept point is, never WHICH points are kept:
 *   1. The two-view evaluation (Sampson gate, DLT, reprojection, cheirality, parallax against k) runs unchanged and decides
 *      keep, group, colour and the debug match.  A sample that is not kept is finished.
 *   2. Candidates of a kept sample: every neighbour slot q with group[q] == q (a uid listed twice counts once),
 *      group[q] != group[k], certainty at the pixel >= f32(multiview_min_cert) (after post-processing: with raw planes the
 *      floor and the masks apply), a finite ideal pixel, and, when sampson_thresh > 0, Sampson(F[q]) < sampson_thresh
 *      (the two-view gate's f64 decision).  Pixels are decoded and undistorted as in the two-view path; the reference
 *      pixel is the winner's.
 *   3. One DLT over the reference, the winner and all candidates: the two-view path's f32 rows, two per view, summed into
 *      the f64 Gram matrix A^T A and solved by the same null-vector code (inverse iteration; Jacobi in the fix-up).
 *   4. Trim once: every candidate whose reprojection error (lens-aware) is > reproj_thresh, or whose depth is <= 0, is
 *      dropped; the winner never is.  If something was dropped and a candidate is left, the DLT is solved again; if none is
 *      left, the two-view point stands.
 *   5. The refined point is accepted if in EVERY included view (reference and winner too) its error is <= reproj_thresh and
 *      its depth > 0, and the reference-winner parallax test passes; otherwise the two-view point stands.
 *   6. xyz = the accepted point, err = the largest error over the included views, view_mask[point] = bit q for every
 *      neighbour slot that contributed (the winner's bit always).  A solve that does not converge is redone by the fix-up
 *      with Jacobi; a converged two-view verdict is never re-evaluated.
 * sel_idx, sample_flags, group_order, group_count, ref_offset, rgb, the debug outputs and the sample_xyzerr taps (two-view
 * values) are those of the same launch without multiview; so are xyz and err of every point whose mask is the winner's
 * bit alone.  ldp_workspace_bytes grows by 20 bytes per sample slot when multiview is set. */

/* Lens model of a camera (COLMAP's models map onto two families; see CameraRecord.from_colmap).  Pixel coordinates are
 * normalised with the record's f32 intrinsics, x = (u - cx) / fx, y = (v - cy) / fy, in f64; with r^2 = x^2 + y^2:
 *   LDP_LENS_OPENCV   k = {k1, k2, p1, p2, k3, k4, k5, k6} (cv2.projectPoints order):
 *                       radial = (1 + k1 r^2 + k2 r^4 + k3 r^6) / (1 + k4 r^2 + k5 r^4 + k6 r^6)
 *                       x_d = x radial + 2 p1 x y + p2 (r^2 + 2 x^2),  y_d = y radial + p1 (r^2 + 2 y^2) + 2 p2 x y
 *   LDP_LENS_FISHEYE  k = {k1, k2, k3, k4, 0...} (cv2.fisheye): theta = atan(r),
 *                       theta_d = theta (1 + k1 theta^2 + k2 theta^4 + k3 theta^6 + k4 theta^8), (x_d, y_d) = theta_d / r (x, y)
 * The observed (distorted) pixels are undistorted by Newton's method in f64 (ldp_undistort_points); a point with no valid
 * inverse (no convergence, non-positive Jacobian determinant: past the fold of the polynomial; fisheye theta outside
 * [0, pi/2)) becomes NaN and its sample is dropped. */
typedef enum ldp_lens_model {
    LDP_LENS_PINHOLE = 0,
    LDP_LENS_OPENCV = 1,
    LDP_LENS_FISHEYE = 2
} ldp_lens_model;

typedef struct ldp_lens {
    int32_t model;             /* ldp_lens_model */
    float fx, fy, cx, cy;      /* the record's f32 K[0,0], K[1,1], K[0,2], K[1,2] (the K that built P and F) */
    int32_t pad;
    double k[8];               /* coefficients, unused ones zero */
} ldp_lens;

/* Per reference view: where its matcher outputs live and its camera constants.  Array of n_refs in
 * DEVICE memory.  Camera constants are computed on the host exactly like the reference does
 * (densify.py:226-230, core/geometry.py:122-130) and uploaded; the kernels stage them in shared memory. */
typedef struct ldp_ref_desc {
    const float* cert[LDP_MAX_NN];   /* [H*W] f32 per neighbour       (cert_list_cpu, core/pipeline.py:630) */
    const float* warp[LDP_MAX_NN];   /* [H*W*4] f32 per neighbour: xA,yA,xB,yB in [-1,1] (warp_list_cpu, :629);
                                        16-byte aligned; read only at sampled pixels */
    const uint8_t* image;            /* [img_h*img_w*3] u8 resized reference image (packed.imA_np, :611) */
    int32_t nn;                      /* neighbours present (len(nn_ids)) */
    int32_t img_w, img_h;
    uint32_t rng_stream;             /* Philox stream id (stable across sharding: global reference index) */
    float weight_sum_override;       /* > 0: use as the f32 normaliser s (core/sampling.py:26); else computed */
    float sxA, syA;                  /* f32(wA_cam / w_match), f32(hA_cam / h_match)     core/pipeline.py:681-682 */
    float sx_img, sy_img;            /* f32(img_w / w_match), f32(img_h / h_match)       core/pipeline.py:662-663 */
    float P1[12];                    /* reference camera P [3,4] row-major */
    float C1[3];
    float P2[LDP_MAX_NN][12];        /* neighbour cameras */
    float C2[LDP_MAX_NN][3];
    float F[LDP_MAX_NN][9];          /* fundamental_from_world2cam(ref, nbr), f32, row-major */
    float sxB[LDP_MAX_NN], syB[LDP_MAX_NN];   /* f32(wB_cam / w_match), ...   core/pipeline.py:697-699 */
    int32_t group[LDP_MAX_NN];       /* output group of neighbour k: smallest k' with nn_ids[k'] == nn_ids[k]
                                        (the reference groups by neighbour uid, core/pipeline.py:685-688) */
    /* read only when ldp_params.prologue is set; all masks of a view share one resolution */
    const uint8_t* mask_a;           /* [mask_h*mask_w] u8 reference-view mask or NULL (packed.maskA_np, core/pipeline.py:415-417) */
    const uint8_t* mask_b[LDP_MAX_NN]; /* per-neighbour mask or NULL (packed.nn_masks[k], core/pipeline.py:419-430) */
    int32_t mask_w, mask_h;
    float mask_sx, mask_sy;          /* f32(mask_w) / f32(W), f32(mask_h) / f32(H): F.interpolate(mode="nearest") source
                                        index = min(floor(dst * scale), size - 1) (core/pipeline.py:373-378) */
    /* read only when ldp_params.lens is set */
    ldp_lens lens_a;                 /* reference camera */
    ldp_lens lens_b[LDP_MAX_NN];     /* neighbour cameras */
} ldp_ref_desc;

/* Caller-allocated DEVICE outputs.  Optional pointers may be NULL. */
typedef struct ldp_outputs {
    /* packed point cloud, reference emission order (refs in launch order; inside a ref: neighbour groups in
       first-appearance order over the sample order, samples ascending inside a group; core/pipeline.py:685-780) */
    float* xyz;                /* [capacity,3] */
    float* rgb;                /* [capacity,3]  in [0,1] */
    float* err;                /* [capacity]    max reprojection error, px */
    int64_t capacity;          /* >= n_refs * ldp_sel_capacity(M) is always enough */
    int64_t* ref_offset;       /* [n_refs+1] exclusive prefix of kept points per reference view */
    int32_t* status;           /* [n_refs] ldp_ref_status */
    int32_t* n_samples;        /* [n_refs] S = |sel_idx| */
    int32_t* group_count;      /* [n_refs*LDP_MAX_NN] kept points per group id */
    int32_t* group_order;      /* [n_refs*LDP_MAX_NN] group ids in emission order, -1 padded */
    /* optional */
    float* dbg_matches;        /* [capacity,4] clipped match-res px (xA,yA,xB,yB)      core/pipeline.py:762-766 */
    float* dbg_cert;           /* [capacity]   clip(cert / cap, 0, 1)                  core/pipeline.py:767 */
    int32_t* sel_idx;          /* [n_refs*sel_capacity] sampled flat pixel indices (ascending; top-M order if no_filter) */
    uint8_t* sample_flags;     /* [n_refs*sel_capacity] bit0 keep, bit1 sampson-pass, bits 2.. = group id */
    float* sample_xyzerr;      /* [n_refs*sel_capacity*4] per-sample X,Y,Z,err before filtering (parity taps) */
    int32_t* uniforms_used;    /* [n_refs] doubles consumed from the stream */
    int32_t* rounds;           /* [n_refs] rejection rounds of the weighted draw */
    float* weight_sum;         /* [n_refs] the f32 normaliser s actually used */
    int32_t* view_mask;        /* [capacity] optional, multiview launches only (LDP_ERR_INVALID otherwise): per point, bit q set
                                  for every neighbour slot q whose match contributed to it; the winner's bit always */
} ldp_outputs;

/* ---- entry points ------------------------------------------------------------------------------- */

int ldp_abi_version(void);
const char* ldp_last_error_string(void);

/* Rows each reference view can emit at most: S <= max(M, int(0.85*M)+1), rounded up to 4. */
int64_t ldp_sel_capacity(int32_t matches_per_ref);

/* Bytes of device scratch ldp_densify_refs needs for this shape (n_refs, H, W, matches_per_ref are read). */
int ldp_workspace_bytes(const ldp_params* params, size_t* bytes_out);

/* The whole path for n_refs reference views: replaces the body of core.pipeline._triangulate_ref
 * (core/pipeline.py:632-780) and its callees select_samples_with_coverage (core/sampling.py:8-53),
 * sampson_error / dlt_triangulate_batch / reprojection_errors / cheirality_mask / parallax_mask
 * (core/geometry.py:58-141).  refs, uniforms (explicit mode; may be NULL otherwise), workspace and
 * every pointer inside *out are DEVICE pointers.  Enqueues on `stream` (a cudaStream_t) and returns. */
int ldp_densify_refs(const ldp_params* params, const ldp_ref_desc* refs, const double* uniforms,
                     const ldp_outputs* out, void* workspace, size_t workspace_bytes, void* stream);

/* Stage entry points (same kernels, exposed for stage-level parity tests and for callers that already
 * hold sample indices).  ldp_sample_refs = core/sampling.py:8-53 on the per-pixel best certainty
 * (core/pipeline.py:634-635,642-649); ldp_triangulate_samples = core/pipeline.py:652-780 on given indices
 * (out->sel_idx / out->n_samples are INPUTS here). */
int ldp_sample_refs(const ldp_params* params, const ldp_ref_desc* refs, const double* uniforms,
                    const ldp_outputs* out, void* workspace, size_t workspace_bytes, void* stream);
int ldp_triangulate_samples(const ldp_params* params, const ldp_ref_desc* refs,
                            const ldp_outputs* out, void* workspace, size_t workspace_bytes, void* stream);

/* The lens inversion the geometry kernels apply to the observed pixels, alone: uv_out[i] = the ideal pinhole pixel of the
 * distorted pixel uv_in[i] (f32 [n,2] DEVICE arrays; may alias), NaN where the lens has no valid inverse (see ldp_lens).
 * `lens` is a HOST pointer.  A PINHOLE lens copies the input.  For tests of the lens arithmetic and for integrators. */
int ldp_undistort_points(const ldp_lens* lens, int64_t n, const float* uv_in, float* uv_out, void* stream);

/* The certainty post-processing alone (core/pipeline.py:405-430), for callers that want the reference's
 * cert_list tensors and for stage-level parity tests: for every view r and neighbour k < nn,
 * out[r*ref_stride + k*plane_stride + i] = processed certainty of pixel i (strides in floats).  params->prologue is
 * ignored (the step is always applied); certainty_floor, H, W, n_refs are read. */
int ldp_postprocess_certainty(const ldp_params* params, const ldp_ref_desc* refs, float* out,
                              size_t ref_stride, size_t plane_stride, void* stream);

/* ---- output contract on the device (SURVEY 8a row a15, 8f row 2) ---------------------------------
 * The reference converts colours with to_uint8_rgb (core/image_utils.py:24-26: clip(round(rgb * 255), 0, 255), half to
 * even) and writes one struct.pack per point (core/writers.py:15-46).  These build the same bytes where the points are:
 * the caller copies the records to the host and writes header + records (byte-identical files).
 * xyz, rgb: [n,3] f32 device; err: [n] f32 device or NULL (zeros, like errors=None); n_dev: optional DEVICE pointer
 * to the actual point count (then n is an upper bound that sizes the launch and min(n, *n_dev) records are written:
 * no host synchronisation between the path and the packing); records_out: device, n * 15 / n * 43 bytes.
 *   ldp_pack_ply_records       per vertex  <fff xyz, BBB rgb                           core/writers.py:44-45
 *   ldp_pack_ply_normal_records  per vertex  <fff xyz, <fff normal, BBB rgb (27 bytes; not in the reference: the
 *                              PLY of core/writers.py write_ply(..., normals=), nx ny nz between z and red)
 *   ldp_pack_points3d_records  per point   <Q first_id + i, <ddd xyz, <BBB rgb, <d err  core/writers.py:23-26
 *                              (first_id = 1 for a whole file; a rank writing rows [a, b) passes a + 1)
 *   ldp_rgb_to_uint8           to_uint8_rgb on n_values floats                         core/image_utils.py:24-26
 *   ldp_gather_points          xyz[sel], rgb[sel], err[sel] for the int64 indices the point cap drew on the host
 *                              (densify.py:110-120, np.random.default_rng(seed).choice(n, m, replace=False));
 *                              negative indices wrap like numpy's; an index outside [-n, n) sets *bad_index_flag
 *                              (device int32, may be NULL) and leaves the row unwritten. */
int ldp_pack_ply_records(const float* xyz, const float* rgb, int64_t n, const int64_t* n_dev, uint8_t* records_out, void* stream);
int ldp_pack_ply_normal_records(const float* xyz, const float* rgb, const float* normals, int64_t n, const int64_t* n_dev,
                                uint8_t* records_out, void* stream);
int ldp_pack_points3d_records(const float* xyz, const float* rgb, const float* err, int64_t n, const int64_t* n_dev,
                              uint64_t first_id, uint8_t* records_out, void* stream);
int ldp_rgb_to_uint8(const float* rgb, int64_t n_values, uint8_t* out, void* stream);
int ldp_gather_points(const float* xyz, const float* rgb, const float* err, const int64_t* sel, int64_t m, int64_t n,
                      float* xyz_out, float* rgb_out, float* err_out, int32_t* bad_index_flag, void* stream);

/* out[i,:] = src[sel[i],:] for rows of row_floats f32 values: the debug preview's subsample of the kept matches [K,4]
 * and their normalised certainties [K] (core/pipeline.py:573-582; indices from default_rng(pair seed).choice on the host). */
int ldp_gather_rows(const float* src, int32_t row_floats, const int64_t* sel, int64_t m, int64_t n, float* out,
                    int32_t* bad_index_flag, void* stream);

/* Concatenation of packed point segments on the device: replaces the reference's final np.concatenate of the per-view arrays
 * (core/pipeline.py:914-928) for callers that keep several launches, or several ranks' all-gathered blocks, in device memory.
 * Segment q holds *count_src[q] points (a DEVICE int64, e.g. ldp_outputs.ref_offset + n_refs of a launch) at the start of
 * its padded arrays xyz_src[q] [seg_cap,3], rgb_src[q] [seg_cap,3], err_src[q] [seg_cap]; its rows are written to
 * xyz_out / rgb_out / err_out at row sum(count_src[0..q)).  The four pointer tables are DEVICE arrays of n_seg device
 * pointers.  seg_offset_out: optional device int64 [n_seg + 1], the exclusive prefix of the counts (last = total);
 * total_out: optional device int64, the total alone (e.g. the header of a buffer that goes into a collective).
 * No host synchronisation: the counts never leave the device. */
int ldp_concat_points(const float* const* xyz_src, const float* const* rgb_src, const float* const* err_src,
                      const int64_t* const* count_src, int32_t n_seg, int64_t seg_cap, float* xyz_out, float* rgb_out,
                      float* err_out, int64_t out_capacity, int64_t* seg_offset_out, int64_t* total_out, void* stream);

/* The all-gather of the ranks' clouds as a push over NVLink peer memory (no reference counterpart: the reference is one process;
 * replaces its final np.concatenate, core/pipeline.py:914-928, across ranks).  This rank's first *count_src[rank] rows of
 * xyz / rgb / err are written into EVERY destination p < world at row sum(count_src[0..rank)): xyz_dst[p], rgb_dst[p],
 * err_dst[p] are device arrays of `world` pointers (peer-mapped memory for p != rank); count_src[q] points at rank q's
 * count (peer-mapped).  seg_offset_out [world + 1] / total_out: optional LOCAL outputs (every rank's row offset, total).
 * The caller brackets the call with cross-rank barriers (all counts and clouds complete before; all pushes landed after). */
int ldp_scatter_points(const float* xyz, const float* rgb, const float* err, const int64_t* const* count_src, int32_t rank,
                       int32_t world, int64_t seg_cap, float* const* xyz_dst, float* const* rgb_dst, float* const* err_dst,
                       int64_t out_capacity, int64_t* seg_offset_out, int64_t* total_out, void* stream);

/* ---- pair generation on the device (SURVEY 8f row 3) ---------------------------------------------
 * flat_poses: [n,16] f32 device, the row-major 4x4 world-to-camera transforms (CameraRecord.flat_pose()).
 *   ldp_select_kcenters    core/selection.py:36-54 select_cameras_kcenters: normalise the columns (mean, std + 1e-8), start
 *                          from the row of largest norm, then k - 1 greedy farthest-point picks.  numpy's float32
 *                          operation order is mirrored, so the picks are numpy's.  scratch: [n,16] f32 device.
 *                          centers_sorted [k] = sorted(centers) (what the reference returns); centers_order [k] = pick order.
 *                          1 <= k <= n <= 8192 (the reference clamps k the same way before the loop).
 *   ldp_nearest_neighbors  core/selection.py:57-70 nearest_neighbors: for every view the k nearest other views by Euclidean
 *                          distance of the poses, ascending.  idx_out [n,k] int64.  k <= min(n - 1, 16).  The reference's
 *                          table index for index: the distances are torch.cdist's own float32 values (n <= 25: the direct
 *                          kernel's sequential sum of squared differences; above: |x|^2 + |y|^2 - 2 x.y
 *                          as ONE K = 18 dot product of float32 FMAs in index order, row norms as eight lanes added left to
 *                          right; measured against torch), so near-equal distances - the left / right neighbours of a ring
 *                          camera - come out in the reference's order; and EXACTLY equal float32 distances are ordered by
 *                          torch.topk's own CPU selection (std::partial_sort for k * 64 <= n, else std::nth_element +
 *                          std::sort over (value, index) pairs, libstdc++'s moves restated one for one). */
int ldp_select_kcenters(const float* flat_poses, int32_t n, int32_t k, float* scratch, int32_t* centers_sorted,
                        int32_t* centers_order, void* stream);
int ldp_nearest_neighbors(const float* flat_poses, int32_t n, int32_t k, int64_t* idx_out, void* stream);

/* ---- voxel-grid downsample (SURVEY 8f row 2) -------------------------------------------------------
 * densify.py:29-50 _voxel_downsample = Open3D's PointCloud::voxel_down_sample: voxel index
 * floor((p - (min_bound - voxel_size / 2)) / voxel_size) per axis in f64, every voxel replaced by the f64 mean (in point
 * order) of its points and colours, cast to f32; colours are divided by 255 first when their maximum exceeds 1
 * (densify.py:41-44).  PARITY UNPINNED: Open3D is not in the reference tree nor in this image; the algorithm is restated
 * from its published source.  Open3D emits voxels in std::unordered_map order; here in order of each voxel's first point.
 * xyz, rgb [n,3] f32 device; xyz_out, rgb_out [n,3] f32 device (first status_out[1] rows are written);
 * status_out: device int32[2] = {1 if a voxel index does not fit 21 bits per axis or a coordinate is NaN, voxel count}. */
int ldp_voxel_workspace_bytes(int64_t n, size_t* bytes_out);
int ldp_voxel_downsample(const float* xyz, const float* rgb, int64_t n, double voxel_size, float* xyz_out, float* rgb_out,
                         int32_t* status_out, void* workspace, size_t workspace_bytes, void* stream);

/* ---- statistical outlier removal ------------------------------------------------------------------------------------
 * Open3D's PointCloud::RemoveStatisticalOutliers(nb_neighbors, std_ratio), restated from its published source.  PARITY
 * UNPINNED: Open3D is not in the reference tree nor in this image.  Inputs: xyz [n,3] f32 device, k = nb_neighbors in
 * [1, 64], std_ratio > 0; k_eff = min(k, n).
 *   1. For every point i, the k_eff nearest points of the cloud, the point itself included (at distance 0), by
 *      d^2 = (dx*dx + dy*dy) + dz*dz in f64 with dx = f64(x_j) - f64(x_i), no FMA contraction; d = sqrt(d^2).
 *   2. m_i = (sum of those k_eff distances in ascending order, added sequentially in f64) / k_eff.
 *   3. V = n; mean = (sum over m_i > 0 of m_i) / V; Q = sum over m_i > 0 of (m_i - mean)^2; std = sqrt(Q / (V - 1));
 *      threshold = mean + std_ratio * std (no FMA).
 *   4. Point i is kept iff m_i > 0 && m_i < threshold; kept_idx_out lists the kept points in ascending index.
 * Open3D's quirks are kept: a point whose k nearest are all exact duplicates has m_i = 0 and is dropped (and left out of the
 * sums but not out of V); n = 1 gives std = NaN and keeps nothing; k = 1 keeps nothing.
 * Order of the two sums of step 3 (Open3D adds in index order; ours differs from it only for points within a few ulps of
 * the threshold): (a) partial p = sequential sum over points [256 p, 256 p + 256) in index order; (b) t = 0..1023: v_t =
 * sequential sum of partials t, t + 1024, t + 2048, ...; (c) for s = 512, 256, ..., 1: v_t = v_t + v_{t+s} for t < s; the
 * sum is v_0.  The terms of points with m_i <= 0 are skipped.  Nothing depends on the grid, the launch configuration or
 * the stream; m_i is exact (bit-identical to the rule) whatever the density: the k-NN search stops only on a conservative
 * bound (DESIGN.md §4.5).
 * kept_idx_out: int64 [n] device, the first status_out[1] entries are written; mean_dist_out: f64 [n] device (m_i) or NULL;
 * stats_out: f64 [3] device = {mean, std, threshold} or NULL; status_out: int32 [3] device = {1 if a coordinate is not
 * finite (then nothing else is written), kept count, points whose search left the finest grid}.  n = 0 zeroes status_out
 * and writes nothing else.  Synchronises the stream once (the finest cell size follows from a trial grid's cell count). */
int ldp_outlier_workspace_bytes(int64_t n, int32_t nb_neighbors, size_t* bytes_out);
int ldp_statistical_outliers(const float* xyz, int64_t n, int32_t nb_neighbors, double std_ratio,
                             int64_t* kept_idx_out, double* mean_dist_out, double* stats_out, int32_t* status_out,
                             void* workspace, size_t workspace_bytes, void* stream);
/* Test hook: R, the shells of cells searched per grid level before a point moves to the next coarser level (0 restores the
 * default, 2).  Results do not depend on it. */
int ldp_debug_outlier_max_shells(int shells);

/* ---- oriented point normals (not in the reference) ------------------------------------------------------------------
 * Inputs: xyz [n,3] f32 device, k in [3, 64]; k_eff = min(k, n).
 *   1. Neighbourhood of point i: the k_eff points j with the smallest (d^2, j), compared lexicographically, with d^2 the
 *      outlier rule's (dx*dx + dy*dy) + dz*dz in f64 without FMA and j the row index; i itself is a candidate at d^2 = 0.
 *      The index breaks ties, so the set is unique (on a lattice, tied neighbours would change the normal).
 *   2. In f64, over the neighbourhood in ascending (d^2, j) order, added sequentially, no FMA: mu = (sum x_j) / k_eff;
 *      C = (sum (x_j - mu)(x_j - mu)^T) / k_eff (upper triangle; each entry its own sequential sum).
 *   3. Eigenvalues l0 <= l1 <= l2 of C by cyclic Jacobi in f64 (to convergence).  The normal is the unit eigenvector of
 *      l0; curvature (surface variation) = l0 / ((l0 + l1) + l2).
 *   4. Undefined when k_eff < 3, trace(C) = 0 (all duplicates) or l1 <= 1e-12 * l2 (a line): normal (0, 0, 0),
 *      curvature NaN, counted in status_out[1].
 *   5. Sign: first canonical (the component of largest magnitude positive, the lowest axis on ties); then, when the point
 *      has a centre c, flipped iff n . (c - x) < 0, in f64.  A point triangulated from a camera faces that camera.
 * Steps 1 and 2 are bit-exact: the k-NN search stops only on a conservative bound (DESIGN.md §4.6); step 3 matches
 * numpy.linalg.eigh within eigenvector conditioning.  Parity with Open3D's estimate_normals is not claimed.
 * centers: f32 [n_centers,3] device or NULL (no orientation step); center_idx: int32 [n] device, the centre of every point,
 * or NULL for centers[0] (needs centers).  normals_out f32 [n,3] device; curvature_out f32 [n] device or NULL; knn_idx_out
 * int32 [n,k_eff] device or NULL (row i: the neighbourhood of step 1, ascending).  status_out: int32 [3] device = {bit mask:
 * 1 a coordinate is not finite (then nothing else is written), 2 a centre index is out of range (that point keeps its
 * canonical sign); undefined normals; points whose search left the finest grid}.  n = 0 zeroes status_out and writes
 * nothing else.  Synchronises the stream once (the trial grid, as ldp_statistical_outliers); ldp_debug_outlier_max_shells
 * applies.  Results do not depend on the grid, the launch or the stream. */
int ldp_normals_workspace_bytes(int64_t n, int32_t k, size_t* bytes_out);
int ldp_estimate_normals(const float* xyz, int64_t n, int32_t k, const float* centers, int32_t n_centers, const int32_t* center_idx,
                         float* normals_out, float* curvature_out, int32_t* knn_idx_out, int32_t* status_out, void* workspace,
                         size_t workspace_bytes, void* stream);

/* SMs the one-CTA-per-SM first draw kernel leaves free when ldp_params.sm_reserve is -1 (process-wide default, initially 0; the
 * environment variable LDP_SM_RESERVE, when set, wins over both).  With several launches in flight on different streams (engine.DensifyRing) or a
 * collective running beside the path, the free SMs let the other kernels make progress: measured 0.1445 -> 0.1420 ms per
 * step at 3 launches in flight with 16. */
int ldp_set_sm_reserve(int n_sms);

/* Kernel launches enqueued by the last ldp_* call on this thread (for bench.py's gpu_launches). */
int ldp_last_launch_count(void);

/* Per-kernel device timing of subsequent ldp_* calls on this thread (CUDA events recorded on the call's
 * stream around every kernel; no synchronisation at record time).  ldp_profile_read synchronises on the
 * last event and returns, for the LAST call, up to max_n kernel durations in ms in launch order
 * (stream, prep, draw | stream, topm; then geometry, pack); returns the number of kernels, or a negative ldp_error. */
int ldp_profile_enable(int on);
int ldp_profile_read(float* ms_out, int max_n);
const char* ldp_profile_name(int i);      /* name of the i-th kernel of the last profiled call */

/* Test hook: force the thread-block-cluster size of the draw kernel (CTAs per reference view, 1..8);
 * 0 restores the automatic choice.  Results do not depend on it. */
int ldp_debug_set_cluster(int csize);
int ldp_debug_last_cluster(void);          /* cluster size the last draw kernel was launched with */
/* Debug builds (-DLDP_PHASE_CLOCKS) only: copy the draw kernel's per-view phase timestamps [n_refs][32] (SM clocks)
 * to host memory; synchronises.  Release builds return zeros. */
int ldp_debug_read_clocks(const ldp_params* params, void* workspace, long long* host_out);
/* Test hooks for the fix-up worklist of the geometry kernels.  ldp_debug_force_fixup: in subsequent MULTIVIEW launches on any
 * thread (0, 0 restores the default), every sample i (position in its view's sample list) with i % two_view_every == 0 is sent
 * to the fix-up as if its two-view null-vector iteration had not converged, and every kept sample with i % multiview_every == 0
 * as if its multi-view solve had not converged (0 = never); the fix-up solves them with Jacobi.  The plain path's kernels do not
 * read it.  ldp_debug_read_fixups: after a launch (synchronises), host_out[0] = entries of the worklist, host_out[1] = those
 * that redo only a multi-view solve; params and workspace as given to that launch. */
int ldp_debug_force_fixup(int two_view_every, int multiview_every);
int ldp_debug_read_fixups(const ldp_params* params, void* workspace, int32_t* host_out);
/* Test hook: pipeline a launch over n sub-batches of views on internal streams (1..8; 0 restores the default, which is
 * one batch unless LDP_SUBBATCH is set).  Results do not depend on it. */
int ldp_debug_set_subbatches(int n);

/* Measurement hook: enqueue `reps` back-to-back launches of the path's first (dominant, HBM-bound) kernel alone on
 * `stream`, so that bench.py can time its average launch duration with two CUDA events instead of bracketing every
 * launch.  Writes only the scratch workspace. */
int ldp_debug_launch_stream(const ldp_params* params, const ldp_ref_desc* refs, void* workspace, size_t workspace_bytes,
                            void* stream, int reps);

/* sizeof() of the ABI structs as this library was compiled: which = 0 ldp_params, 1 ldp_ref_desc,
 * 2 ldp_outputs.  Bindings check these against their own struct definitions at load time. */
int64_t ldp_struct_size(int which);

#ifdef __cplusplus
}
#endif
#endif /* LDP_B200_H */
