/*
 * gsb200.h -- C ABI of libgsb200.so: the B200-native (sm_100a) replacement for the rasteriser
 * hot path of wanmeihuali/taichi_3d_gaussian_splatting.
 *
 * This header is the drop-in boundary.  Every entry point names the reference interface it
 * replaces (file:line relative to the reference repo; GPCR =
 * taichi_3d_gaussian_splatting/GaussianPointCloudRasterisation.py).
 *
 * Conventions
 *  - extern "C", plain pointers and sizes only; no C++/torch types cross the boundary.
 *  - All pointers in the *Args structs are DEVICE pointers unless the field name says "host".
 *  - The caller owns every buffer, including the workspace; the library allocates nothing
 *    persistent and keeps no global mutable state except a thread-local error string.
 *  - Every call enqueues work on the given cudaStream_t (passed as void*) and returns without
 *    synchronising, except the *_host entry points which return after the result is in host memory.
 *  - Return value: 0 on success, negative GSB_E* code on failure; gsb200_last_error() gives text.
 *  - dtypes are the reference's: f32 data, i32 indices, i8 masks (GPCR:31-45, 239-259, 318-343).
 */
#ifndef GSB200_H_
#define GSB200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSB200_VERSION 102 /* major*100 + minor */

#define GSB_TILE_WIDTH 16     /* GPCR:27 */
#define GSB_TILE_HEIGHT 16    /* GPCR:28 */
#define GSB_BOUNDARY_TILES 3  /* GPCR:26 */
#define GSB_FEATURE_DIM 56    /* GPCR:208-236: q(4) s(3) alpha(1) R/G/B SH(16 each) */
#define GSB_RECORD_FLOATS 12  /* packed per-splat record written by the preprocess kernel */
#define GSB_ACCUM_FLOATS 12   /* per-splat backward accumulator row */

enum {
    GSB_OK = 0,
    GSB_EINVAL = -1,     /* bad argument (null pointer, H/W not multiple of 16, ...) */
    GSB_ECUDA = -2,      /* a CUDA runtime call failed */
    GSB_EWORKSPACE = -3, /* workspace too small for (N, key_capacity, H, W) */
    GSB_EUNSUPPORTED = -4
};

/* flags */
#define GSB_FLAG_EXACT_EXP 1u    /* blend kernels use expf instead of ex2.approx */
#define GSB_FLAG_FORCE_KEY64 2u  /* always sort (tile<<32 | depth) 64-bit keys like GPCR:158-170 */
#define GSB_FLAG_KEEP_ALL_TILE_PAIRS 8u   /* emit a key for every tile of the reference's 3-sigma square (GPCR:81-172) instead of
                                            only those where the splat can reach alpha >= 1/255 on some pixel; outputs are
                                            identical either way, this only makes the sorted list equal to the reference's */
#define GSB_FLAG_Q_ALREADY_NORMALISED 4u /* forward only: take q as stored and do not rewrite it.  Used when a
                                            frame is re-run after a key-capacity overflow, so that the second
                                            pass is bit-identical to the first (normalising twice is not). */
#define GSB_FLAG_BACKWARD_TRANSPOSED 16u /* backward only: loop A accumulates per splat in registers after a shared-memory
                                            transposition (csrc/blend_bwd_transposed.cu; what the Python operator passes by
                                            default: 769 us at C3 on a B200) instead of a warp butterfly per (warp, splat)
                                            (csrc/blend_bwd.cu, 997 us; flag clear) */
#define GSB_FLAG_NO_HOOK_STATS 32u       /* backward only, opt-in: skip the statistics only a
                                            backward hook reads (|d/duv| magnitude, affected-pixel count, magnitude image) --
                                            the reference's need_extra_info = False, GPCR:521, 690-704.  accum[:, 9:11] and
                                            magnitude_grad_viewspace_on_image are then left untouched (the pointer must still be valid) */

#define GSB_POSE_MAX_OBJECTS 16          /* gsb200_backward_with_pose: most objects (pose rows) one call can differentiate */

#define GSB_FLAG_COMPACT_GRADS 64u        /* backward only (view-parallel training, parallel.py): the per-point kernel writes
                                            grad_sum_compact (N,12) and grad_color_compact (N,3) instead of the dense
                                            gradients; gsb200_expand_view_gradients rebuilds them after the exchange */

/* Byte offsets of the sub-buffers inside the caller-owned workspace blob.  Filled by
 * gsb200_workspace_layout(); the Python shim uses it to expose saved-for-backward tensors as views. */
typedef struct GsbWorkspaceLayout {
    int64_t total_bytes;
    int64_t zero_bytes;        /* [0, zero_bytes) is memset to 0 at the start of every forward */
    int64_t counters;          /* int64[8]: [0]=M in-frustum points, [1]=K (tile,splat) pairs emitted/needed,
                                  [2]=overflow (K > key_capacity), [4]=largest depth key int32(depth * scale) of the frame
                                  (low 32 bits): the sort only runs the passes its live bits need */
    int64_t tickets;           /* uint32[16] dynamic block tickets */
    int64_t scan_state;        /* uint64[scan_blocks+1] decoupled look-back state of the compaction scan (one word per 128-point CTA) */
    int64_t sort_hist;         /* uint32[8][1024] global digit histograms */
    int64_t sort_state;        /* uint32[passes][sort_blocks][2^radix_bits] onesweep look-back state */
    int64_t tile_start;        /* int32[T]  GPCR:952-957 tile_points_start */
    int64_t tile_end;          /* int32[T]  tile_points_end */
    int64_t poses;             /* float[num_objects][20]: T_camera_pointcloud 3x4, camera centre, pad */
    int64_t point_id;          /* int32[N]  point_id_in_camera_list (first M valid), GPCR:864 */
    int64_t point_offset;      /* int32[N]  inverse map: in-camera offset of point id, -1 if outside the frustum */
    int64_t num_tiles;         /* int32[N]  num_overlap_tiles, GPCR:904-911 */
    int64_t records;           /* float[N][12]: u v a b | c rescale opacity depth | r g b radius */
    int64_t point_in_camera;   /* float[N][3] GPCR:877 */
    int64_t keys_a, keys_b;    /* sort keys, key_bytes each, key_capacity_padded entries: a = as emitted (never written by
                                  the sort), b = sorted (whatever the number of radix passes that ran) */
    int64_t vals_a, vals_b;    /* int32 payload = in-camera offset, GPCR:930 */
    int64_t keys_c, vals_c;    /* scratch of the radix passes (third buffer of the a -> [c -> b ->] ... -> b rotation); after
                                  the sort the forward blend (unless rgb_only) reuses keys_c for one uint8 per sorted key: the
                                  mask of the 8x4-pixel patches of its tile that the splat can reach, read by the backward */
    int32_t key_bytes;         /* 4 or 8 */
    int32_t tile_bits, depth_bits, sort_passes;
    int64_t key_capacity_padded;
    int32_t sort_blocks, scan_blocks;
    int32_t radix_bits;        /* 8 or 10: digit width of the key sort */
    int32_t reserved;
} GsbWorkspaceLayout;

/* Inputs of GaussianPointCloudRasterisationInput (GPCR:788-804) + config (GPCR:776-786). */
typedef struct GsbForwardArgs {
    int64_t num_points;                 /* N */
    const float *pointcloud;            /* (N,3) */
    float *pointcloud_features;         /* (N,56); q of in-frustum rows normalised IN PLACE (GPCR:264-266) */
    const int8_t *point_invalid_mask;   /* (N) 1 = slot unused */
    const int32_t *point_object_id;     /* (N) */
    int32_t num_objects;
    const float *q_pointcloud_camera;   /* (num_objects,4) xyzw, camera->pointcloud */
    const float *t_pointcloud_camera;   /* (num_objects,3) */
    const float *camera_intrinsics;     /* (3,3) row-major, device */
    int32_t camera_height, camera_width;
    float near_plane, far_plane, depth_to_sort_key_scale;
    int32_t rgb_only;                   /* GPCR:781; aux outputs are left untouched when set */
    uint32_t flags;
    void *workspace;
    int64_t workspace_bytes;
    int64_t key_capacity;               /* capacity (entries) of the key/value buffers */
    float *rasterized_image;            /* (H,W,3) */
    float *rasterized_depth;            /* (H,W) */
    float *pixel_accumulated_alpha;     /* (H,W) */
    int32_t *pixel_offset_of_last_effective_point; /* (H,W) */
    int32_t *pixel_valid_point_count;   /* (H,W) */
    void *stream;
    /* Optional early read-back: if both are non-NULL, gsb200_forward copies counters[0..3] = {M, K, overflow, -}
     * to the PINNED HOST buffer right after the per-point stage and records the event (a cudaEvent_t) behind
     * the copy; the remaining stages are enqueued regardless.  The host can wait on the event (it fires after
     * ~the preprocess kernel, long before the frame ends), learn M and K and whether the key buffers overflowed,
     * and return to its caller with the rest of the frame still in flight. */
    int64_t *host_counters;
    void *host_counters_event;
} GsbForwardArgs;

typedef struct GsbBackwardArgs {
    int64_t num_points;
    const float *pointcloud;
    const float *pointcloud_features;   /* as left by forward (q normalised) */
    const int32_t *point_object_id;
    int32_t num_objects;
    const float *t_pointcloud_camera;   /* camera centre for the SH direction, GPCR:731-732 */
    const float *camera_intrinsics;
    int32_t camera_height, camera_width;
    float far_plane, depth_to_sort_key_scale; /* same values as the forward (fix the workspace layout) */
    int32_t color_max_sh_band;          /* GPCR:1167-1182; any value outside {0,1,2} clears nothing */
    float grad_q_factor, grad_s_factor, grad_alpha_factor, grad_color_factor,
        grad_high_order_color_factor;   /* GPCR:782-786, 1105-1125 */
    uint32_t flags;
    void *workspace;                    /* the SAME workspace the forward of this frame used */
    int64_t workspace_bytes;
    int64_t key_capacity;
    const float *grad_rasterized_image; /* (H,W,3) */
    const float *pixel_accumulated_alpha;
    const int32_t *pixel_offset_of_last_effective_point;
    float *accum;                       /* (>=M,12) zero-initialised by this call:
                                           guv.x guv.y gcov00 gcov01 gcov11 gr gg gb glogit magnitude n_pixels(as f32) pad */
    int64_t accum_rows;
    float *grad_pointcloud;             /* (N,3) fully written by the per-point kernel (zeros outside the frustum) */
    float *grad_pointcloud_features;    /* (N,56) fully written, band-masked and factor-scaled */
    float *magnitude_grad_viewspace_on_image; /* (H,W,2) */
    void *stream;
    /* GSB_FLAG_COMPACT_GRADS only (then grad_pointcloud / grad_pointcloud_features may be NULL): per scene row, zeros outside
     * the frustum -- grad_sum_compact (N,12) = xyz(3) q(4) s(3) logit(1) pad, factors applied: the columns that add up over
     * views; grad_color_compact (N,3) = dL/d(SH colour argument) of THIS view (its 48 SH gradients are the outer product
     * with this view's SH basis, GPCR:749-756). */
    float *grad_sum_compact;
    float *grad_color_compact;
    /* Optional, all NULL or all set: the densification controller's accumulators (GaussianPointAdaptiveController.py:108-116),
     * updated for every in-camera point in the epilogue of the per-point kernel exactly as GaussianPointAdaptiveController.update
     * does from the hook tensors (:130-143) -- no gathers, no extra launch.  (N) each, accumulated_position_gradients (N,3). */
    int32_t *ctl_accumulated_num_in_camera;
    int32_t *ctl_accumulated_num_pixels;
    float *ctl_accumulated_view_space_position_gradients;
    float *ctl_accumulated_view_space_position_gradients_avg;
    float *ctl_accumulated_position_gradients;
    float *ctl_accumulated_position_gradients_norm;
} GsbBackwardArgs;

/* Gradients of the per-object camera poses (the q_pointcloud_camera / t_pointcloud_camera slots of GPCR:1027, 1157-1163,
 * which the reference declares and leaves empty), for gsb200_backward_with_pose.  They are the gradients of the same surrogate
 * the xyz and feature gradients differentiate (J inside Sigma', the SH view direction and `rescale` held fixed, the 0.99 clamp
 * straight through): the pose reaches the image through the point means p_cam = W x + t_c and through the rotation of the
 * covariance, U = J W, with W = the rotation polynomial of conj(q) as given and t_c = -rotate(conj(q) / |conj(q)|, t), exactly
 * as the forward builds them.  Per view: a view-parallel (GSB_FLAG_COMPACT_GRADS) call returns this view's pose gradients. */
typedef struct GsbPoseGradArgs {
    const float *q_pointcloud_camera;  /* (num_objects,4) the forward's */
    const float *t_pointcloud_camera;  /* (num_objects,3) the forward's */
    float *grad_q_pointcloud_camera;   /* (num_objects,4) out, fully written (zeros for an object with no point in the frustum) */
    float *grad_t_pointcloud_camera;   /* (num_objects,3) out, fully written */
    void *temp;                        /* >= gsb200_pose_grad_temp_bytes(num_objects) bytes, 16-byte aligned; no initialisation */
    int64_t temp_bytes;
} GsbPoseGradArgs;

/* View-parallel training (SURVEY 8(e); the reference is single-GPU): after the ranks have exchanged their COMPACT rows --
 * all-reduce(sum) of grad_sum_compact, all-gather of [grad_color_compact | t_pointcloud_camera] -- rebuild the dense
 * gradients of the whole batch of views: (N,3) and (N,56) exactly as the sum over views of what gsb200_backward writes
 * per view (SH gradient of view v = colour-argument gradient (x) SH basis along xyz - camera centre of v, times the
 * colour factors, masked by color_max_sh_band; GPCR:749-756, 1105-1125, 1167-1182), summed in view order.
 * 14 instead of 59 floats per Gaussian cross NVLink. */
typedef struct GsbExpandArgs {
    int64_t num_points;
    int32_t num_views, num_objects;
    const float *grad_sum;          /* (N,12), already summed over the views */
    const float *grad_color_views;  /* num_views blocks, view_stride floats apart: [N*3 colour-argument gradients |
                                       num_objects*3 camera centres (that view's t_pointcloud_camera)] */
    int64_t view_stride;            /* >= 3*N + 3*num_objects */
    const float *pointcloud;        /* (N,3) */
    const int32_t *point_object_id; /* (N) */
    int32_t color_max_sh_band;
    float grad_color_factor, grad_high_order_color_factor;
    int32_t part;                    /* 0: everything.  1: only the 48 SH columns (reads the blocks, not grad_sum); 2: only xyz and the
                                        q / s / logit columns (reads grad_sum, not the blocks).  1 and 2 write disjoint pieces of
                                        the outputs, so 1 can run on another stream while the all-reduce of grad_sum is in flight */
    float *grad_pointcloud;          /* (N,3) out */
    float *grad_pointcloud_features; /* (N,56) out */
    void *stream;
} GsbExpandArgs;

/* version / errors */
int gsb200_version(void);
const char *gsb200_last_error(void);
/* sizeof(GsbWorkspaceLayout), sizeof(GsbForwardArgs), sizeof(GsbBackwardArgs) as compiled: lets a
 * foreign-language binding verify its struct mirrors. */
void gsb200_abi_sizes(int64_t *out3);
/* ... and of the first n of {GsbWorkspaceLayout, GsbForwardArgs, GsbBackwardArgs, GsbExpandArgs, GsbTrainStepArgs,
 * GsbPoseGradArgs} */
void gsb200_abi_sizes_ext(int64_t *out, int32_t n);

/* Workspace sizing.  far_plane*depth_to_sort_key_scale fixes the depth-key width; (H/16)*(W/16)
 * the tile-id width; both <= 32 bits total selects 32-bit sort keys.
 * Limits (GSB_EUNSUPPORTED beyond them): num_points < 2^26, key_capacity < 2^30.  The single-pass scan of the per-point stage
 * carries (in-camera count, pair count) in one 64-bit word with 26 + 36 bits: a frame whose REFERENCE pair count (sum of
 * num_overlap_tiles, before the reach filter and regardless of key_capacity) reached 2^36 = 6.9e10 would carry into the
 * point count -- such a frame needs > 0.8 TB of keys in the reference and is far beyond key_capacity < 2^30, but it is the
 * caller's responsibility not to submit one (e.g. millions of screen-filling splats at 4K). */
int gsb200_workspace_layout(int64_t num_points, int32_t num_objects, int64_t key_capacity,
                            int32_t camera_height, int32_t camera_width, float far_plane,
                            float depth_to_sort_key_scale, uint32_t flags,
                            GsbWorkspaceLayout *out);

/* Forward: replaces _module_function.forward, GPCR:830-1023 (K1 filter_point_in_camera GPCR:31-78,
 * mask compaction GPCR:861-864, K2 generate_point_attributes_in_camera_plane GPCR:239-315,
 * K3 generate_num_overlap_tiles GPCR:106-128, cumsum GPCR:913-922,
 * K4 generate_point_sort_key_by_num_overlap_tiles GPCR:131-172, sort GPCR:947-950,
 * K5 find_tile_start_and_end GPCR:175-193, K6 gaussian_point_rasterisation GPCR:318-485). */
int gsb200_forward(const GsbForwardArgs *args);

/* Backward: replaces _module_function.backward, GPCR:1025-1125 (K7
 * gaussian_point_rasterisation_backward GPCR:488-772, _clear_grad_by_color_max_sh_band
 * GPCR:1167-1182, factor scaling GPCR:1105-1125). */
int gsb200_backward(const GsbBackwardArgs *args);

int gsb200_expand_view_gradients(const GsbExpandArgs *args);

/* gsb200_backward plus the gradients of the object poses (GsbPoseGradArgs): every output of gsb200_backward is computed as it
 * computes it, bit for bit, and the pose gradients are summed in a fixed order (deterministic).  args->num_objects poses;
 * GSB_EUNSUPPORTED above GSB_POSE_MAX_OBJECTS, GSB_EINVAL for a null pointer or a short temp -- both checked before anything
 * is enqueued.  The pose part adds a second instantiation of the per-point kernel and one small finalisation kernel.
 * (Present since version 102; detect it by the symbol.) */
int64_t gsb200_pose_grad_temp_bytes(int32_t num_objects);
int gsb200_backward_with_pose(const GsbBackwardArgs *args, const GsbPoseGradArgs *pose);

/* The two collectives of the compact exchange as ONE hand-written kernel over NVSwitch multicast memory (NVLS; csrc/exchange.cu):
 * a two-shot all-reduce of grad_sum (multimem.ld_reduce of this rank's 1/R of the rows, multimem.st of the sums to all ranks)
 * and an all-gather of the per-view blocks (multimem.st of this rank's block into slot `rank` on all ranks).  The buffers must
 * live in one symmetric allocation mapped to a multicast address (torch.distributed._symmetric_memory); the caller brackets the
 * call with two cross-rank barriers on the same stream: all ranks' compact rows written before, all multicast stores landed
 * after (parallel.MulticastViewParallelExchange).  The alternative to ncclAllReduce + ncclAllGather of the NCCL path. */
typedef struct GsbMultimemExchangeArgs {
    int64_t num_points;
    int32_t num_objects, rank, world_size;
    int32_t num_blocks;          /* CTAs to launch; 0 = 2 per SM */
    int32_t phases;              /* 0 or 3 = both; 1 = only the all-gather push of this rank's block (needs no barrier in front if
                                    the caller alternates the blocks buffer with the step parity); 2 = only the all-reduce */
    int32_t reserved;
    float *multicast_grad_sum;   /* multicast address of the (N,12) rows */
    float *multicast_blocks;     /* multicast address of the (world_size, block_stride) blocks */
    const float *local_block;    /* this rank's own block [3N | 3 n_obj], local address */
    int64_t block_stride;        /* floats, multiple of 4, >= 3N + 3 n_obj */
    void *stream;
} GsbMultimemExchangeArgs;
int gsb200_exchange_multimem(const GsbMultimemExchangeArgs *args);

/* One WHOLE training iteration of the reference loop (GaussianPointTrainer.py:138-180) enqueued by one call, without any host
 * interaction: forward (gsb200_forward) -> clamp + L1 + D-SSIM loss and its gradient (gsb200_image_loss, LossFunction.py:20-38
 * without the optional scale regulariser) -> backward (gsb200_backward, with the controller accumulators if set) -> Adam on the
 * features and on the positions (gsb200_adam_step, GaussianPointTrainer.py:126-129, 176-177).  The scene tensors of `forward`
 * are updated in place.  `backward` must describe the same frame (same scene / workspace / sizes), with
 * grad_rasterized_image = the (H,W,3) buffer the loss gradient is written to and accum_rows >= num_points (the number of
 * in-camera points is not known on the host).  If the frame needs more (tile, splat) pairs than forward.key_capacity the
 * device-side overflow counter makes the accumulator update and both Adam steps no-ops; the host sees it in
 * forward.host_counters[2] (async copy, never waited on here) and must repeat the iteration with a larger capacity. */
typedef struct GsbTrainStepArgs {
    GsbForwardArgs forward;
    GsbBackwardArgs backward;
    const float *ground_truth_image; /* (3,H,W) as the dataset yields it */
    float lambda_value;              /* LossFunction.py:23 */
    float *loss_out3;                /* device: {loss, L1, 1 - SSIM} */
    void *loss_temp;                 /* gsb200_image_loss_temp_bytes(H, W), first 16 bytes zero before the first use */
    int64_t loss_temp_bytes;
    float *feature_exp_avg, *feature_exp_avg_sq;   /* (N,56) Adam state, zero before the first step */
    float *position_exp_avg, *position_exp_avg_sq; /* (N,3) */
    double feature_learning_rate, position_learning_rate, beta1, beta2, eps;
    int32_t step;                    /* 1-based Adam step count */
} GsbTrainStepArgs;
int gsb200_train_step(const GsbTrainStepArgs *args);

/* Individual stages (same workspace), for tests and profiling. */
int gsb200_stage_preprocess(const GsbForwardArgs *args);   /* K1+P1+K2+K3+P2+K4 fused */
int gsb200_stage_sort(const GsbForwardArgs *args);         /* P3 */
int gsb200_stage_tile_ranges(const GsbForwardArgs *args);  /* K5 */
int gsb200_stage_blend(const GsbForwardArgs *args);        /* K6 */

/* Diagnostic variants of forward/backward: identical launches with a CUDA event recorded on the
 * launching stream between stages; block until done and return device milliseconds per stage in
 * stage_ms_out[8] (host): forward = {workspace memset, preprocess, sort, tile ranges, blend};
 * backward = {grad/accumulator memsets, blend backward, per-point chain rule}.  (The reference's
 * counterpart is the Taichi kernel profiler, GaussianPointTrainer.py:217-219.) */
int gsb200_forward_timed(const GsbForwardArgs *args, float *stage_ms_out);
int gsb200_backward_timed(const GsbBackwardArgs *args, float *stage_ms_out);

/* Diagnostics: the blend kernels' real work, counted on the device (SURVEY 8(d) "E": pixel x splat evaluations).  Call after
 * gsb200_forward (same args / workspace; re-renders the same outputs) resp. after it with the backward args of the same frame
 * (adds into accum like gsb200_backward's loop A; pass a scratch accumulator).  host_out2[0] = (warp, splat) visits -- 32
 * pixel x splat evaluations each --, host_out2[1] = evaluations that contribute (alpha >= 1/255 on a live pixel).  The forward
 * variant fills 8 slots: [2..4] are what-if counters taken at staging time -- (patch, splat) pairs with the kernel's 8x4 patches,
 * with 8x8 patches (two pixels per thread) and with 16x4 patches -- the evidence for the patch shape in DESIGN.md.  Blocks.
 * (The reference's counterpart is the Taichi kernel profiler, GaussianPointTrainer.py:217-219.) */
int gsb200_forward_blend_work(const GsbForwardArgs *args, uint64_t *host_out8);
int gsb200_backward_blend_work(const GsbBackwardArgs *args, uint64_t *host_out2);

/* Checks the two hardware facts the default arithmetic path relies on: rcp.approx(1.0f) == 1.0f (a non-contributing
 * (pixel, splat) pair leaves the transmittance untouched in the branch-free backward, csrc/blend_bwd_transposed.cu) and
 * ex2.approx(0) == 1.  Returns GSB_OK or GSB_EUNSUPPORTED.  Blocks. */
int gsb200_device_selftest(void *stream);

/* find_tile_start_and_end, GPCR:175-193, on the reference's own key packing: sorted int64 keys
 * (tile << 32 | depth) -> [start, end) per tile; outputs must be zero-initialised (GPCR:954-957). */
int gsb200_find_tile_start_and_end(const int64_t *sorted_keys, int64_t num_keys, int32_t *tile_points_start,
                                   int32_t *tile_points_end, int32_t num_tiles, void *stream);

/* Stand-alone stable LSD radix sort of (key, int32 payload) pairs on the device; key_bytes 4 or 8,
 * bits [0, end_bit) are sorted.  temp must hold gsb200_sort_temp_bytes(n, key_bytes). Result is
 * left in keys_out / vals_out.  (Replaces torch.sort + gather, GPCR:947-950.) */
int64_t gsb200_sort_temp_bytes(int64_t n, int32_t key_bytes);
int gsb200_sort_pairs(const void *keys_in, const int32_t *vals_in, void *keys_out, int32_t *vals_out,
                      int64_t n, int32_t key_bytes, int32_t end_bit, void *temp, int64_t temp_bytes,
                      void *stream);

/* Host-buffer entry point (end-to-end inference call): the scene stays resident on the device, the
 * per-view inputs (pose, intrinsics) come from HOST memory and the image is returned to HOST memory.
 * host pointers should be pinned.  Blocks until the image is in host memory.
 * Replaces the render loop body gaussian_point_render.py:106-121 (pose .cuda(), forward, image .cpu()). */
int gsb200_render_host(const GsbForwardArgs *device_args, const float *host_q_pointcloud_camera,
                       const float *host_t_pointcloud_camera, const float *host_camera_intrinsics,
                       float *staging_device_pose /* >= num_objects*7+9 floats, device */,
                       float *host_image_out /* (H,W,3) */, int64_t *host_counters_out /* int64[4] or NULL */);

/* Fused clamp + L1 loss + gradient for the trainer step around the operator (SURVEY 8(f)-2):
 * loss = mean |clamp01(pred) - gt| (GaussianPointTrainer.py:168-170 clamp, LossFunction.py:29 L1) and, when
 * grad_predicted_out is not NULL, d(upstream_grad * loss)/d pred = upstream_grad * sign(.)/n inside the clamp
 * range, 0 outside -- what torch autograd produces with ~8 elementwise kernels.  All pointers are device
 * memory, 16-byte aligned; temp holds gsb200_l1_loss_temp_bytes() bytes and must be ZERO before its first use
 * (the call leaves it ready for the next one).  Deterministic (fixed grid, fixed summation order). */
int64_t gsb200_l1_loss_temp_bytes(void);
int gsb200_l1_loss(const float *predicted_image, const float *ground_truth_image, int64_t num_elements,
                   int32_t clamp01, float upstream_grad, float *loss_out, float *grad_predicted_out, void *temp,
                   int64_t temp_bytes, void *stream);

/* The trainer's whole image loss and its gradient (SURVEY 8(f)-2/3) in two kernels:
 *   pred = clamp(rasterized_image, 0, 1)                                  GaussianPointTrainer.py:168-170
 *   L    = (1 - lambda) * mean|pred - gt| + lambda * (1 - SSIM(pred, gt))  LossFunction.py:20-38
 * SSIM = the published pytorch_msssim algorithm the reference calls (LossFunction.py:4,31): 11-tap Gaussian window,
 * sigma 1.5, VALID padding, K = (0.01, 0.03), data_range 1, mean over the map.  rasterized_image is (H,W,3) as the
 * rasteriser returns it, ground_truth_image (3,H,W) as the dataset yields it; H, W > 10.  loss_out3 = {L, L1, 1 - SSIM};
 * grad_rasterized_image (H,W,3), if not NULL, receives upstream_grad * dL/d rasterized_image (zero where the clamp is
 * active).  temp holds gsb200_image_loss_temp_bytes(H, W) bytes, 16-byte aligned; its first 16 bytes must be ZERO before
 * the first use (the call leaves them ready for the next one).  Deterministic (fixed grid, fixed summation order).
 * Replaces ~60 autograd kernels per step (5 grouped convolutions, their transposes, ~25 elementwise). */
int64_t gsb200_image_loss_temp_bytes(int32_t camera_height, int32_t camera_width);
int gsb200_image_loss(const float *rasterized_image, const float *ground_truth_image, int32_t camera_height,
                      int32_t camera_width, float lambda_value, float upstream_grad, float *loss_out3,
                      float *grad_rasterized_image, void *temp, int64_t temp_bytes, void *stream);

/* One Adam step on a flat float32 tensor in ONE kernel (SURVEY 8(f)-2): the update of torch.optim.Adam as the reference
 * trainer configures it (GaussianPointTrainer.py:126-129: betas given, eps 1e-8, no weight decay, no amsgrad; stepped at
 * :176-177) -- m += (g - m)(1 - b1); v = v b2 + (1 - b2) g^2; p -= lr / (1 - b1^t) * m / (sqrt(v) / sqrt(1 - b2^t) + eps).
 * `step` is the 1-based step count t.  All pointers device memory, 16-byte aligned; exp_avg / exp_avg_sq are the
 * caller-owned state (zero before the first step).  lr / betas / eps are doubles like torch's Python floats (1 - beta is
 * formed in double).  HBM-bound: 28 B per element. */
int gsb200_adam_step(float *param, const float *grad, float *exp_avg, float *exp_avg_sq, int64_t num_elements, double lr,
                     double beta1, double beta2, double eps, int32_t step, void *stream);

/* The densification controller's per-iteration accumulator update in ONE kernel (SURVEY 8(f)-1): what
 * GaussianPointAdaptiveController.update does with the backward-hook tensors, GaussianPointAdaptiveController.py:130-143
 * (six indexed accumulations, mag / n_pixels with NaN -> 0, row norm; ~15 torch launches).  The first five arguments are
 * fields of BackwardValidPointHookInput (M entries), the last six the controller's accumulators (N entries; int32 / float32).
 * ids must be unique (they are: GPCR:861-864).  All pointers device memory. */
int gsb200_controller_update(const int32_t *point_id_in_camera_list, int64_t num_points_in_camera,
                             const int32_t *num_affected_pixels, const float *magnitude_grad_viewspace,
                             const float *grad_point_in_camera, int32_t *accumulated_num_in_camera,
                             int32_t *accumulated_num_pixels, float *accumulated_view_space_position_gradients,
                             float *accumulated_view_space_position_gradients_avg, float *accumulated_position_gradients,
                             float *accumulated_position_gradients_norm, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* GSB200_H_ */
