// api.cu -- extern "C" entry points of libgsb200.so (see include/gsb200.h).
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "common.cuh"

namespace gsb {

static thread_local char g_error[512] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

static inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

static int bit_width(uint64_t v) {
    int b = 0;
    while (v) {
        ++b;
        v >>= 1;
    }
    return b;
}

static int compute_layout(int64_t N, int32_t n_obj, int64_t key_capacity, int32_t H, int32_t W,
                          float far_plane, float depth_scale, uint32_t flags, GsbWorkspaceLayout *L) {
    if (!L) {
        set_error("workspace_layout: out is null");
        return GSB_EINVAL;
    }
    if (N < 0 || n_obj < 0 || key_capacity < 0 || H <= 0 || W <= 0) {
        set_error("workspace_layout: negative size (N=%lld n_obj=%d K_cap=%lld H=%d W=%d)", (long long)N,
                  n_obj, (long long)key_capacity, H, W);
        return GSB_EINVAL;
    }
    if (H % GSB_TILE_HEIGHT != 0 || W % GSB_TILE_WIDTH != 0) {  // GPCR:1193-1194
        set_error("camera size %dx%d must be a multiple of the 16x16 tile", W, H);
        return GSB_EINVAL;
    }
    if (N >= (1LL << 26) || key_capacity >= (1LL << 30)) {
        set_error("scene too large for the packed scan state (N < 2^26, key_capacity < 2^30)");
        return GSB_EUNSUPPORTED;
    }
    memset(L, 0, sizeof(*L));
    const int64_t T = (int64_t)(H / GSB_TILE_HEIGHT) * (W / GSB_TILE_WIDTH);
    L->tile_bits = bit_width((uint64_t)(T > 0 ? T - 1 : 0));
    const float mk = far_plane * depth_scale;  // f32 product, like the kernel's depth * scale
    int64_t max_key = mk >= 2147483648.0f ? 2147483647LL : (mk > 0.0f ? (int64_t)(int32_t)mk : 0);
    L->depth_bits = bit_width((uint64_t)max_key);
    if (L->depth_bits < 1) L->depth_bits = 1;
    if ((flags & GSB_FLAG_FORCE_KEY64) || L->tile_bits + L->depth_bits > 32) {
        L->key_bytes = 8;
        L->depth_bits = 32;  // exactly the reference's (tile << 32) + depth packing
    } else {
        L->key_bytes = 4;
    }
    L->radix_bits = sort_radix_bits(L->tile_bits + L->depth_bits);
    L->sort_passes = (L->tile_bits + L->depth_bits + L->radix_bits - 1) / L->radix_bits;
    if (L->sort_passes < 1) L->sort_passes = 1;
    L->key_capacity_padded = align_up(key_capacity > 0 ? key_capacity : 1, SORT_TILE);
    L->sort_blocks = (int32_t)(L->key_capacity_padded / SORT_TILE);
    L->scan_blocks = (int32_t)((N + SCAN_BLOCK_THREADS - 1) / SCAN_BLOCK_THREADS);

    int64_t off = 0;
    auto take = [&](int64_t bytes) {
        int64_t o = off;
        off = align_up(off + bytes, 256);
        return o;
    };
    L->counters = take(8 * sizeof(int64_t));
    L->tickets = take(16 * sizeof(uint32_t));
    L->scan_state = take((int64_t)(L->scan_blocks + 1) * 8);
    L->sort_hist = take(8 * 1024 * 4);
    L->sort_state = take((int64_t)L->sort_passes * L->sort_blocks * (1 << L->radix_bits) * 4);
    L->tile_start = take(T * 4);
    L->tile_end = take(T * 4);
    L->zero_bytes = off;
    L->poses = take((int64_t)(n_obj > 0 ? n_obj : 1) * sizeof(PoseBlock));
    L->point_id = take(N * 4);
    L->point_offset = take(N * 4);
    L->num_tiles = take(N * 4);
    L->records = take(N * GSB_RECORD_FLOATS * 4);
    L->point_in_camera = take(N * 3 * 4);
    L->keys_a = take(L->key_capacity_padded * L->key_bytes);
    L->keys_b = take(L->key_capacity_padded * L->key_bytes);
    L->vals_a = take(L->key_capacity_padded * 4);
    L->vals_b = take(L->key_capacity_padded * 4);
    L->keys_c = take(L->key_capacity_padded * L->key_bytes);
    L->vals_c = take(L->key_capacity_padded * 4);
    L->total_bytes = off;
    return GSB_OK;
}

int resolve_workspace(void *base, int64_t bytes, int64_t N, int32_t n_obj, int64_t key_capacity,
                      int32_t H, int32_t W, float far_plane, float depth_scale, uint32_t flags,
                      Workspace *ws) {
    int rc = compute_layout(N, n_obj, key_capacity, H, W, far_plane, depth_scale, flags, &ws->layout);
    if (rc != GSB_OK) return rc;
    const GsbWorkspaceLayout &L = ws->layout;
    if (!base || bytes < L.total_bytes) {
        set_error("workspace too small: have %lld bytes, need %lld", (long long)bytes, (long long)L.total_bytes);
        return GSB_EWORKSPACE;
    }
    if (reinterpret_cast<uintptr_t>(base) % 256 != 0) {
        set_error("workspace must be 256-byte aligned");
        return GSB_EINVAL;
    }
    char *b = static_cast<char *>(base);
    ws->counters = reinterpret_cast<long long *>(b + L.counters);
    ws->tickets = reinterpret_cast<unsigned int *>(b + L.tickets);
    ws->scan_state = reinterpret_cast<unsigned long long *>(b + L.scan_state);
    ws->sort_hist = reinterpret_cast<unsigned int *>(b + L.sort_hist);
    ws->sort_state = reinterpret_cast<unsigned int *>(b + L.sort_state);
    ws->tile_start = reinterpret_cast<int *>(b + L.tile_start);
    ws->tile_end = reinterpret_cast<int *>(b + L.tile_end);
    ws->poses = reinterpret_cast<PoseBlock *>(b + L.poses);
    ws->point_id = reinterpret_cast<int *>(b + L.point_id);
    ws->point_offset = reinterpret_cast<int *>(b + L.point_offset);
    ws->num_tiles = reinterpret_cast<int *>(b + L.num_tiles);
    ws->records = reinterpret_cast<float4 *>(b + L.records);
    ws->point_in_camera = reinterpret_cast<float *>(b + L.point_in_camera);
    ws->keys_a = b + L.keys_a;
    ws->keys_b = b + L.keys_b;
    ws->vals_a = reinterpret_cast<int *>(b + L.vals_a);
    ws->vals_b = reinterpret_cast<int *>(b + L.vals_b);
    ws->keys_c = b + L.keys_c;
    ws->vals_c = reinterpret_cast<int *>(b + L.vals_c);
    ws->patch_masks = reinterpret_cast<unsigned char *>(b + L.keys_c);  // key_capacity_padded * key_bytes >= one byte per key
    return GSB_OK;
}

static int check_forward_args(const GsbForwardArgs *a) {
    if (!a) {
        set_error("forward: args is null");
        return GSB_EINVAL;
    }
    if (a->num_points > 0 && (!a->pointcloud || !a->pointcloud_features || !a->point_invalid_mask ||
                              !a->point_object_id)) {
        set_error("forward: null scene pointer");
        return GSB_EINVAL;
    }
    if (a->num_points > 0 && (a->num_objects <= 0 || !a->q_pointcloud_camera || !a->t_pointcloud_camera)) {
        set_error("forward: need at least one object pose");
        return GSB_EINVAL;
    }
    if (!a->camera_intrinsics || !a->rasterized_image) {
        set_error("forward: null camera_intrinsics / rasterized_image");
        return GSB_EINVAL;
    }
    if (!a->rgb_only && (!a->rasterized_depth || !a->pixel_accumulated_alpha ||
                         !a->pixel_offset_of_last_effective_point || !a->pixel_valid_point_count)) {
        set_error("forward: aux outputs are required unless rgb_only");
        return GSB_EINVAL;
    }
    if (a->near_plane < 0.0f) {
        set_error("forward: near_plane must be >= 0 (depth keys are unsigned)");
        return GSB_EUNSUPPORTED;
    }
    if (reinterpret_cast<uintptr_t>(a->pointcloud_features) % 16 != 0) {
        set_error("forward: pointcloud_features must be 16-byte aligned");
        return GSB_EINVAL;
    }
    return GSB_OK;
}

static int resolve_fwd(const GsbForwardArgs *a, Workspace *ws) {
    int rc = check_forward_args(a);
    if (rc != GSB_OK) return rc;
    return resolve_workspace(a->workspace, a->workspace_bytes, a->num_points, a->num_objects,
                             a->key_capacity, a->camera_height, a->camera_width, a->far_plane,
                             a->depth_to_sort_key_scale, a->flags, ws);
}

}  // namespace gsb

using namespace gsb;

extern "C" {

int gsb200_version(void) { return GSB200_VERSION; }

const char *gsb200_last_error(void) { return g_error; }

void gsb200_abi_sizes(int64_t *out3) {
    out3[0] = (int64_t)sizeof(GsbWorkspaceLayout);
    out3[1] = (int64_t)sizeof(GsbForwardArgs);
    out3[2] = (int64_t)sizeof(GsbBackwardArgs);
}

void gsb200_abi_sizes_ext(int64_t *out, int32_t n) {
    const int64_t all[6] = {(int64_t)sizeof(GsbWorkspaceLayout), (int64_t)sizeof(GsbForwardArgs), (int64_t)sizeof(GsbBackwardArgs),
                            (int64_t)sizeof(GsbExpandArgs), (int64_t)sizeof(GsbTrainStepArgs), (int64_t)sizeof(GsbPoseGradArgs)};
    for (int i = 0; i < n && i < 6; ++i) out[i] = all[i];
}

int gsb200_workspace_layout(int64_t num_points, int32_t num_objects, int64_t key_capacity,
                            int32_t camera_height, int32_t camera_width, float far_plane,
                            float depth_to_sort_key_scale, uint32_t flags, GsbWorkspaceLayout *out) {
    return compute_layout(num_points, num_objects, key_capacity, camera_height, camera_width, far_plane,
                          depth_to_sort_key_scale, flags, out);
}

int gsb200_stage_preprocess(const GsbForwardArgs *a) {
    Workspace ws;
    int rc = resolve_fwd(a, &ws);
    if (rc != GSB_OK) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(a->stream);
    GSB_CUDA_CHECK(cudaMemsetAsync(a->workspace, 0, (size_t)ws.layout.zero_bytes, st));
    return launch_preprocess(*a, ws, st);
}

int gsb200_stage_sort(const GsbForwardArgs *a) {
    Workspace ws;
    int rc = resolve_fwd(a, &ws);
    if (rc != GSB_OK) return rc;
    return launch_sort(ws, a->key_capacity, static_cast<cudaStream_t>(a->stream));
}

int gsb200_stage_tile_ranges(const GsbForwardArgs *a) {
    Workspace ws;
    int rc = resolve_fwd(a, &ws);
    if (rc != GSB_OK) return rc;
    const int T = (a->camera_height / GSB_TILE_HEIGHT) * (a->camera_width / GSB_TILE_WIDTH);
    return launch_tile_ranges(ws, a->key_capacity, T, static_cast<cudaStream_t>(a->stream));
}

int gsb200_stage_blend(const GsbForwardArgs *a) {
    Workspace ws;
    int rc = resolve_fwd(a, &ws);
    if (rc != GSB_OK) return rc;
    return launch_blend_forward(*a, ws, static_cast<cudaStream_t>(a->stream));
}

int gsb200_forward(const GsbForwardArgs *a) {
    Workspace ws;
    int rc = resolve_fwd(a, &ws);
    if (rc != GSB_OK) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(a->stream);
    GSB_CUDA_CHECK(cudaMemsetAsync(a->workspace, 0, (size_t)ws.layout.zero_bytes, st));
    if ((rc = launch_preprocess(*a, ws, st)) != GSB_OK) return rc;
    if (a->host_counters && a->host_counters_event) {
        GSB_CUDA_CHECK(cudaMemcpyAsync(a->host_counters, ws.counters, 4 * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        GSB_CUDA_CHECK(cudaEventRecord(static_cast<cudaEvent_t>(a->host_counters_event), st));
    }
    if ((rc = launch_sort(ws, a->key_capacity, st)) != GSB_OK) return rc;
    const int T = (a->camera_height / GSB_TILE_HEIGHT) * (a->camera_width / GSB_TILE_WIDTH);
    if ((rc = launch_tile_ranges(ws, a->key_capacity, T, st)) != GSB_OK) return rc;
    return launch_blend_forward(*a, ws, st);
}

static int backward_impl(const GsbBackwardArgs *a, bool skip_on_overflow, const GsbPoseGradArgs *pose = nullptr) {
    if (!a) {
        set_error("backward: args is null");
        return GSB_EINVAL;
    }
    const bool compact = (a->flags & GSB_FLAG_COMPACT_GRADS) != 0;
    if (!a->grad_rasterized_image || !a->pixel_accumulated_alpha ||
        !a->pixel_offset_of_last_effective_point || !a->magnitude_grad_viewspace_on_image ||
        !a->camera_intrinsics ||
        (a->num_points > 0 && (!a->pointcloud || !a->pointcloud_features || !a->point_object_id || !a->t_pointcloud_camera)) ||
        (a->num_points > 0 && !compact && (!a->grad_pointcloud || !a->grad_pointcloud_features)) ||
        (a->num_points > 0 && compact && (!a->grad_sum_compact || !a->grad_color_compact))) {
        set_error("backward: null pointer argument");
        return GSB_EINVAL;
    }
    {
        const void *ctl[6] = {a->ctl_accumulated_num_in_camera, a->ctl_accumulated_num_pixels,
                              a->ctl_accumulated_view_space_position_gradients,
                              a->ctl_accumulated_view_space_position_gradients_avg, a->ctl_accumulated_position_gradients,
                              a->ctl_accumulated_position_gradients_norm};
        int set = 0;
        for (const void *c : ctl) set += c != nullptr;
        if (set != 0 && set != 6) {
            set_error("backward: the six controller accumulators must be all NULL or all set");
            return GSB_EINVAL;
        }
        if (set == 6 && (a->flags & GSB_FLAG_NO_HOOK_STATS)) {
            set_error("backward: the controller accumulators need the hook statistics (GSB_FLAG_NO_HOOK_STATS is set)");
            return GSB_EINVAL;
        }
    }
    if (compact && reinterpret_cast<uintptr_t>(a->grad_sum_compact) % 16 != 0) {
        set_error("backward: grad_sum_compact must be 16-byte aligned");
        return GSB_EINVAL;
    }
    if (a->accum_rows > 0 && !a->accum) {
        set_error("backward: accum is null");
        return GSB_EINVAL;
    }
    Workspace ws;
    int rc = resolve_workspace(a->workspace, a->workspace_bytes, a->num_points, a->num_objects,
                               a->key_capacity, a->camera_height, a->camera_width, a->far_plane,
                               a->depth_to_sort_key_scale, a->flags, &ws);
    if (rc != GSB_OK) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(a->stream);
    if (a->accum_rows > 0)
        GSB_CUDA_CHECK(cudaMemsetAsync(a->accum, 0, (size_t)a->accum_rows * GSB_ACCUM_FLOATS * 4, st));
    if ((rc = launch_blend_backward(*a, ws, st)) != GSB_OK) return rc;
    return launch_backward_points(*a, ws, st, skip_on_overflow ? ws.counters + CNT_OVERFLOW : nullptr, pose);
}

int gsb200_backward(const GsbBackwardArgs *a) { return backward_impl(a, false); }

int64_t gsb200_pose_grad_temp_bytes(int32_t num_objects) {
    return num_objects > 0 ? (int64_t)POSE_MAX_BLOCKS * num_objects * 12 * (int64_t)sizeof(float) : 0;
}

int gsb200_backward_with_pose(const GsbBackwardArgs *a, const GsbPoseGradArgs *pose) {
    if (!a || !pose) {
        set_error("backward_with_pose: args or pose is null");
        return GSB_EINVAL;
    }
    if (a->num_objects > GSB_POSE_MAX_OBJECTS) {
        set_error("backward_with_pose: %d objects, at most %d poses can be differentiated", a->num_objects, GSB_POSE_MAX_OBJECTS);
        return GSB_EUNSUPPORTED;
    }
    if (a->num_objects < 1 || !pose->q_pointcloud_camera || !pose->t_pointcloud_camera || !pose->grad_q_pointcloud_camera ||
        !pose->grad_t_pointcloud_camera || !pose->temp) {
        set_error("backward_with_pose: null pointer argument or no object");
        return GSB_EINVAL;
    }
    if (pose->temp_bytes < gsb200_pose_grad_temp_bytes(a->num_objects) || reinterpret_cast<uintptr_t>(pose->temp) % 16 != 0) {
        set_error("backward_with_pose: temp must hold %lld bytes, 16-byte aligned (have %lld)",
                  (long long)gsb200_pose_grad_temp_bytes(a->num_objects), (long long)pose->temp_bytes);
        return GSB_EINVAL;
    }
    return backward_impl(a, false, pose);
}

int gsb200_image_loss(const float *rasterized_image, const float *ground_truth_image, int32_t camera_height,
                      int32_t camera_width, float lambda_value, float upstream_grad, float *loss_out3,
                      float *grad_rasterized_image, void *temp, int64_t temp_bytes, void *stream);

int gsb200_train_step(const GsbTrainStepArgs *t) {
    if (!t || !t->ground_truth_image || !t->loss_out3 || !t->loss_temp || !t->feature_exp_avg || !t->feature_exp_avg_sq ||
        !t->position_exp_avg || !t->position_exp_avg_sq || t->step < 1) {
        set_error("train_step: null pointer argument or step < 1");
        return GSB_EINVAL;
    }
    const GsbForwardArgs &f = t->forward;
    const GsbBackwardArgs &b = t->backward;
    if (f.rgb_only || f.num_points != b.num_points || f.workspace != b.workspace || f.camera_height != b.camera_height ||
        f.camera_width != b.camera_width || f.stream != b.stream || b.accum_rows < f.num_points ||
        (b.flags & GSB_FLAG_COMPACT_GRADS) || !b.grad_rasterized_image || !b.grad_pointcloud || !b.grad_pointcloud_features ||
        b.pointcloud != f.pointcloud || b.pointcloud_features != f.pointcloud_features) {
        set_error("train_step: forward / backward blocks do not describe one frame (or rgb_only / compact gradients set)");
        return GSB_EINVAL;
    }
    int rc = gsb200_forward(&f);
    if (rc != GSB_OK) return rc;
    rc = gsb200_image_loss(f.rasterized_image, t->ground_truth_image, f.camera_height, f.camera_width, t->lambda_value, 1.0f,
                           t->loss_out3, const_cast<float *>(b.grad_rasterized_image), t->loss_temp, t->loss_temp_bytes, f.stream);
    if (rc != GSB_OK) return rc;
    if ((rc = backward_impl(&b, true)) != GSB_OK) return rc;
    Workspace ws;
    if ((rc = resolve_fwd(&f, &ws)) != GSB_OK) return rc;
    const long long *skip = ws.counters + CNT_OVERFLOW;
    cudaStream_t st = static_cast<cudaStream_t>(f.stream);
    rc = launch_adam_step(f.pointcloud_features, b.grad_pointcloud_features, t->feature_exp_avg, t->feature_exp_avg_sq,
                          (long long)f.num_points * GSB_FEATURE_DIM, t->feature_learning_rate, t->beta1, t->beta2, t->eps, t->step,
                          skip, st);
    if (rc != GSB_OK) return rc;
    return launch_adam_step(const_cast<float *>(f.pointcloud), b.grad_pointcloud, t->position_exp_avg, t->position_exp_avg_sq,
                            (long long)f.num_points * 3, t->position_learning_rate, t->beta1, t->beta2, t->eps, t->step, skip, st);
}

int gsb200_expand_view_gradients(const GsbExpandArgs *a) {
    if (!a || a->num_points < 0 || a->num_views < 1 || a->num_objects < 1 || a->part < 0 || a->part > 2 ||
        (a->num_points > 0 && (!a->grad_sum || !a->grad_color_views || !a->pointcloud || !a->point_object_id ||
                               !a->grad_pointcloud || !a->grad_pointcloud_features)) ||
        a->view_stride < 3 * a->num_points + 3 * (int64_t)a->num_objects) {
        set_error("expand_view_gradients: bad arguments");
        return GSB_EINVAL;
    }
    if (reinterpret_cast<uintptr_t>(a->grad_sum) % 16 != 0 || reinterpret_cast<uintptr_t>(a->grad_pointcloud_features) % 16 != 0) {
        set_error("expand_view_gradients: grad_sum and grad_pointcloud_features must be 16-byte aligned");
        return GSB_EINVAL;
    }
    return launch_expand_view_gradients(*a, static_cast<cudaStream_t>(a->stream));
}

// ---- diagnostic variants: same launches as gsb200_forward / gsb200_backward with a CUDA event recorded
// on the launching stream between stages; returns device milliseconds per stage (host array of 8).
namespace {
struct StageTimer {
    cudaEvent_t ev[9];
    int n = 0;
    cudaStream_t st;
    bool ok = true;
    explicit StageTimer(cudaStream_t s) : st(s) {
        for (auto &e : ev) ok = ok && cudaEventCreate(&e) == cudaSuccess;
    }
    ~StageTimer() {
        for (auto &e : ev) cudaEventDestroy(e);
    }
    void mark() {
        if (n < 9) cudaEventRecord(ev[n++], st);
    }
    int finish(float *out) {
        if (cudaStreamSynchronize(st) != cudaSuccess) return GSB_ECUDA;
        for (int i = 0; i < 8; ++i) out[i] = 0.0f;
        for (int i = 0; i + 1 < n; ++i) cudaEventElapsedTime(&out[i], ev[i], ev[i + 1]);
        return GSB_OK;
    }
};
}  // namespace

int gsb200_forward_timed(const GsbForwardArgs *a, float *stage_ms_out) {
    Workspace ws;
    int rc = resolve_fwd(a, &ws);
    if (rc != GSB_OK) return rc;
    if (!stage_ms_out) return GSB_EINVAL;
    cudaStream_t st = static_cast<cudaStream_t>(a->stream);
    StageTimer t(st);
    if (!t.ok) {
        set_error("forward_timed: cudaEventCreate failed");
        return GSB_ECUDA;
    }
    const int T = (a->camera_height / GSB_TILE_HEIGHT) * (a->camera_width / GSB_TILE_WIDTH);
    t.mark();
    GSB_CUDA_CHECK(cudaMemsetAsync(a->workspace, 0, (size_t)ws.layout.zero_bytes, st));
    t.mark();
    if ((rc = launch_preprocess(*a, ws, st)) != GSB_OK) return rc;
    t.mark();
    if ((rc = launch_sort(ws, a->key_capacity, st)) != GSB_OK) return rc;
    t.mark();
    if ((rc = launch_tile_ranges(ws, a->key_capacity, T, st)) != GSB_OK) return rc;
    t.mark();
    if ((rc = launch_blend_forward(*a, ws, st)) != GSB_OK) return rc;
    t.mark();
    return t.finish(stage_ms_out);
}

int gsb200_backward_timed(const GsbBackwardArgs *a, float *stage_ms_out) {
    if (!a || !stage_ms_out) return GSB_EINVAL;
    Workspace ws;
    int rc = resolve_workspace(a->workspace, a->workspace_bytes, a->num_points, a->num_objects,
                               a->key_capacity, a->camera_height, a->camera_width, a->far_plane,
                               a->depth_to_sort_key_scale, a->flags, &ws);
    if (rc != GSB_OK) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(a->stream);
    StageTimer t(st);
    if (!t.ok) {
        set_error("backward_timed: cudaEventCreate failed");
        return GSB_ECUDA;
    }
    t.mark();
    if (a->accum_rows > 0)
        GSB_CUDA_CHECK(cudaMemsetAsync(a->accum, 0, (size_t)a->accum_rows * GSB_ACCUM_FLOATS * 4, st));
    t.mark();
    if ((rc = launch_blend_backward(*a, ws, st)) != GSB_OK) return rc;
    t.mark();
    if ((rc = launch_backward_points(*a, ws, st)) != GSB_OK) return rc;
    t.mark();
    return t.finish(stage_ms_out);
}

int gsb200_forward_blend_work(const GsbForwardArgs *a, uint64_t *host_out8) {
    Workspace ws;
    int rc = resolve_fwd(a, &ws);
    if (rc != GSB_OK) return rc;
    if (!host_out8 || a->rgb_only) {
        set_error("forward_blend_work: host_out8 is null or rgb_only is set");
        return GSB_EINVAL;
    }
    cudaStream_t st = static_cast<cudaStream_t>(a->stream);
    unsigned long long *cnt = nullptr;  // a blocking diagnostic: its own small allocation
    GSB_CUDA_CHECK(cudaMalloc(&cnt, 64));
    cudaError_t e = cudaMemsetAsync(cnt, 0, 64, st);
    if (e == cudaSuccess) {
        rc = launch_blend_forward_count(*a, ws, cnt, st);
        if (rc == GSB_OK) e = cudaMemcpyAsync(host_out8, cnt, 64, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    }
    cudaFree(cnt);
    if (rc != GSB_OK) return rc;
    if (e != cudaSuccess) {
        set_error("forward_blend_work: %s", cudaGetErrorString(e));
        return GSB_ECUDA;
    }
    return GSB_OK;
}

int gsb200_backward_blend_work(const GsbBackwardArgs *a, uint64_t *host_out2) {
    if (!a || !host_out2 || !a->grad_rasterized_image || !a->pixel_accumulated_alpha ||
        !a->pixel_offset_of_last_effective_point || !a->accum) {
        set_error("backward_blend_work: null pointer argument");
        return GSB_EINVAL;
    }
    Workspace ws;
    int rc = resolve_workspace(a->workspace, a->workspace_bytes, a->num_points, a->num_objects,
                               a->key_capacity, a->camera_height, a->camera_width, a->far_plane,
                               a->depth_to_sort_key_scale, a->flags, &ws);
    if (rc != GSB_OK) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(a->stream);
    unsigned long long *cnt = reinterpret_cast<unsigned long long *>(ws.counters + 6);
    GSB_CUDA_CHECK(cudaMemsetAsync(cnt, 0, 16, st));
    if ((rc = launch_blend_backward_work(*a, ws, cnt, st)) != GSB_OK) return rc;
    GSB_CUDA_CHECK(cudaMemcpyAsync(host_out2, cnt, 16, cudaMemcpyDeviceToHost, st));
    GSB_CUDA_CHECK(cudaStreamSynchronize(st));
    return GSB_OK;
}

namespace {
__global__ void selftest_kernel(unsigned int *out) {
    float one = 1.0f, zero = 0.0f, r, e;
    asm volatile("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(one));
    asm volatile("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(zero));
    out[0] = __float_as_uint(r);
    out[1] = __float_as_uint(e);
}
}  // namespace

int gsb200_device_selftest(void *stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    unsigned int *dev = nullptr, host[2] = {0u, 0u};
    GSB_CUDA_CHECK(cudaMalloc(&dev, 8));
    selftest_kernel<<<1, 1, 0, st>>>(dev);
    cudaError_t e = cudaMemcpyAsync(host, dev, 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(dev);
    if (e != cudaSuccess) {
        set_error("device_selftest: %s", cudaGetErrorString(e));
        return GSB_ECUDA;
    }
    if (host[0] != 0x3f800000u || host[1] != 0x3f800000u) {
        set_error("device_selftest: rcp.approx(1) = 0x%08x, ex2.approx(0) = 0x%08x (both must be 1.0f exactly)", host[0], host[1]);
        return GSB_EUNSUPPORTED;
    }
    return GSB_OK;
}

int gsb200_find_tile_start_and_end(const int64_t *sorted_keys, int64_t num_keys, int32_t *tile_points_start,
                                   int32_t *tile_points_end, int32_t num_tiles, void *stream) {
    if (num_keys < 0 || num_tiles < 0 || (num_keys > 0 && (!sorted_keys || !tile_points_start || !tile_points_end))) {
        set_error("find_tile_start_and_end: bad arguments");
        return GSB_EINVAL;
    }
    return launch_tile_ranges_raw(reinterpret_cast<const long long *>(sorted_keys), num_keys, tile_points_start,
                                  tile_points_end, num_tiles, static_cast<cudaStream_t>(stream));
}

int64_t gsb200_sort_temp_bytes(int64_t n, int32_t key_bytes) {
    const int64_t padded = align_up(n > 0 ? n : 1, SORT_TILE);
    const int64_t blocks = padded / SORT_TILE;
    int64_t off = 0;
    off += 256;                                      // n_dev
    off += 256;                                      // tickets
    off += 8 * 1024 * 4;                             // hist (up to 8 passes of up to 1024 bins)
    off += align_up(8 * blocks * 1024 * 4, 256);     // look-back state (up to 8 passes x 1024 digits)
    off += align_up(padded * key_bytes, 256);        // tmp keys
    off += align_up(padded * 4, 256);                // tmp vals
    return off;
}

int gsb200_sort_pairs(const void *keys_in, const int32_t *vals_in, void *keys_out, int32_t *vals_out,
                      int64_t n, int32_t key_bytes, int32_t end_bit, void *temp, int64_t temp_bytes,
                      void *stream) {
    if (n < 0 || (key_bytes != 4 && key_bytes != 8) || end_bit < 1 || end_bit > key_bytes * 8) {
        set_error("sort_pairs: bad arguments (n=%lld key_bytes=%d end_bit=%d)", (long long)n, key_bytes, end_bit);
        return GSB_EINVAL;
    }
    if (n == 0) return GSB_OK;
    if (n >= (1LL << 30)) {
        set_error("sort_pairs: n must be < 2^30");
        return GSB_EUNSUPPORTED;
    }
    if (!keys_in || !vals_in || !keys_out || !vals_out || !temp || temp_bytes < gsb200_sort_temp_bytes(n, key_bytes)) {
        set_error("sort_pairs: null pointer or temp too small");
        return GSB_EINVAL;
    }
    if (reinterpret_cast<uintptr_t>(keys_in) % 16 != 0 || reinterpret_cast<uintptr_t>(temp) % 256 != 0) {
        set_error("sort_pairs: keys_in must be 16-byte aligned and temp 256-byte aligned");
        return GSB_EINVAL;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int64_t padded = align_up(n, SORT_TILE);
    const int64_t blocks = padded / SORT_TILE;
    char *b = static_cast<char *>(temp);
    long long *n_dev = reinterpret_cast<long long *>(b);
    unsigned int *tickets = reinterpret_cast<unsigned int *>(b + 256);
    unsigned int *hist = reinterpret_cast<unsigned int *>(b + 512);
    unsigned int *state = reinterpret_cast<unsigned int *>(b + 512 + 8 * 1024 * 4);
    const int64_t state_bytes = align_up(8 * blocks * 1024 * 4, 256);
    void *tmp_keys = b + 512 + 8 * 1024 * 4 + state_bytes;
    int *tmp_vals = reinterpret_cast<int *>(static_cast<char *>(tmp_keys) + align_up(padded * key_bytes, 256));
    GSB_CUDA_CHECK(cudaMemsetAsync(b, 0, (size_t)(512 + 8 * 1024 * 4 + state_bytes), st));
    const long long n_host = n;
    GSB_CUDA_CHECK(cudaMemcpyAsync(n_dev, &n_host, sizeof(n_host), cudaMemcpyHostToDevice, st));
    return sort_pairs_device(keys_in, vals_in, keys_out, vals_out, n_dev, padded, key_bytes, 0, end_bit, nullptr, hist,
                             state, tickets, tmp_keys, tmp_vals, st);
}

int gsb200_render_host(const GsbForwardArgs *device_args, const float *host_q, const float *host_t,
                       const float *host_K, float *staging, float *host_image_out,
                       int64_t *host_counters_out) {
    if (!device_args || !host_q || !host_t || !host_K || !staging || !host_image_out) {
        set_error("render_host: null pointer argument");
        return GSB_EINVAL;
    }
    GsbForwardArgs a = *device_args;
    cudaStream_t st = static_cast<cudaStream_t>(a.stream);
    const int n = a.num_objects;
    float *d_q = staging, *d_t = staging + 4 * n, *d_K = staging + 7 * n;
    GSB_CUDA_CHECK(cudaMemcpyAsync(d_q, host_q, sizeof(float) * 4 * n, cudaMemcpyHostToDevice, st));
    GSB_CUDA_CHECK(cudaMemcpyAsync(d_t, host_t, sizeof(float) * 3 * n, cudaMemcpyHostToDevice, st));
    GSB_CUDA_CHECK(cudaMemcpyAsync(d_K, host_K, sizeof(float) * 9, cudaMemcpyHostToDevice, st));
    a.q_pointcloud_camera = d_q;
    a.t_pointcloud_camera = d_t;
    a.camera_intrinsics = d_K;
    int rc = gsb200_forward(&a);
    if (rc != GSB_OK) return rc;
    GSB_CUDA_CHECK(cudaMemcpyAsync(host_image_out, a.rasterized_image,
                                   sizeof(float) * 3 * (size_t)a.camera_height * a.camera_width,
                                   cudaMemcpyDeviceToHost, st));
    if (host_counters_out)
        GSB_CUDA_CHECK(cudaMemcpyAsync(host_counters_out, a.workspace, sizeof(int64_t) * 4,
                                       cudaMemcpyDeviceToHost, st));
    GSB_CUDA_CHECK(cudaStreamSynchronize(st));
    return GSB_OK;
}

}  // extern "C"
