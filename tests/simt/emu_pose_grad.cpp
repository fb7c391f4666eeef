// emu_pose_grad.cpp -- the per-point kernel of the backward with and without its pose epilogue (backward_points_kernel<*, POSE>)
// and the finalisation of the pose gradients (pose_grad_finalize_kernel), compiled as host C++ under simt_emu.h.
// TEST INFRASTRUCTURE, see simt_emu.h; built by tests/test_simt_pose_gradients_cpu.py with g++.
#include "simt_emu.h"
// the kernel sources, unmodified (their launchers are compiled out under GSB_HOST_EMU)
#include "../../taichi_3d_gaussian_splatting_b200/csrc/blend_bwd.cu"

namespace gsb {
void set_error(const char *, ...) {}
}  // namespace gsb

// emu_backward_points of emu_blend.cpp plus, with pose != 0, the POSE instantiation: pose_partials receives
// [blocks][n_obj][12] and grad_q (n_obj,4) / grad_t (n_obj,3) the finalised gradients.  The grid is
// min(ceil(N / 128), max_blocks) CTAs (the device launch caps it at 16 per SM); returns the number of CTAs.
extern "C" int emu_backward_points_pose(long long N, const int *point_offset, const float *records, const float *point_in_camera,
                                        const float *accum, const float *poses, const float *xyz, const float *features,
                                        const int *obj_id, const float *t_pc_cam, const float *K, int color_max_sh_band,
                                        float q_f, float s_f, float a_f, float c_f, float h_f, float *grad_xyz, float *grad_feat,
                                        float *grad_sum, float *grad_col, int *ctl_num_in_camera, int *ctl_num_pixels,
                                        float *ctl_vs_grad, float *ctl_vs_grad_avg, float *ctl_pos_grad,
                                        float *ctl_pos_grad_norm, int max_blocks, int pose, int n_obj, const float *q_pc,
                                        float *pose_partials, float *grad_q, float *grad_t) {
    using namespace gsb;
    PointsBwdParams p;
    p.N = N;
    p.point_offset = point_offset;
    p.records = reinterpret_cast<const float4 *>(records);
    p.point_in_camera = point_in_camera;
    p.accum = accum;
    p.poses = reinterpret_cast<const PoseBlock *>(poses);
    p.xyz = xyz;
    p.features = features;
    p.obj_id = obj_id;
    p.t_pc_cam = t_pc_cam;
    p.K = K;
    const int band = color_max_sh_band;
    p.first_cleared = band <= 0 ? 1 : band == 1 ? 4 : band == 2 ? 9 : 16;  // as launch_backward_points
    p.q_f = q_f;
    p.s_f = s_f;
    p.a_f = a_f;
    p.c_f = c_f;
    p.h_f = h_f;
    p.grad_xyz = grad_xyz;
    p.grad_feat = grad_feat;
    p.grad_sum_compact = grad_sum;
    p.grad_color_compact = grad_col;
    p.ctl_num_in_camera = ctl_num_in_camera;
    p.ctl_num_pixels = ctl_num_pixels;
    p.ctl_vs_grad = ctl_vs_grad;
    p.ctl_vs_grad_avg = ctl_vs_grad_avg;
    p.ctl_pos_grad = ctl_pos_grad;
    p.ctl_pos_grad_norm = ctl_pos_grad_norm;
    p.skip_flag = nullptr;
    p.pose_num_objects = pose ? n_obj : 0;
    p.pose_partials = pose ? pose_partials : nullptr;
    const int blocks = (int)std::min<long long>((N + GSB_POINTS_THREADS - 1) / GSB_POINTS_THREADS, max_blocks);
    const bool compact = grad_sum != nullptr;
    if (N > 0) {
        if (pose && compact) simt_emu::launch(backward_points_kernel<true, true>, blocks, GSB_POINTS_THREADS, p);
        else if (pose) simt_emu::launch(backward_points_kernel<false, true>, blocks, GSB_POINTS_THREADS, p);
        else if (compact) simt_emu::launch(backward_points_kernel<true>, blocks, GSB_POINTS_THREADS, p);
        else simt_emu::launch(backward_points_kernel<false>, blocks, GSB_POINTS_THREADS, p);
    }
    if (pose) {
        struct FinArgs {
            const float *partials;
            int blocks, n_obj;
            const float *q, *t;
            float *gq, *gt;
        } fa{pose_partials, N > 0 ? blocks : 0, n_obj, q_pc, t_pc_cam, grad_q, grad_t};
        simt_emu::launch([](const FinArgs &a) { pose_grad_finalize_kernel(a.partials, a.blocks, a.n_obj, a.q, a.t, a.gq, a.gt); },
                         n_obj, POSE_FINALIZE_THREADS, fa);
    }
    return N > 0 ? blocks : 0;
}
