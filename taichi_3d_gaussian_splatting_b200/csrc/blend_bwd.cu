// blend_bwd.cu -- backward of the blend (replaces gaussian_point_rasterisation_backward, GPCR:488-772).
//
// Kernel A (loop A, GPCR:531-705): one CTA per tile replays its splat list back-to-front.  The
// reference issues 11 global atomics per contributing (pixel, splat); here the 11 per-splat partials
// (d/duv x2, d/dcov x3, d/dcolour x3, d/dlogit, |d/duv|, pixel count) are reduced across the warp
// with a transposing butterfly (13 shuffles for all of them) and flushed with ONE 11-lane RED.ADD.F32
// per (warp patch, splat) -- per-warp culling (common.cuh) leaves ~2 of the 8 patches per (tile, splat).
// Kernel B (loop B, GPCR:708-772 + GPCR:1102-1125, 1167-1182): per in-frustum point chain rule to
// xyz / q / s / SH with the SH-band masking and the constant gradient factors fused in.
#include "blend_bwd.cuh"

namespace gsb {

// Reduce 11 per-lane values across the warp with 13 shuffles (transposing butterfly: at every stage a lane hands
// one half of its live values to its partner and keeps the other half, 11 -> 6 -> 3 -> 2 -> 1; the odd value of a
// stage is summed on both sides).  On return v[0] of lane l holds the warp total of value index
// reduce11_slot(l); the lanes for which reduce11_writer(l) is true cover 0..10 exactly once.
__device__ __forceinline__ void warp_transpose_reduce11(float (&v)[11], int lane) {
    {
        const bool hi = lane & 16;  // keeps values 6..10 (and a duplicate of 5), partner keeps 0..5
#pragma unroll
        for (int i = 0; i < 5; ++i) {
            const float send = hi ? v[i] : v[i + 6];
            const float keep = hi ? v[i + 6] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
        v[5] += __shfl_xor_sync(0xffffffffu, v[5], 16);
    }
    {
        const bool hi = lane & 8;  // slots 3..5 vs 0..2
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const float send = hi ? v[i] : v[i + 3];
            const float keep = hi ? v[i + 3] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
    }
    {
        const bool hi = lane & 4;  // slot 2 vs slot 0; slot 1 on both sides
        const float send = hi ? v[0] : v[2];
        const float keep = hi ? v[2] : v[0];
        v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
        v[1] += __shfl_xor_sync(0xffffffffu, v[1], 4);
    }
    {
        const bool hi = lane & 2;  // slot 1 vs slot 0
        const float send = hi ? v[0] : v[1];
        const float keep = hi ? v[1] : v[0];
        v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
    }
    v[0] += __shfl_xor_sync(0xffffffffu, v[0], 1);
}
__device__ __forceinline__ int reduce11_slot(int lane) {
    const int s2 = (lane & 2) ? 1 : ((lane & 4) ? 2 : 0);
    const int s1 = s2 + ((lane & 8) ? 3 : 0);
    return (lane & 16) ? (s1 == 5 ? 5 : s1 + 6) : s1;
}
__device__ __forceinline__ bool reduce11_writer(int lane) {
    if (lane & 1) return false;
    if ((lane & 2) && (lane & 4)) return false;         // slot 1 is duplicated over bit 2
    if ((lane & 16) && (lane & 8) && !(lane & 2) && (lane & 4)) return false;  // duplicate of value 5 in the upper half
    return true;
}


#ifndef GSB_BWD_MIN_BLOCKS
#define GSB_BWD_MIN_BLOCKS 4
#endif
// STATS = false (GSB_FLAG_NO_HOOK_STATS, opt-in): the |d/duv| magnitude, the affected-pixel count and the per-pixel magnitude
// image -- read only by a backward hook, the reference's need_extra_info (GPCR:521, 690-704) -- are not computed; slots 9 and
// 10 of the butterfly then carry zeros.
template <bool EXACT_EXP, bool STATS = true>
__global__ void __launch_bounds__(GSB_TILE_PIXELS, GSB_BWD_MIN_BLOCKS)
blend_backward_kernel(const BlendBwdParams p) {
    // double-buffered staging area: [buf][plane][splat]; planes: u v a b | c rescale opacity depth | r g b radius
    __shared__ float4 s_rec[2 * 3 * GSB_TILE_PIXELS];
    __shared__ int s_off[2][GSB_TILE_PIXELS];
    constexpr int PLANE = GSB_TILE_PIXELS * 16;
    __shared__ unsigned int s_bits[2][8][8];  // [buf][consumer warp patch][loader warp]
    __shared__ int s_max_last;

    const int tile = blockIdx.x;
    const int tu = tile % p.tiles_x, tv = tile / p.tiles_x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int pu = tu * GSB_TILE_WIDTH + (warp & 1) * 8 + (lane & 7);
    const int pv = tv * GSB_TILE_HEIGHT + (warp >> 1) * 4 + (lane >> 3);
    const float px = (float)pu + 0.5f, py = (float)pv + 0.5f;
    const float tile_x0 = (float)(tu * GSB_TILE_WIDTH), tile_y0 = (float)(tv * GSB_TILE_HEIGHT);
    const size_t pix = (size_t)pv * p.W + pu;
    const int start = p.tile_start[tile];

    const int last = p.last_effective[pix];
    float T = 1.0f - p.acc_alpha[pix];  // GPCR:559-560
    float w0 = 0.0f, w1 = 0.0f, w2 = 0.0f;
    const float g0 = p.grad_image[3 * pix], g1 = p.grad_image[3 * pix + 1], g2 = p.grad_image[3 * pix + 2];
    float mag0 = 0.0f, mag1 = 0.0f;
    const unsigned int sa = smem_u32(s_rec);
    const int red_slot = reduce11_slot(lane);
    const bool red_writer = reduce11_writer(lane);

    // deepest effective splat of this warp's patch and of the whole tile (GPCR:609-610: nothing at or
    // behind a pixel's last effective offset contributes to it)
    int warp_last = last;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) warp_last = max(warp_last, __shfl_xor_sync(0xffffffffu, warp_last, d));
    if (tid == 0) s_max_last = start;
    __syncthreads();
    if (lane == 0) atomicMax(&s_max_last, warp_last);
    __syncthreads();
    const int end = min(p.tile_end[tile], s_max_last);

    // One barrier per batch (double-buffered staging, see blend_fwd.cu).
    int buf = 0;
    for (int block_end = end; block_end > start; block_end -= GSB_TILE_PIXELS, buf ^= 1) {
        const int block_start = max(block_end - GSB_TILE_PIXELS, start);
        float4 *const s_r0 = s_rec + buf * 3 * GSB_TILE_PIXELS;
        float4 *const s_r1 = s_r0 + GSB_TILE_PIXELS, *const s_r2 = s_r0 + 2 * GSB_TILE_PIXELS;
        {
            const int idx = block_end - 1 - tid;  // element j <-> sorted index block_end-1-j
            unsigned int mask = 0;
            if (idx >= block_start) {
                const int o = __ldg(&p.sorted_vals[idx]);
                const float4 *rec = p.records + 3 * (size_t)o;
                const float4 r0 = __ldg(rec), r1 = __ldg(rec + 1);
                s_r0[tid] = r0;
                // fast path: the loop needs rescale*opacity and 1-opacity, not the two factors
                s_r1[tid] = EXACT_EXP ? r1 : make_float4(r1.x, r1.y * r1.z, 1.0f - r1.z, r1.w);
                s_r2[tid] = __ldg(rec + 2);
                s_off[buf][tid] = o;
                mask = splat_patch_mask(r0.x, r0.y, r0.z, r0.w, r1.x, r1.y * r1.z, tile_x0, tile_y0);
            }
#pragma unroll
            for (int w = 0; w < 8; ++w) {
                const unsigned int bits = __ballot_sync(0xffffffffu, (mask >> w) & 1u);
                if (lane == 0) s_bits[buf][w][warp] = bits;
            }
        }
        __syncthreads();
        const unsigned int sb = sa + buf * (3 * PLANE);
        if (block_start < warp_last) {  // otherwise every splat of this batch is behind the whole patch
            // element j <-> sorted index block_end-1-j: the first `skip` elements of the batch lie at or behind the
            // patch's deepest effective splat and are dropped from the bit lists wholesale (warp-uniform)
            const int skip = block_end - warp_last;
#pragma unroll 1
            for (int lw = skip > 0 ? (skip >> 5) : 0; lw < 8; ++lw) {
                unsigned int bits = s_bits[buf][warp][lw];
                if (skip > lw * 32) bits &= ~((1u << (skip - lw * 32)) - 1u);  // 0 < skip - 32 lw < 32 here
                while (bits) {
                    const int j = lw * 32 + __ffs(bits) - 1;
                    bits &= bits - 1;
                    const int idx = block_end - 1 - j;
                    float v[11];
                    bool contributes;
                    // Branch-free: every lane evaluates the splat; lanes that do not contribute (behind their
                    // last effective splat, or alpha < 1/255) get zero weights, so all partials vanish and the
                    // pixel state is left untouched by predicated selects.
                    {
                        const unsigned int ja = sb + j * 16;
                        const float4 r0 = lds128<0>(ja);          // u v a b
                        const float4 r1 = lds128<PLANE>(ja);      // c rescale opacity depth
                        const float4 r2 = lds128<2 * PLANE>(ja);  // r g b radius
                        const float d0 = px - r0.x, d1 = py - r0.y;
                        const float q0 = r0.z * d0 + r0.w * d1;
                        const float q1 = r0.w * d0 + r1.x * d1;
                        if (EXACT_EXP) {
                            const float gp = expf(-0.5f * (d0 * q0 + d1 * q1)) * r1.y;
                            const float opa = r1.z;
                            const float prod_alpha = gp * opa;
                            contributes = (idx < last) && (prod_alpha >= 1.0f / 255.0f);
                            const float alpha = fminf(prod_alpha, 0.99f);
                            const float inv = 1.0f / (1.0f - alpha);
                            const float Tn = T * inv;
                            const float aT = contributes ? alpha * Tn : 0.0f;
                            const float a_grad = contributes ? (r2.x * Tn - w0 * inv) * g0 + (r2.y * Tn - w1 * inv) * g1 +
                                                                   (r2.z * Tn - w2 * inv) * g2
                                                             : 0.0f;
                            T = contributes ? Tn : T;
                            w0 = fmaf(r2.x, aT, w0);
                            w1 = fmaf(r2.y, aT, w1);
                            w2 = fmaf(r2.z, aT, w2);
                            const float G = a_grad * opa * gp;
                            const float vs0 = G * q0, vs1 = G * q1;
                            if (STATS) {
                                mag0 += fabsf(vs0);
                                mag1 += fabsf(vs1);
                            }
                            v[0] = vs0;
                            v[1] = vs1;
                            v[2] = vs0 * q0;  // the 1/2 of UT:345 is applied once per point in the epilogue
                            v[3] = vs0 * q1;
                            v[4] = vs1 * q1;
                            v[5] = aT * g0;
                            v[6] = aT * g1;
                            v[7] = aT * g2;
                            v[8] = a_grad * gp * (1.0f - opa) * opa;
                            v[9] = STATS ? sqrtf(vs0 * vs0 + vs1 * vs1) : 0.0f;
                        } else {
                            // r1 = c | rescale*opacity | 1-opacity | depth.  The colour recursion of GPCR:653-657,
                            // sum_c (col_c T - w_c/(1-a)) g_c, is carried as ONE scalar: with cg = sum_c col_c g_c and
                            // w0 = sum_c w_c g_c it is  cg T - w0/(1-a),  and w0 += cg a T.
                            // alpha exactly as the forward computes it (fast_alpha on the forward's pre-scaled conic, common.cuh): both
                            // passes take the alpha >= 1/255 decision on identical bits
                            const float P = fast_alpha(d0, d1, (-0.5f * GSB_L2E) * r0.z, -GSB_L2E * r0.w,
                                                       (-0.5f * GSB_L2E) * r1.x, r1.y);
                            contributes = (idx < last) && (P >= 1.0f / 255.0f);
                            const float alpha = fminf(P, 0.99f);
                            const float inv = rcp_approx(1.0f - alpha);
                            const float Tn = T * inv;
                            const float aT = contributes ? alpha * Tn : 0.0f;
                            const float cg = fmaf(r2.z, g2, fmaf(r2.y, g1, r2.x * g0));
                            const float a_grad = contributes ? fmaf(cg, Tn, -(w0 * inv)) : 0.0f;
                            T = contributes ? Tn : T;
                            w0 = fmaf(cg, aT, w0);
                            const float G = a_grad * P;  // d L / d gaussian exponent weight: a_grad * opacity * p
                            const float vs0 = G * q0, vs1 = G * q1;
                            if (STATS) {
                                mag0 += fabsf(vs0);
                                mag1 += fabsf(vs1);
                            }
                            v[0] = vs0;
                            v[1] = vs1;
                            v[2] = vs0 * q0;
                            v[3] = vs0 * q1;
                            v[4] = vs1 * q1;
                            v[5] = aT * g0;
                            v[6] = aT * g1;
                            v[7] = aT * g2;
                            v[8] = G * r1.z;  // a_grad * p * opacity * (1 - opacity)
                            v[9] = STATS ? sqrt_approx(vs0 * vs0 + vs1 * vs1) : 0.0f;
                        }
                        v[10] = (STATS && contributes) ? 1.0f : 0.0f;
                    }
                    if (lane == 0) GSB_EMU_COUNT(EC_BF_VISITS, 1);
                    GSB_EMU_COUNT(EC_BF_PAIRS, contributes ? 1 : 0);
                    if (__any_sync(0xffffffffu, contributes)) {
                        if (lane == 0) GSB_EMU_COUNT(EC_BF_VISITS_ANY, 1);
                        // 11 partials of this (warp, splat) -> 11 lanes -> one RED.ADD.F32 row update
                        warp_transpose_reduce11(v, lane);
                        if (red_writer && (STATS || red_slot < 9))
                            atomicAdd(p.accum + (size_t)s_off[buf][j] * GSB_ACCUM_FLOATS + red_slot, v[0]);
                    }
                }
            }
        }
    }
    if (STATS) {
        p.mag_image[2 * pix] = mag0;  // GPCR:700-704
        p.mag_image[2 * pix + 1] = mag1;
    }
}

#ifndef GSB_HOST_EMU
static BlendBwdParams make_blend_bwd_params(const GsbBackwardArgs &a, const Workspace &ws);

int launch_blend_backward_work(const GsbBackwardArgs &a, const Workspace &ws, unsigned long long *counters_dev,
                               cudaStream_t stream) {
    BlendBwdParams p = make_blend_bwd_params(a, ws);
    p.work_counters = counters_dev;
    const int tiles = p.tiles_x * (a.camera_height / GSB_TILE_HEIGHT);
    if (tiles <= 0) return GSB_OK;
    return launch_blend_backward_count(p, tiles, stream);
}

static BlendBwdParams make_blend_bwd_params(const GsbBackwardArgs &a, const Workspace &ws) {
    BlendBwdParams p;
    p.H = a.camera_height;
    p.W = a.camera_width;
    p.tiles_x = a.camera_width / GSB_TILE_WIDTH;
    p.tile_start = ws.tile_start;
    p.tile_end = ws.tile_end;
    p.sorted_vals = ws.vals_b;  // the sort always ends in b
    p.records = ws.records;
    p.grad_image = a.grad_rasterized_image;
    p.acc_alpha = a.pixel_accumulated_alpha;
    p.last_effective = a.pixel_offset_of_last_effective_point;
    p.patch_masks = ws.patch_masks;
    p.accum = a.accum;
    p.mag_image = a.magnitude_grad_viewspace_on_image;
    p.work_counters = nullptr;
    return p;
}

int launch_blend_backward(const GsbBackwardArgs &a, const Workspace &ws, cudaStream_t stream) {
    BlendBwdParams p;
    p.H = a.camera_height;
    p.W = a.camera_width;
    p.tiles_x = a.camera_width / GSB_TILE_WIDTH;
    p.tile_start = ws.tile_start;
    p.tile_end = ws.tile_end;
    p.sorted_vals = ws.vals_b;  // the sort always ends in b
    p.records = ws.records;
    p.grad_image = a.grad_rasterized_image;
    p.acc_alpha = a.pixel_accumulated_alpha;
    p.last_effective = a.pixel_offset_of_last_effective_point;
    p.patch_masks = ws.patch_masks;
    p.accum = a.accum;
    p.mag_image = a.magnitude_grad_viewspace_on_image;
    p.work_counters = nullptr;
    const int tiles = p.tiles_x * (a.camera_height / GSB_TILE_HEIGHT);
    if (tiles <= 0) return GSB_OK;
    if (a.flags & GSB_FLAG_BACKWARD_TRANSPOSED)  // experimental, see blend_bwd_transposed.cu
        return launch_blend_backward_transposed(p, tiles, (a.flags & GSB_FLAG_EXACT_EXP) != 0,
                                                (a.flags & GSB_FLAG_NO_HOOK_STATS) == 0, stream);
    const bool exact = (a.flags & GSB_FLAG_EXACT_EXP) != 0;
    if (a.flags & GSB_FLAG_NO_HOOK_STATS) {  // opt-in
        if (exact) blend_backward_kernel<true, false><<<tiles, GSB_TILE_PIXELS, 0, stream>>>(p);
        else blend_backward_kernel<false, false><<<tiles, GSB_TILE_PIXELS, 0, stream>>>(p);
    } else if (exact) {
        blend_backward_kernel<true><<<tiles, GSB_TILE_PIXELS, 0, stream>>>(p);
    } else {
        blend_backward_kernel<false><<<tiles, GSB_TILE_PIXELS, 0, stream>>>(p);
    }
    GSB_CUDA_CHECK(cudaGetLastError());
    return GSB_OK;
}
#endif  // GSB_HOST_EMU

// ------------------------------------------------------------------ loop B + P4
// Real SH basis up to band 3 along the (un-normalised) direction (dx, dy, dz)  (SH:10-32; GPCR:731-732, 749)
__device__ __forceinline__ void sh_basis(float dx, float dy, float dz, float (&sh)[16]) {
    const float dinv = 1.0f / sqrtf(dx * dx + dy * dy + dz * dz);
    dx *= dinv; dy *= dinv; dz *= dinv;
    sh[0] = 0.28209479177387814f;
    sh[1] = -0.48860251190291987f * dy;
    sh[2] = 0.48860251190291987f * dz;
    sh[3] = -0.48860251190291987f * dx;
    sh[4] = 1.0925484305920792f * dx * dy;
    sh[5] = -1.0925484305920792f * dy * dz;
    sh[6] = 0.94617469575755997f * dz * dz - 0.31539156525251999f;
    sh[7] = -1.0925484305920792f * dx * dz;
    sh[8] = 0.54627421529603959f * dx * dx - 0.54627421529603959f * dy * dy;
    sh[9] = 0.59004358992664352f * dy * (-3.0f * dx * dx + dy * dy);
    sh[10] = 2.8906114426405538f * dx * dy * dz;
    sh[11] = 0.45704579946446572f * dy * (1.0f - 5.0f * dz * dz);
    sh[12] = 0.3731763325901154f * dz * (5.0f * dz * dz - 3.0f);
    sh[13] = 0.45704579946446572f * dx * (1.0f - 5.0f * dz * dz);
    sh[14] = 1.4453057213202769f * dz * (dx * dx - dy * dy);
    sh[15] = 0.59004358992664352f * dx * (-dx * dx + 3.0f * dy * dy);
}

struct PointsBwdParams {
    long long N;
    const int *point_offset;
    const float4 *records;
    const float *point_in_camera;
    const float *accum;
    const PoseBlock *poses;
    const float *xyz;
    const float *features;
    const int *obj_id;
    const float *t_pc_cam;
    const float *K;
    int first_cleared;  // first SH coefficient index whose gradient is zeroed (GPCR:1167-1182)
    float q_f, s_f, a_f, c_f, h_f;
    float *grad_xyz;
    float *grad_feat;
    // optional: the densification controller's accumulators, updated in this epilogue (GaussianPointAdaptiveController.py:130-143)
    int *ctl_num_in_camera;     // (N) or nullptr = not fused
    int *ctl_num_pixels;        // (N)
    float *ctl_vs_grad;         // (N)   accumulated_view_space_position_gradients
    float *ctl_vs_grad_avg;     // (N)   accumulated_view_space_position_gradients_avg
    float *ctl_pos_grad;        // (N,3) accumulated_position_gradients
    float *ctl_pos_grad_norm;   // (N)   accumulated_position_gradients_norm
    const long long *skip_flag; // optional device flag (the frame's key-capacity overflow counter): non-zero = leave the
                                //   controller accumulators alone (fused train step: the whole step becomes a no-op)
    float *grad_sum_compact;    // COMPACT: (N,12) xyz(3) q(4) s(3) logit(1) pad -- the columns that simply add up over views
    float *grad_color_compact;  // COMPACT: (N,3) d L / d (SH colour argument), per VIEW (its SH basis depends on the camera centre)
    // POSE: per-CTA sums of the 12 pose values of every object -> pose_partials[block][obj][12] (pose_grad_finalize_kernel)
    int pose_num_objects;       // <= GSB_POSE_MAX_OBJECTS
    float *pose_partials;
};

// Sum 12 per-lane values over the warp with 13 shuffles (the transposing butterfly of warp_transpose_reduce11 with an even
// split at every stage: 12 -> 6 -> 3 -> 2 -> 1).  On return v[0] of lane l holds the warp total of value reduce12_slot(l);
// the lanes for which reduce12_writer(l) is true cover 0..11 exactly once.  Fixed shuffle pattern: deterministic.
__device__ __forceinline__ void warp_transpose_reduce12(float (&v)[12], int lane) {
    {
        const bool hi = lane & 16;  // keeps values 6..11, partner keeps 0..5
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            const float send = hi ? v[i] : v[i + 6];
            const float keep = hi ? v[i + 6] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
    }
    {
        const bool hi = lane & 8;  // slots 3..5 vs 0..2
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const float send = hi ? v[i] : v[i + 3];
            const float keep = hi ? v[i + 3] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
    }
    {
        const bool hi = lane & 4;  // slot 2 vs slot 0; slot 1 on both sides
        const float send = hi ? v[0] : v[2];
        const float keep = hi ? v[2] : v[0];
        v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
        v[1] += __shfl_xor_sync(0xffffffffu, v[1], 4);
    }
    {
        const bool hi = lane & 2;  // slot 1 vs slot 0
        const float send = hi ? v[0] : v[1];
        const float keep = hi ? v[1] : v[0];
        v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
    }
    v[0] += __shfl_xor_sync(0xffffffffu, v[0], 1);
}
__device__ __forceinline__ int reduce12_slot(int lane) {
    return ((lane & 16) ? 6 : 0) + ((lane & 8) ? 3 : 0) + ((lane & 2) ? 1 : ((lane & 4) ? 2 : 0));
}
__device__ __forceinline__ bool reduce12_writer(int lane) { return !(lane & 1) && !((lane & 2) && (lane & 4)); }

#ifndef GSB_POINTS_THREADS
#define GSB_POINTS_THREADS 128
#endif
constexpr int PT_ROW = 60;  // staged feature row stride in floats: 16-B aligned, float4 stores of 8 lanes hit 32 banks
constexpr int PT_ROW_COMPACT = 20;  // COMPACT: 16 staged floats per row, same bank property
// COMPACT = true (GSB_FLAG_COMPACT_GRADS, the view-parallel exchange of parallel.py): instead of the dense (N,3) / (N,56)
// gradients the kernel writes, per scene row, the 11 values that add up over views -- xyz(3) q(4) s(3) logit(1), factors
// applied -- and the 3 colour-argument gradients that must stay per view: the 48 SH gradients of a view are their outer product
// with the view's SH basis, which gsb200_expand_view_gradients rebuilds AFTER the exchange (14 instead of 59 floats per row
// cross NVLink, and this kernel writes 60 instead of 236 bytes per row).
// POSE = true (gsb200_backward_with_pose): every in-frustum row also forms the 12 values through which the pose of its object
// reaches the image under the same surrogate as the xyz gradient (DESIGN.md section 9): dL/dt_c (3) and dL/dW (9), with
// p_cam = W x + t_c.  They are summed per object in a fixed order -- lanes grouped by object (__match_any_sync) and folded with
// a fixed shuffle butterfly, groups added into per-warp shared slots, the warps added in warp order at the end of the CTA --
// and written as pose_partials[block][obj][12]; pose_grad_finalize_kernel adds the blocks and applies the chain rule to (q, t).
// Every other output is computed by the same code as with POSE = false.
template <bool COMPACT, bool POSE = false>
__global__ void __launch_bounds__(GSB_POINTS_THREADS, 6)  // 6 x 33 KB of staging per SM (+3 KB of pose slots with POSE)
backward_points_kernel(const PointsBwdParams p) {
    // One thread per scene row: rows outside the frustum get their zeros here (no separate memset of the
    // dense (N,3)/(N,56) gradients), rows inside get the chain rule.  A warp owns 32 consecutive rows, i.e. one
    // contiguous 7 KB piece of the (N,56) gradient and 384 B of the (N,3) one: each lane stages its row in
    // shared memory and the warp then streams the piece out with full 512-B stores (a lane writing its own
    // 224-B row directly touches 32 different lines per store instruction and stalls on the LSU queue).
    constexpr int ROW = COMPACT ? PT_ROW_COMPACT : PT_ROW;
    __shared__ __align__(16) float s_feat[GSB_POINTS_THREADS / 32][32 * ROW];
    __shared__ float s_xyz[GSB_POINTS_THREADS / 32][96];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float *const my_feat = &s_feat[warp][lane * ROW];
    float *const my_xyz = &s_xyz[warp][lane * 3];
    __shared__ float s_pose[POSE ? GSB_POINTS_THREADS / 32 : 1][POSE ? GSB_POSE_MAX_OBJECTS : 1][12];
    if (POSE) {  // each warp clears and later fills only its own slots
        for (int k = lane; k < p.pose_num_objects * 12; k += 32) s_pose[warp][k / 12][k % 12] = 0.0f;
        __syncwarp();
    }
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long base = (long long)blockIdx.x * blockDim.x + warp * 32; base < p.N; base += stride) {
      const long long id = base + lane;
      const int o = id < p.N ? p.point_offset[id] : -1;
      int pose_obj = -1;  // POSE: object of this lane's row if it is in the frustum
      float pv[12];       // POSE: dL/dt_c (3) | dL/dW row-major (9) of this row
      if (o < 0) {
          if (!COMPACT) { my_xyz[0] = 0.0f; my_xyz[1] = 0.0f; my_xyz[2] = 0.0f; }
#pragma unroll
          for (int k = 0; k < (COMPACT ? 4 : GSB_FEATURE_DIM / 4); ++k)
              reinterpret_cast<float4 *>(my_feat)[k] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      } else {
        const float4 *accp = reinterpret_cast<const float4 *>(p.accum + (size_t)o * GSB_ACCUM_FLOATS);
        const float4 a0 = accp[0], a1 = accp[1], a2 = accp[2];
        // a0 = guv.x guv.y g00 g01 | a1 = g11 gr gg gb | a2 = glogit mag n pad
        const float4 r2 = __ldg(p.records + 3 * (size_t)o + 2);  // r g b radius
        const float pcx = p.point_in_camera[3 * o], pcy = p.point_in_camera[3 * o + 1],
                    pcz = p.point_in_camera[3 * o + 2];
        const int ob = p.obj_id[id];
        const PoseBlock *pb = p.poses + ob;
        float Wm[9] = {pb->T[0], pb->T[1], pb->T[2], pb->T[4], pb->T[5], pb->T[6], pb->T[8], pb->T[9], pb->T[10]};
        float Kc[9];
#pragma unroll
        for (int k = 0; k < 9; ++k) Kc[k] = __ldg(&p.K[k]);
        const float x = p.xyz[3 * (size_t)id], y = p.xyz[3 * (size_t)id + 1], z = p.xyz[3 * (size_t)id + 2];
        const float4 *frow = reinterpret_cast<const float4 *>(p.features + (size_t)GSB_FEATURE_DIM * id);
        const float4 qv = __ldg(frow);
        const float4 sv = __ldg(frow + 1);  // s0 s1 s2 logit

        // d uv / d xyz (GP3D:132-159): full-K projection Jacobian times W
        const float iz = 1.0f / pcz, iz2 = iz * iz;
        float dj[6] = {Kc[0] * iz, Kc[1] * iz, (-Kc[0] * pcx - Kc[1] * pcy) * iz2,
                       Kc[3] * iz, Kc[4] * iz, (-Kc[3] * pcx - Kc[4] * pcy) * iz2};
        float gx[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float d0 = dj[0] * Wm[c] + dj[1] * Wm[3 + c] + dj[2] * Wm[6 + c];
            const float d1 = dj[3] * Wm[c] + dj[4] * Wm[3 + c] + dj[5] * Wm[6 + c];
            gx[c] = a0.x * d0 + a0.y * d1;
        }
        // Sigma' = U Sigma U^T, U = J W with J from fx, fy only (GP3D:65-87, 237-331)
        const float fx = Kc[0], fy = Kc[4];
        float J[6] = {fx * iz, 0.0f, -(fx * pcx) * iz2, 0.0f, fy * iz, -(fy * pcy) * iz2};
        float U[6];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            U[c] = J[0] * Wm[c] + J[1] * Wm[3 + c] + J[2] * Wm[6 + c];
            U[3 + c] = J[3] * Wm[c] + J[4] * Wm[3 + c] + J[5] * Wm[6 + c];
        }
        const float g00 = 0.5f * a0.z, g01 = 0.5f * a0.w, g11 = 0.5f * a1.x;  // UT:345's 1/2, see the blend loop
        // V = U^T G U  (dL/dSigma with the (g00,g01,g01,g11) weighting of GPCR:716-721)
        float V[9];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float t0 = g00 * U[k] + g01 * U[3 + k];
            const float t1 = g01 * U[k] + g11 * U[3 + k];
#pragma unroll
            for (int l = 0; l < 3; ++l) V[k * 3 + l] = t0 * U[l] + t1 * U[3 + l];
        }
        // R(q) (GP3D:30-48), M = R S
        const float qx = qv.x, qy = qv.y, qz = qv.z, qw = qv.w;
        float R[9];
        R[0] = 1 - 2 * (qy * qy + qz * qz); R[1] = 2 * (qx * qy - qw * qz); R[2] = 2 * (qx * qz + qw * qy);
        R[3] = 2 * (qx * qy + qw * qz); R[4] = 1 - 2 * (qx * qx + qz * qz); R[5] = 2 * (qy * qz - qw * qx);
        R[6] = 2 * (qx * qz - qw * qy); R[7] = 2 * (qy * qz + qw * qx); R[8] = 1 - 2 * (qx * qx + qy * qy);
        const float es[3] = {expf(sv.x), expf(sv.y), expf(sv.z)};
        // dL/dM = (V + V^T) M,  M_ij = R_ij es_j
        float dM[9];
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = 0; b < 3; ++b) {
                float acc = 0.0f;
#pragma unroll
                for (int l = 0; l < 3; ++l) acc += (V[a * 3 + l] + V[l * 3 + a]) * (R[l * 3 + b] * es[b]);
                dM[a * 3 + b] = acc;
            }
        // d/ds_j = sum_i dM_ij R_ij es_j
        float gs[3];
#pragma unroll
        for (int j = 0; j < 3; ++j) gs[j] = (dM[j] * R[j] + dM[3 + j] * R[3 + j] + dM[6 + j] * R[6 + j]) * es[j];
        // d/dq = sum_ij dM_ij es_j dR_ij/dq  (table GP3D:316-329)
        const float sx = es[0], sy = es[1], sz = es[2];
        float gq[4];
        gq[0] = dM[1] * (2 * sy * qy) + dM[2] * (2 * sz * qz) + dM[3] * (2 * sx * qy) + dM[4] * (-4 * sy * qx) +
                dM[5] * (-2 * sz * qw) + dM[6] * (2 * sx * qz) + dM[7] * (2 * sy * qw) + dM[8] * (-4 * sz * qx);
        gq[1] = dM[0] * (-4 * sx * qy) + dM[1] * (2 * sy * qx) + dM[2] * (2 * sz * qw) + dM[3] * (2 * sx * qx) +
                dM[5] * (2 * sz * qz) + dM[6] * (-2 * sx * qw) + dM[7] * (2 * sy * qz) + dM[8] * (-4 * sz * qy);
        gq[2] = dM[0] * (-4 * sx * qz) + dM[1] * (-2 * sy * qw) + dM[2] * (2 * sz * qx) + dM[3] * (2 * sx * qw) +
                dM[4] * (-4 * sy * qz) + dM[5] * (2 * sz * qy) + dM[6] * (2 * sx * qx) + dM[7] * (2 * sy * qy);
        gq[3] = dM[1] * (-2 * sy * qz) + dM[2] * (2 * sz * qy) + dM[3] * (2 * sx * qz) + dM[5] * (-2 * sz * qx) +
                dM[6] * (-2 * sx * qy) + dM[7] * (2 * sy * qx);
        // sigmoid'(.) from the stored colour: c (1 - c)  (UT:356-359)
        const float gcol[3] = {a1.y * (r2.x * (1.0f - r2.x)), a1.z * (r2.y * (1.0f - r2.y)),
                               a1.w * (r2.z * (1.0f - r2.z))};
        if (p.ctl_num_in_camera != nullptr && !(p.skip_flag != nullptr && *p.skip_flag != 0)) {
            // GaussianPointAdaptiveController.update (:130-143) for this in-camera point: ids are unique, one thread per row,
            // so plain read-modify-writes.  a2.y = sum |d/duv| over pixels, a2.z = number of affected pixels (exact in f32)
            const int npix = __float2int_rn(a2.z);
            p.ctl_num_in_camera[id] += 1;
            p.ctl_num_pixels[id] += npix;
            p.ctl_vs_grad[id] += a2.y;
            float avg = a2.y / (float)npix;  // 0/0 -> NaN -> 0; x/0 stays inf like the reference
            if (avg != avg) avg = 0.0f;
            p.ctl_vs_grad_avg[id] += avg;
            p.ctl_pos_grad[3 * id] += gx[0];
            p.ctl_pos_grad[3 * id + 1] += gx[1];
            p.ctl_pos_grad[3 * id + 2] += gx[2];
            p.ctl_pos_grad_norm[id] += sqrtf(gx[0] * gx[0] + gx[1] * gx[1] + gx[2] * gx[2]);
        }
        if (POSE) {
            // mean: dL/dp_cam = dj^T guv;  dL/dt_c = dL/dp_cam,  dL/dW += dL/dp_cam (x) xyz
            // covariance (J held fixed): Sigma' = J W Sigma W^T J^T  ->  dL/dW += 2 J^T G U Sigma,  Sigma = R diag(es^2) R^T
            pose_obj = ob;
#pragma unroll
            for (int r = 0; r < 3; ++r) pv[r] = a0.x * dj[r] + a0.y * dj[3 + r];
            float B0[3], B1[3];  // (G U Sigma) rows
            {
                float A0[3], A1[3];  // (G U R diag(es^2)) rows
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    float u0 = 0.0f, u1 = 0.0f;
#pragma unroll
                    for (int l = 0; l < 3; ++l) {
                        u0 += (g00 * U[l] + g01 * U[3 + l]) * R[l * 3 + j];
                        u1 += (g01 * U[l] + g11 * U[3 + l]) * R[l * 3 + j];
                    }
                    const float e2 = es[j] * es[j];
                    A0[j] = u0 * e2;
                    A1[j] = u1 * e2;
                }
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    B0[c] = A0[0] * R[c * 3] + A0[1] * R[c * 3 + 1] + A0[2] * R[c * 3 + 2];
                    B1[c] = A1[0] * R[c * 3] + A1[1] * R[c * 3 + 1] + A1[2] * R[c * 3 + 2];
                }
            }
            const float xv[3] = {x, y, z};
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                pv[3 + c] = pv[0] * xv[c] + 2.0f * (J[0] * B0[c]);
                pv[6 + c] = pv[1] * xv[c] + 2.0f * (J[4] * B1[c]);
                pv[9 + c] = pv[2] * xv[c] + 2.0f * (J[2] * B0[c] + J[5] * B1[c]);
            }
        }
        if (COMPACT) {
            float4 *gc = reinterpret_cast<float4 *>(my_feat);
            gc[0] = make_float4(gx[0], gx[1], gx[2], gq[0] * p.q_f);
            gc[1] = make_float4(gq[1] * p.q_f, gq[2] * p.q_f, gq[3] * p.q_f, gs[0] * p.s_f);
            gc[2] = make_float4(gs[1] * p.s_f, gs[2] * p.s_f, a2.x * p.a_f, 0.0f);
            gc[3] = make_float4(gcol[0], gcol[1], gcol[2], 0.0f);
        } else {
        // SH basis along xyz - camera centre (GPCR:731-732, 749; SH:10-32)
        float sh[16];
        sh_basis(x - p.t_pc_cam[3 * ob], y - p.t_pc_cam[3 * ob + 1], z - p.t_pc_cam[3 * ob + 2], sh);

        my_xyz[0] = gx[0]; my_xyz[1] = gx[1]; my_xyz[2] = gx[2];
        float4 *gf = reinterpret_cast<float4 *>(my_feat);
        gf[0] = make_float4(gq[0] * p.q_f, gq[1] * p.q_f, gq[2] * p.q_f, gq[3] * p.q_f);
        gf[1] = make_float4(gs[0] * p.s_f, gs[1] * p.s_f, gs[2] * p.s_f, a2.x * p.a_f);
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            float o16[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                const float factor = k == 0 ? p.c_f : p.h_f;
                o16[k] = k < p.first_cleared ? gcol[ch] * sh[k] * factor : 0.0f;
            }
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4)
                gf[2 + 4 * ch + k4] = make_float4(o16[4 * k4], o16[4 * k4 + 1], o16[4 * k4 + 2], o16[4 * k4 + 3]);
        }
        }
      }
      if (POSE) {
          // one fold per object present in the warp's 32 rows, lowest lane's object first
          const unsigned int group = __match_any_sync(0xffffffffu, pose_obj);
          unsigned int todo = __ballot_sync(0xffffffffu, pose_obj >= 0);
          while (todo) {
              const int leader = __ffs(todo) - 1;
              const int obj = __shfl_sync(0xffffffffu, pose_obj, leader);
              todo &= ~__shfl_sync(0xffffffffu, group, leader);
              const bool mine = pose_obj == obj;
              float v[12];
#pragma unroll
              for (int k = 0; k < 12; ++k) v[k] = mine ? pv[k] : 0.0f;
              warp_transpose_reduce12(v, lane);
              if (reduce12_writer(lane)) s_pose[warp][obj][reduce12_slot(lane)] += v[0];
          }
      }
      __syncwarp();
      const long long rows = p.N - base < 32 ? p.N - base : 32;
      if (COMPACT) {
          // 32 rows -> 3 x 512 B of summable columns, 3 x 128 B of per-view colour gradients
          float4 *const out_s = reinterpret_cast<float4 *>(p.grad_sum_compact + 12 * (size_t)base);
          float *const out_c = p.grad_color_compact + 3 * (size_t)base;
#pragma unroll
          for (int it = 0; it < 3; ++it) {
              const int f = it * 32 + lane;
              const int row = f / 3, c = f - row * 3;
              if (row < rows) {
                  out_s[f] = *reinterpret_cast<const float4 *>(&s_feat[warp][row * ROW + 4 * c]);
                  out_c[f] = s_feat[warp][row * ROW + 12 + c];
              }
          }
      } else {
      // stream the warp's 32 rows out: 14 x 512 B of feature gradients, 3 x 128 B of position gradients
      float4 *const out_f = reinterpret_cast<float4 *>(p.grad_feat + (size_t)GSB_FEATURE_DIM * base);
#pragma unroll
      for (int it = 0; it < GSB_FEATURE_DIM / 4; ++it) {
          const int f = it * 32 + lane;           // float4 index inside the piece
          const int row = f / (GSB_FEATURE_DIM / 4), c4 = f - row * (GSB_FEATURE_DIM / 4);
          if (row < rows) out_f[f] = *reinterpret_cast<const float4 *>(&s_feat[warp][row * ROW + 4 * c4]);
      }
      float *const out_x = p.grad_xyz + 3 * (size_t)base;
#pragma unroll
      for (int it = 0; it < 3; ++it) {
          const int f = it * 32 + lane;
          if (f < 3 * rows) out_x[f] = s_xyz[warp][f];
      }
      }
      __syncwarp();
    }
    if (POSE) {  // the CTA's sums, warps added in warp order
        __syncthreads();
        for (int k = threadIdx.x; k < p.pose_num_objects * 12; k += blockDim.x) {
            float acc = s_pose[0][k / 12][k % 12];
#pragma unroll
            for (int w = 1; w < GSB_POINTS_THREADS / 32; ++w) acc += s_pose[w][k / 12][k % 12];
            p.pose_partials[(size_t)blockIdx.x * p.pose_num_objects * 12 + k] = acc;
        }
    }
}

// d/d(x,y,z,w) of sum_ab G_ab R_ab for the rotation polynomial R(x,y,z,w) of GP3D:30-48 (no normalisation)
__device__ __forceinline__ void rotation_polynomial_vjp(float x, float y, float z, float w, const float (&G)[9], float (&g)[4]) {
    g[0] = 2 * y * G[1] + 2 * z * G[2] + 2 * y * G[3] - 4 * x * G[4] - 2 * w * G[5] + 2 * z * G[6] + 2 * w * G[7] - 4 * x * G[8];
    g[1] = -4 * y * G[0] + 2 * x * G[1] + 2 * w * G[2] + 2 * x * G[3] + 2 * z * G[5] - 2 * w * G[6] + 2 * z * G[7] - 4 * y * G[8];
    g[2] = -4 * z * G[0] - 2 * w * G[1] + 2 * x * G[2] + 2 * w * G[3] - 4 * z * G[4] + 2 * y * G[5] + 2 * x * G[6] + 2 * y * G[7];
    g[3] = -2 * z * G[1] + 2 * y * G[2] + 2 * z * G[3] - 2 * x * G[5] - 2 * y * G[6] + 2 * x * G[7];
}

// One CTA per object: adds the per-CTA partials of backward_points_kernel<*, true> (each thread a fixed, strided set of
// blocks in block order, then a fixed tree over the threads) and takes (dL/dW, dL/dt_c) to (dL/dq, dL/dt) through what
// pose_kernel (preprocess.cu) computes from q_pointcloud_camera, t_pointcloud_camera:
//   qi = conj(q),  W = R(qi) (polynomial, qi NOT normalised),  t_c = -R(qi / |qi|) t.
constexpr int POSE_FINALIZE_THREADS = 128;
__global__ void __launch_bounds__(POSE_FINALIZE_THREADS)
pose_grad_finalize_kernel(const float *partials, int num_blocks, int n_obj, const float *q_pc, const float *t_pc,
                          float *grad_q, float *grad_t) {
    __shared__ float s_sum[12][POSE_FINALIZE_THREADS];
    const int obj = blockIdx.x, tid = threadIdx.x;
    float acc[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) acc[k] = 0.0f;
    for (int b = tid; b < num_blocks; b += POSE_FINALIZE_THREADS) {
        const float *row = partials + ((size_t)b * n_obj + obj) * 12;
#pragma unroll
        for (int k = 0; k < 12; ++k) acc[k] += row[k];
    }
#pragma unroll
    for (int k = 0; k < 12; ++k) s_sum[k][tid] = acc[k];
    for (int h = POSE_FINALIZE_THREADS / 2; h > 0; h >>= 1) {
        __syncthreads();
        if (tid < h) {
#pragma unroll
            for (int k = 0; k < 12; ++k) s_sum[k][tid] += s_sum[k][tid + h];
        }
    }
    __syncthreads();
    if (tid != 0) return;
    const float gtc[3] = {s_sum[0][0], s_sum[1][0], s_sum[2][0]};
    float gW[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) gW[k] = s_sum[3 + k][0];
    const float qi[4] = {-q_pc[4 * obj], -q_pc[4 * obj + 1], -q_pc[4 * obj + 2], q_pc[4 * obj + 3]};
    const float t[3] = {t_pc[3 * obj], t_pc[3 * obj + 1], t_pc[3 * obj + 2]};
    const float n = sqrtf(qi[0] * qi[0] + qi[1] * qi[1] + qi[2] * qi[2] + qi[3] * qi[3]);
    const float qn[4] = {qi[0] / n, qi[1] / n, qi[2] / n, qi[3] / n};
    const float x = qn[0], y = qn[1], z = qn[2], w = qn[3];
    const float Rn[9] = {1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y),
                         2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x),
                         2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)};
    // t_c = -Rn t:  dL/dt = -Rn^T dL/dt_c,  dL/dRn = -dL/dt_c (x) t
#pragma unroll
    for (int c = 0; c < 3; ++c) grad_t[3 * obj + c] = -(Rn[c] * gtc[0] + Rn[3 + c] * gtc[1] + Rn[6 + c] * gtc[2]);
    float gRn[9];
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) gRn[a * 3 + b] = -gtc[a] * t[b];
    float gqn[4], gqi[4];
    rotation_polynomial_vjp(x, y, z, w, gRn, gqn);
    rotation_polynomial_vjp(qi[0], qi[1], qi[2], qi[3], gW, gqi);
    // qn = qi / |qi|:  dL/dqi += (dL/dqn - qn (qn . dL/dqn)) / |qi|
    const float dot = qn[0] * gqn[0] + qn[1] * gqn[1] + qn[2] * gqn[2] + qn[3] * gqn[3];
#pragma unroll
    for (int k = 0; k < 4; ++k) gqi[k] += (gqn[k] - qn[k] * dot) / n;
    // qi = conj(q)
    grad_q[4 * obj] = -gqi[0];
    grad_q[4 * obj + 1] = -gqi[1];
    grad_q[4 * obj + 2] = -gqi[2];
    grad_q[4 * obj + 3] = gqi[3];
}

// ------------------------------------------------------------------ view-parallel exchange: rebuild the dense gradients
// After the exchange of the COMPACT rows (parallel.py): grad_sum holds the sum over views of xyz / q / s / logit gradients,
// grad_color_views the per-view colour-argument gradients (3 per row) followed by that view's camera centres.  The SH
// gradient of a view is gcol (x) SH basis(direction from the view's camera centre) * factor (GPCR:749-756, 1105-1125,
// 1167-1182) -- exactly what the dense kernel writes per view -- summed here over the views in rank order (deterministic).
struct ExpandParams {
    long long N;
    int R;
    const float *grad_sum;
    const float *grad_color_views;
    long long view_stride;  // floats between two views' blocks
    const float *xyz;
    const int *obj_id;
    int first_cleared;
    float c_f, h_f;
    float *grad_xyz;
    float *grad_feat;
};

// PART: 0 = everything; 1 = only the 48 SH columns (needs the all-gathered blocks, not the summed rows); 2 = only the summed
// columns xyz / q / s / logit (needs the all-reduced rows, not the blocks).  Parts 1 and 2 write disjoint 32-byte-aligned
// pieces of every row, so part 1 can run -- on another stream -- while the all-reduce is still on the wire (parallel.py).
template <int PART>
__global__ void __launch_bounds__(GSB_POINTS_THREADS, 4)
expand_view_gradients_kernel(const ExpandParams p) {
    __shared__ __align__(16) float s_feat[GSB_POINTS_THREADS / 32][32 * PT_ROW];
    __shared__ float s_xyz[GSB_POINTS_THREADS / 32][96];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float *const my_feat = &s_feat[warp][lane * PT_ROW];
    float *const my_xyz = &s_xyz[warp][lane * 3];
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long base = (long long)blockIdx.x * blockDim.x + warp * 32; base < p.N; base += stride) {
        const long long id = base + lane;
        if (id < p.N) {
            float4 *gf = reinterpret_cast<float4 *>(my_feat);
            if (PART != 1) {
                const float4 *srow = reinterpret_cast<const float4 *>(p.grad_sum + 12 * (size_t)id);
                const float4 s0 = __ldg(srow), s1 = __ldg(srow + 1), s2 = __ldg(srow + 2);
                my_xyz[0] = s0.x; my_xyz[1] = s0.y; my_xyz[2] = s0.z;
                gf[0] = make_float4(s0.w, s1.x, s1.y, s1.z);
                gf[1] = make_float4(s1.w, s2.x, s2.y, s2.z);
            }
            if (PART != 2) {
            float acc[3][16];
#pragma unroll
            for (int ch = 0; ch < 3; ++ch)
#pragma unroll
                for (int k = 0; k < 16; ++k) acc[ch][k] = 0.0f;
            const float x = p.xyz[3 * (size_t)id], y = p.xyz[3 * (size_t)id + 1], z = p.xyz[3 * (size_t)id + 2];
            const int ob = p.obj_id[id];
#pragma unroll 1
            for (int v = 0; v < p.R; ++v) {
                const float *blk = p.grad_color_views + (size_t)v * p.view_stride;
                const float g[3] = {__ldg(blk + 3 * (size_t)id), __ldg(blk + 3 * (size_t)id + 1), __ldg(blk + 3 * (size_t)id + 2)};
                if (g[0] == 0.0f && g[1] == 0.0f && g[2] == 0.0f) continue;  // outside this view's frustum
                const float *centre = blk + 3 * (size_t)p.N + 3 * ob;
                float sh[16];
                sh_basis(x - __ldg(centre), y - __ldg(centre + 1), z - __ldg(centre + 2), sh);
#pragma unroll
                for (int ch = 0; ch < 3; ++ch)
#pragma unroll
                    for (int k = 0; k < 16; ++k) acc[ch][k] += g[ch] * sh[k] * (k == 0 ? p.c_f : p.h_f);
            }
#pragma unroll
            for (int ch = 0; ch < 3; ++ch)
#pragma unroll
                for (int k4 = 0; k4 < 4; ++k4)
                    gf[2 + 4 * ch + k4] = make_float4(4 * k4 < p.first_cleared ? acc[ch][4 * k4] : 0.0f,
                                                      4 * k4 + 1 < p.first_cleared ? acc[ch][4 * k4 + 1] : 0.0f,
                                                      4 * k4 + 2 < p.first_cleared ? acc[ch][4 * k4 + 2] : 0.0f,
                                                      4 * k4 + 3 < p.first_cleared ? acc[ch][4 * k4 + 3] : 0.0f);
            }
        }
        __syncwarp();
        const long long rows = p.N - base < 32 ? p.N - base : 32;
        float4 *const out_f = reinterpret_cast<float4 *>(p.grad_feat + (size_t)GSB_FEATURE_DIM * base);
#pragma unroll
        for (int it = 0; it < GSB_FEATURE_DIM / 4; ++it) {
            const int f = it * 32 + lane;
            const int row = f / (GSB_FEATURE_DIM / 4), c4 = f - row * (GSB_FEATURE_DIM / 4);
            const bool mine = PART == 0 || (PART == 1 ? c4 >= 2 : c4 < 2);  // float4 0..1 = q s logit, 2..13 = SH
            if (row < rows && mine) out_f[f] = *reinterpret_cast<const float4 *>(&s_feat[warp][row * PT_ROW + 4 * c4]);
        }
        if (PART != 1) {
            float *const out_x = p.grad_xyz + 3 * (size_t)base;
#pragma unroll
            for (int it = 0; it < 3; ++it) {
                const int f = it * 32 + lane;
                if (f < 3 * rows) out_x[f] = s_xyz[warp][f];
            }
        }
        __syncwarp();
    }
}

#ifndef GSB_HOST_EMU
static int first_cleared_of_band(int band) { return band <= 0 ? 1 : band == 1 ? 4 : band == 2 ? 9 : 16; }

int launch_backward_points(const GsbBackwardArgs &a, const Workspace &ws, cudaStream_t stream, const long long *skip_flag,
                           const GsbPoseGradArgs *pose) {
    if (a.num_points <= 0) {
        if (pose) {  // no rows: every object gets zeros
            pose_grad_finalize_kernel<<<a.num_objects, POSE_FINALIZE_THREADS, 0, stream>>>(
                static_cast<const float *>(pose->temp), 0, a.num_objects, pose->q_pointcloud_camera,
                pose->t_pointcloud_camera, pose->grad_q_pointcloud_camera, pose->grad_t_pointcloud_camera);
            GSB_CUDA_CHECK(cudaGetLastError());
        }
        return GSB_OK;
    }
    PointsBwdParams p;
    p.ctl_num_in_camera = a.ctl_accumulated_num_in_camera;
    p.ctl_num_pixels = a.ctl_accumulated_num_pixels;
    p.ctl_vs_grad = a.ctl_accumulated_view_space_position_gradients;
    p.ctl_vs_grad_avg = a.ctl_accumulated_view_space_position_gradients_avg;
    p.ctl_pos_grad = a.ctl_accumulated_position_gradients;
    p.ctl_pos_grad_norm = a.ctl_accumulated_position_gradients_norm;
    p.skip_flag = skip_flag;
    p.N = a.num_points;
    p.point_offset = ws.point_offset;
    p.records = ws.records;
    p.point_in_camera = ws.point_in_camera;
    p.accum = a.accum;
    p.poses = ws.poses;
    p.xyz = a.pointcloud;
    p.features = a.pointcloud_features;
    p.obj_id = a.point_object_id;
    p.t_pc_cam = a.t_pointcloud_camera;
    p.K = a.camera_intrinsics;
    p.first_cleared = first_cleared_of_band(a.color_max_sh_band);
    p.q_f = a.grad_q_factor;
    p.s_f = a.grad_s_factor;
    p.a_f = a.grad_alpha_factor;
    p.c_f = a.grad_color_factor;
    p.h_f = a.grad_high_order_color_factor;
    p.grad_xyz = a.grad_pointcloud;
    p.grad_feat = a.grad_pointcloud_features;
    p.grad_sum_compact = a.grad_sum_compact;
    p.grad_color_compact = a.grad_color_compact;
    p.pose_num_objects = pose ? a.num_objects : 0;
    p.pose_partials = pose ? static_cast<float *>(pose->temp) : nullptr;
    long long blocks = (a.num_points + GSB_POINTS_THREADS - 1) / GSB_POINTS_THREADS;
    const long long cap = 16LL * num_sms();
    if (blocks > cap) blocks = cap;
    if (pose && blocks > POSE_MAX_BLOCKS) blocks = POSE_MAX_BLOCKS;  // the partials of gsb200_pose_grad_temp_bytes
    if (blocks <= 0) return GSB_OK;
    const bool compact = (a.flags & GSB_FLAG_COMPACT_GRADS) != 0;
    if (pose) {
        if (compact) backward_points_kernel<true, true><<<(int)blocks, GSB_POINTS_THREADS, 0, stream>>>(p);
        else backward_points_kernel<false, true><<<(int)blocks, GSB_POINTS_THREADS, 0, stream>>>(p);
        GSB_CUDA_CHECK(cudaGetLastError());
        pose_grad_finalize_kernel<<<a.num_objects, POSE_FINALIZE_THREADS, 0, stream>>>(
            p.pose_partials, (int)blocks, a.num_objects, pose->q_pointcloud_camera, pose->t_pointcloud_camera,
            pose->grad_q_pointcloud_camera, pose->grad_t_pointcloud_camera);
    } else if (compact) {
        backward_points_kernel<true><<<(int)blocks, GSB_POINTS_THREADS, 0, stream>>>(p);
    } else {
        backward_points_kernel<false><<<(int)blocks, GSB_POINTS_THREADS, 0, stream>>>(p);
    }
    GSB_CUDA_CHECK(cudaGetLastError());
    return GSB_OK;
}

int launch_expand_view_gradients(const GsbExpandArgs &a, cudaStream_t stream) {
    if (a.num_points <= 0) return GSB_OK;
    ExpandParams p;
    p.N = a.num_points;
    p.R = a.num_views;
    p.grad_sum = a.grad_sum;
    p.grad_color_views = a.grad_color_views;
    p.view_stride = a.view_stride;
    p.xyz = a.pointcloud;
    p.obj_id = a.point_object_id;
    p.first_cleared = first_cleared_of_band(a.color_max_sh_band);
    p.c_f = a.grad_color_factor;
    p.h_f = a.grad_high_order_color_factor;
    p.grad_xyz = a.grad_pointcloud;
    p.grad_feat = a.grad_pointcloud_features;
    long long blocks = (a.num_points + GSB_POINTS_THREADS - 1) / GSB_POINTS_THREADS;
    const long long cap = 16LL * num_sms();
    if (blocks > cap) blocks = cap;
    if (a.part == 1) expand_view_gradients_kernel<1><<<(int)blocks, GSB_POINTS_THREADS, 0, stream>>>(p);
    else if (a.part == 2) expand_view_gradients_kernel<2><<<(int)blocks, GSB_POINTS_THREADS, 0, stream>>>(p);
    else expand_view_gradients_kernel<0><<<(int)blocks, GSB_POINTS_THREADS, 0, stream>>>(p);
    GSB_CUDA_CHECK(cudaGetLastError());
    return GSB_OK;
}
#endif  // GSB_HOST_EMU

}  // namespace gsb
