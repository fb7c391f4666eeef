// blend_bwd.cuh -- declarations shared by the two implementations of loop A of the backward
// (blend_bwd.cu: butterfly reduction per (warp, splat); blend_bwd_transposed.cu: splat-per-lane accumulation).
#pragma once
#include "common.cuh"

namespace gsb {

struct BlendBwdParams {
    int H, W, tiles_x;
    const int *tile_start;
    const int *tile_end;
    const int *sorted_vals;
    const float4 *records;
    const float *grad_image;
    const float *acc_alpha;
    const int *last_effective;
    const unsigned char *patch_masks = nullptr;  // the forward's reach mask per sorted key (blend_bwd_transposed.cu only)
    float *accum;      // rows of 12 floats
    float *mag_image;  // (H,W,2)
    unsigned long long *work_counters;  // COUNT instantiation only: [0] (warp, splat) visits, [1] contributing (pixel, splat) pairs
};

#ifdef GSB_HOST_EMU  // tests/simt: the kernels compiled as host C++ under a lock-step SIMT emulator
__device__ __forceinline__ float ex2_approx_b(float x) { return exp2f(x); }
__device__ __forceinline__ float rcp_approx(float x) { return 1.0f / x; }
__device__ __forceinline__ float sqrt_approx(float x) { return sqrtf(x); }
#else
__device__ __forceinline__ float ex2_approx_b(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x) {  // MUFU.RCP, <= 1 ulp
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float sqrt_approx(float x) {  // MUFU.RSQ based, ~1 ulp
    float y;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
#endif

int launch_blend_backward_transposed(const BlendBwdParams &p, int tiles, bool exact_exp, bool stats,
                                     cudaStream_t stream);
int launch_blend_backward_count(const BlendBwdParams &p, int tiles, cudaStream_t stream);

}  // namespace gsb
