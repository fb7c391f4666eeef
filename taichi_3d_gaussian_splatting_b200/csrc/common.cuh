// common.cuh -- shared declarations of libgsb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/gsb200.h"

#define GSB_TILE_PIXELS (GSB_TILE_WIDTH * GSB_TILE_HEIGHT)

namespace gsb {

// ---- error plumbing (thread-local message, C ABI returns a code)
void set_error(const char *fmt, ...);
#define GSB_CUDA_CHECK(expr)                                                                   \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            gsb::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__,   \
                           __LINE__);                                                          \
            return GSB_ECUDA;                                                                  \
        }                                                                                      \
    } while (0)

// ---- counters living at the head of the workspace
// CNT_MAX_DEPTH_KEY: largest int32(depth * scale) over the frame's in-camera points (low 32 bits of the slot; the per-point
// kernel atomicMax-es it, the sort derives the number of live depth bits from it)
enum Counter { CNT_M = 0, CNT_K = 1, CNT_OVERFLOW = 2, CNT_MAX_DEPTH_KEY = 4 };
// gsb200_backward_with_pose: the per-point kernel runs on at most this many CTAs, so that its per-CTA pose partials fit the
// temp size gsb200_pose_grad_temp_bytes gives without asking the device (16 CTAs per SM up to 256 SMs)
constexpr int POSE_MAX_BLOCKS = 4096;
enum Ticket { TICKET_SCAN = 0, TICKET_SORT0 = 1 /* ..+7: one per pass; +8: histogram blocks done */ };

// Per-object pose block in the workspace (20 floats):
//   [0..11]  T_camera_pointcloud 3x4 row-major (R | t)     GP3D:51-62
//   [12..14] camera centre in the pointcloud frame (-R^T t)  UT:495-510
struct PoseBlock {
    float T[12];
    float centre[3];
    float pad[5];
};
static_assert(sizeof(PoseBlock) == 80, "PoseBlock layout");

// Resolved device pointers of one frame's workspace.
struct Workspace {
    long long *counters;
    unsigned int *tickets;
    unsigned long long *scan_state;
    unsigned int *sort_hist;
    unsigned int *sort_state;
    int *tile_start;
    int *tile_end;
    PoseBlock *poses;
    int *point_id;
    int *point_offset;
    int *num_tiles;
    float4 *records;        // 3 float4 per in-camera point
    float *point_in_camera; // 3 floats per in-camera point
    void *keys_a, *keys_b, *keys_c;  // emitted keys (a), sorted keys (b), scratch of the radix passes (c)
    int *vals_a, *vals_b, *vals_c;
    unsigned char *patch_masks;  // one byte per sorted key: the 8-patch reach mask the forward blend computed for it
                                 //   (bit w = patch of warp w); lives in keys_c, which is dead once the sort has finished
    GsbWorkspaceLayout layout;
};

int resolve_workspace(void *base, int64_t bytes, int64_t N, int32_t n_obj, int64_t key_capacity,
                      int32_t H, int32_t W, float far_plane, float depth_scale, uint32_t flags,
                      Workspace *ws);

// ---- stage launchers (each enqueues on `stream`, returns GSB_* code)
int launch_preprocess(const GsbForwardArgs &a, const Workspace &ws, cudaStream_t stream);
int launch_sort(const Workspace &ws, int64_t key_capacity, cudaStream_t stream);
int launch_tile_ranges(const Workspace &ws, int64_t key_capacity, int num_tiles, cudaStream_t stream);
int launch_tile_ranges_raw(const long long *keys_i64, int64_t n, int *tile_start, int *tile_end,
                           int num_tiles, cudaStream_t stream);
int launch_blend_forward(const GsbForwardArgs &a, const Workspace &ws, cudaStream_t stream);
int launch_blend_backward(const GsbBackwardArgs &a, const Workspace &ws, cudaStream_t stream);
// pose: gsb200_backward_with_pose's outputs (the POSE instantiation of the per-point kernel + its finalisation), or nullptr
int launch_backward_points(const GsbBackwardArgs &a, const Workspace &ws, cudaStream_t stream,
                           const long long *skip_flag = nullptr, const GsbPoseGradArgs *pose = nullptr);
int launch_adam_step(float *param, const float *grad, float *exp_avg, float *exp_avg_sq, long long n, double lr, double beta1,
                     double beta2, double eps, int step, const long long *skip_flag, cudaStream_t stream);
int launch_expand_view_gradients(const GsbExpandArgs &a, cudaStream_t stream);
int launch_blend_forward_count(const GsbForwardArgs &a, const Workspace &ws, unsigned long long *counters_dev,
                               cudaStream_t stream);
int launch_blend_backward_work(const GsbBackwardArgs &a, const Workspace &ws, unsigned long long *counters_dev,
                               cudaStream_t stream);

int sort_radix_bits(int bits);
int sort_pairs_device(const void *keys_in, const int *vals_in, void *keys_out, int *vals_out,
                      const long long *n_dev, int64_t n_capacity, int key_bytes, int depth_bits, int end_bit,
                      const int *max_depth_key /*device or NULL*/, unsigned int *hist /*8*256, zeroed*/,
                      unsigned int *state /*zeroed*/, unsigned int *tickets /*9, zeroed*/, void *tmp_keys,
                      int *tmp_vals, cudaStream_t stream);

#ifndef GSB_SORT_ITEMS
#define GSB_SORT_ITEMS 12
#endif
#ifndef GSB_SORT_MIN_BLOCKS
#define GSB_SORT_MIN_BLOCKS 3
#endif
constexpr int SORT_BLOCK_THREADS = 256;
constexpr int SORT_ITEMS_PER_THREAD = GSB_SORT_ITEMS;
constexpr int SORT_TILE = SORT_BLOCK_THREADS * SORT_ITEMS_PER_THREAD;  // 3072 keys per CTA
#ifndef GSB_SCAN_THREADS
#define GSB_SCAN_THREADS 128
#endif
constexpr int SCAN_BLOCK_THREADS = GSB_SCAN_THREADS;

// ---- per-warp culling shared by the forward and backward blend kernels.
// A CTA renders a 16x16 tile with 8 warps; warp w owns the 8x4 pixel patch at ((w & 1) * 8, (w >> 1) * 4).
// When a batch of splats is staged into shared memory the loading thread computes, for its splat, which
// of the 8 patches it can reach with alpha >= 1/255: alpha = exp(-q/2) * rescale * opacity >= 1/255 needs
// q(d) = d^T conic d <= t2 = 2 ln(255 * rescale * opacity).  A patch is kept iff the minimum of the convex
// quadratic q over the rectangle spanned by the patch's pixel centres is <= t2 (0 if the splat centre is
// inside; otherwise attained on one of the four edges, a clamped 1-D minimisation each).  The test is
// conservative (t2 padded by 0.2 % + 1e-3; degenerate or NaN conics keep every patch), so it never
// changes a result -- it only lets a warp skip splats none of its 32 pixels can see.
#if defined(__CUDACC__) || defined(GSB_HOST_EMU)
#ifdef GSB_HOST_EMU
// tests/simt compiles the blend-backward kernels as host C++ under a lock-step SIMT emulator (simt_emu.h): "shared
// space addresses" are 32-bit offsets from an anchor inside the emulator's image, the approximations are libm calls.
template <int BYTE_OFFSET>
inline float4 lds128(unsigned int saddr) {
    return *reinterpret_cast<const float4 *>(simt_emu::smem_anchor() + (long long)(int)saddr + BYTE_OFFSET);
}
inline unsigned int smem_u32(const void *p) {
    return (unsigned int)(int)(reinterpret_cast<const char *>(p) - simt_emu::smem_anchor());
}
inline float rcp_fast(float x) { return 1.0f / x; }
#else
// 128-bit shared-memory load from an explicit shared-space address (keeps the address arithmetic of the
// blend inner loops to one IMAD instead of a generic->shared window computation per access).
template <int BYTE_OFFSET>
__device__ __forceinline__ float4 lds128(unsigned int saddr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4+%5];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "r"(saddr), "n"(BYTE_OFFSET));
    return v;
}
// Shared-space address of a __shared__ object, made opaque so that the compiler keeps it in a register
// instead of re-deriving it (S2R SR_CgaCtaId + LEA chain on sm_100) inside the inner loops.
__device__ __forceinline__ unsigned int smem_u32(const void *p) {
    unsigned int a = (unsigned int)__cvta_generic_to_shared(p);
    asm volatile("" : "+r"(a));
    return a;
}
#endif

// Reach test of one splat: can alpha = exp(-q/2) * ro reach 1/255 anywhere in a rectangle of pixel centres?
// q(d) = d^T conic d <= t2 = 2 ln(255 ro) (padded by 0.2 % + 1e-3).  `mode`: 0 = never (ro too small),
// 1 = test rectangles with rect_reachable(), 2 = always (NaN / degenerate conic: keep the reference behaviour).
// The arithmetic uses explicit FMAs and approximate reciprocals: it only has to be conservative, not exact.
struct SplatReach {
    float a, b2, c;        // conic a, 2b, c
    float nb_ic, nb_ia;    // -b / c, -b / a  (1-D minimisers along vertical / horizontal edges)
    float t2;
    int mode;
};
#ifndef GSB_HOST_EMU
__device__ __forceinline__ float rcp_fast(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
#endif
__device__ __forceinline__ float quad_form(const SplatReach &r, float dx, float dy) {
    return fmaf(dx, fmaf(r.b2, dy, r.a * dx), r.c * dy * dy);
}
__device__ __forceinline__ SplatReach make_splat_reach(float a, float b, float c, float rescale_times_opacity) {
    SplatReach r;
    r.a = a; r.b2 = 2.0f * b; r.c = c;
    const float ro = rescale_times_opacity;
    r.nb_ic = -b * rcp_fast(c);
    r.nb_ia = -b * rcp_fast(a);
    r.t2 = fmaf(2.0f * 1.002f, __logf(fmaxf(255.0f * ro, 1.0f)), 1e-3f);
    const float det = a * c - b * b;
    if (!(ro == ro) || !(det > 0.0f) || !(a > 0.0f) || !(c > 0.0f)) r.mode = 2;
    else if (ro < (1.0f / 255.0f) * 0.999f) r.mode = 0;  // exp(.) <= 1: can never reach 1/255
    else r.mode = 1;
    return r;
}
// Rectangle [X0,X1] x [Y0,Y1] is given RELATIVE to the splat centre.  Minimum of the convex quadratic over the
// rectangle: 0 if the centre is inside, otherwise attained on one of the four edges (clamped 1-D minimisation).
__device__ __forceinline__ bool rect_reachable(const SplatReach &r, float X0, float X1, float Y0, float Y1) {
    if (X0 <= 0.0f && X1 >= 0.0f && Y0 <= 0.0f && Y1 >= 0.0f) return true;
    const float ya = fminf(fmaxf(r.nb_ic * X0, Y0), Y1);
    const float yb = fminf(fmaxf(r.nb_ic * X1, Y0), Y1);
    const float xa = fminf(fmaxf(r.nb_ia * Y0, X0), X1);
    const float xb = fminf(fmaxf(r.nb_ia * Y1, X0), X1);
    const float best = fminf(fminf(quad_form(r, X0, ya), quad_form(r, X1, yb)),
                             fminf(quad_form(r, xa, Y0), quad_form(r, xb, Y1)));
    return !(best > r.t2);  // NaN keeps the rectangle
}

__device__ __forceinline__ unsigned int splat_patch_mask(float u, float v, float a, float b, float c,
                                                         float rescale_times_opacity, float tile_x0,
                                                         float tile_y0) {
    const SplatReach r = make_splat_reach(a, b, c, rescale_times_opacity);
    if (r.mode == 0) return 0u;
    if (r.mode == 2) return 0xFFu;
    unsigned int m = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
        // rectangle of the patch's pixel centres, relative to the splat centre
        const float X0 = tile_x0 + 8.0f * (w & 1) + 0.5f - u;
        const float Y0 = tile_y0 + 4.0f * (w >> 1) + 0.5f - v;
        if (rect_reachable(r, X0, X0 + 7.0f, Y0, Y0 + 3.0f)) m |= 1u << w;
    }
    return m;
}
#endif

// ---- alpha of the default (fast) arithmetic path, shared by the forward blend and both backward kernels so that the
// alpha >= 1/255 decision of a (pixel, splat) pair is taken on bit-identical values in both passes.  The staged record
// carries the conic pre-scaled by -log2(e)/2: A = -log2(e)/2 a, B = -log2(e) b, C = -log2(e)/2 c, and ro = rescale * opacity:
//   alpha = 2^(A dx^2 + B dx dy + C dy^2) * ro  =  exp(-(a dx^2 + 2 b dx dy + c dy^2) / 2) * rescale * opacity   (UT:275-284)
#if defined(__CUDACC__) || defined(GSB_HOST_EMU)
constexpr float GSB_L2E = 1.4426950408889634f;
#ifdef GSB_HOST_EMU
__device__ __forceinline__ float ex2_mufu(float x) { return exp2f(x); }
#else
__device__ __forceinline__ float ex2_mufu(float x) {  // one MUFU.EX2; rel. error ~2^-22
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
#endif
__device__ __forceinline__ float fast_alpha(float dx, float dy, float A, float B, float C, float ro) {
    return ex2_mufu(fmaf(dx, fmaf(A, dx, B * dy), (C * dy) * dy)) * ro;
}
// record planes r0 = u v a b, r1 = c rescale opacity depth  ->  staged fast-path planes u v A B | C ro (1 - opacity) depth
__device__ __forceinline__ void fast_planes(const float4 r0, const float4 r1, float4 &s0, float4 &s1) {
    s0 = make_float4(r0.x, r0.y, (-0.5f * GSB_L2E) * r0.z, -GSB_L2E * r0.w);
    s1 = make_float4((-0.5f * GSB_L2E) * r1.x, r1.y * r1.z, 1.0f - r1.z, r1.w);
}
#endif

// ---- mbarrier + TMA 1-D bulk copy (global -> shared), used by the radix sort (key tiles) and the per-point stage (feature rows)
#if defined(__CUDACC__) || defined(GSB_HOST_EMU)
#ifdef GSB_HOST_EMU  // tests/simt: host build under the SIMT emulator -- the bulk copy is a memcpy that has landed at once
__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned int) { *bar = 0; }
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long *, unsigned int) {}
__device__ __forceinline__ void bulk_copy_g2s(void *dst_smem, const void *src_gmem, unsigned int bytes,
                                              unsigned long long *) {
    memcpy(dst_smem, src_gmem, bytes);
}
// every lane of the warp calls the wait (warp-uniform condition at both call sites): under the emulator it is a warp
// rendezvous, so the lane that issued the (immediate) copy has done so before any lane reads the destination
__device__ __forceinline__ void mbar_wait(unsigned long long *, unsigned int) { simt_emu::warp_exchange(0u); }
// cp.async (16-byte global -> shared copies, per-thread groups): the copy lands at once; the wait is called by every lane
// of the warp and is a warp rendezvous, as above
__device__ __forceinline__ void cp_async16(void *dst_smem, const void *src_gmem) { memcpy(dst_smem, src_gmem, 16); }
__device__ __forceinline__ void cp_async_commit() {}
template <int N>
__device__ __forceinline__ void cp_async_wait() { simt_emu::warp_exchange(0u); }
#else
// ---- mbarrier / bulk-copy helpers (TMA 1-D bulk copy, global -> shared)
__device__ __forceinline__ unsigned int smem_addr(const void *p) {
    return (unsigned int)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long *bar, unsigned int bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_copy_g2s(void *dst_smem, const void *src_gmem, unsigned int bytes,
                                              unsigned long long *bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_addr(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_addr(bar))
        : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned int parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_addr(bar)),
        "r"(parity)
        : "memory");
}
// ---- cp.async: 16-byte global -> shared copy through L1 (.ca: the CTA's other warps read the same records), in per-thread
// groups.  After cp_async_wait<N>() the thread's own copies of all but the N most recent groups have landed; a __syncwarp()
// then makes them visible to the rest of the warp.
__device__ __forceinline__ void cp_async16(void *dst_smem, const void *src_gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(smem_addr(dst_smem)), "l"(src_gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
#endif

#endif

// Work counters for the CPU-side emulation only (tests/simt, scripts/emu_work_stats.py); nothing in a device build.
#ifdef GSB_HOST_EMU
#define GSB_EMU_COUNT(slot, n) (simt_emu::counters()[slot] += (long long)(n))
#else
#define GSB_EMU_COUNT(slot, n) ((void)0)
#endif
enum EmuCounter {
    EC_BF_VISITS = 0,       // butterfly kernel: (warp, splat) visits
    EC_BF_VISITS_ANY = 1,   //   ... with at least one contributing pixel (these pay the butterfly + RED)
    EC_BF_PAIRS = 2,        //   contributing (pixel, splat) pairs
    EC_TB_SPLATS = 3,       // transposed kernel: (warp, splat) list entries
    EC_TB_CHUNKS = 4,       //   chunks processed
    EC_TB_ROWS = 5,         //   accumulator rows flushed (splats with a contributing pixel)
    EC_TB_WINDOWS = 6,      //   32-key windows of the sorted list walked (per warp)
    EC_FW_VISITS = 7,       // forward blend: (warp, splat) visits
    EC_FW_PAIRS = 8,        //   (pixel, splat) pairs with alpha >= 1/255 on a live pixel (blended or saturating)
};

static inline int num_sms() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

}  // namespace gsb
