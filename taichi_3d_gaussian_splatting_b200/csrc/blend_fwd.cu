// blend_fwd.cu -- per-tile front-to-back alpha blending (replaces gaussian_point_rasterisation,
// GPCR:318-485, with get_point_probability_density_from_conic_and_rescale, UT:275-284).
//
// One CTA per 16x16 tile, one pixel per thread; a warp owns an 8x4 pixel patch.  The tile's splat list is
// streamed through shared memory in batches of 256 packed 48-byte records (3 x float4, gathered by the sorted
// in-camera offsets, double-buffered: one barrier per batch).  While staging, every loading thread tests its
// splat against the 8 patches (common.cuh) and the CTA builds per-patch bit lists with ballots.  A warp then
// turns its bit list into an index list, copies the records it has to visit, 32 at a time, into a private
// chunk buffer, and walks the chunk with a BRANCH-FREE body (a splat that fails alpha >= 1/255, or meets a
// saturated pixel, contributes zero weight): 30 SASS instructions per visited (warp, splat) instead of 49
// with the bit-scan loop and its data-dependent branches (94 % of the visits have a contributing pixel, so the
// branches never skipped much).  The CTA leaves the list as soon as every pixel has saturated
// (__syncthreads_and) -- the reference walks the whole list (GPCR:387-394).  Compute-bound (FP32 issue +
// MUFU.EX2), not HBM-bound: 48 B per (tile, splat) are reused by up to 256 pixels.
#include "common.cuh"

namespace gsb {

struct BlendFwdParams {
    int H, W, tiles_x;
    const int *tile_start;
    const int *tile_end;
    const int *sorted_vals;
    const float4 *records;
    float *image;
    float *depth;
    float *acc_alpha;
    int *last_effective;
    int *valid_count;
    unsigned char *patch_masks = nullptr;  // !RGB_ONLY: the reach mask of every staged key, by sorted index (read by the backward)
    unsigned long long *work_counters;  // COUNT instantiation only: [0] (warp, splat) visits, [1] (pixel, splat)
                                        //   evaluations with alpha >= 1/255 on a live pixel (SURVEY 8(d) "E"); what-if
                                        //   counters at staging time (before any saturation exit): [2] (8x4 patch, splat)
                                        //   pairs, [3] the same with 8x8 patches (two pixels per thread, vertical pairs),
                                        //   [4] with 16x4 patches (horizontal pairs), [5] with 4x4 sub-patches
};

__device__ __forceinline__ float ex2_approx(float x) { return ex2_mufu(x); }

#ifdef GSB_HOST_EMU
// tests/simt: the entry points that run the forward blend on its own pass no mask array
inline void store_patch_mask(unsigned char *masks, int idx, unsigned int mask) {
    if (masks) masks[idx] = (unsigned char)mask;
}
#else
__device__ __forceinline__ void store_patch_mask(unsigned char *masks, int idx, unsigned int mask) {
    masks[idx] = (unsigned char)mask;
}
#endif

// cnt += 1 and last = idx for a blended pair (wgt > 0): one FSETP and two predicated moves instead of the four instructions
// the compiler makes of the two selects
__device__ __forceinline__ void count_if_blended(float wgt, int idx, int &cnt, int &last) {
#ifdef GSB_HOST_EMU
    if (wgt > 0.0f) {
        cnt += 1;
        last = idx;
    }
#else
    asm("{\n"
        ".reg .pred p;\n"
        "setp.gt.f32 p, %2, 0f00000000;\n"
        "@p add.s32 %0, %0, 1;\n"
        "@p mov.b32 %1, %3;\n"
        "}\n"
        : "+r"(cnt), "+r"(last)
        : "f"(wgt), "r"(idx));
#endif
}

#ifndef GSB_FWD_MIN_BLOCKS
#define GSB_FWD_MIN_BLOCKS 4
#endif
#ifndef GSB_FWD_UNROLL
#define GSB_FWD_UNROLL 8  // measured at C3: unroll 2 / 4 / 8 at 5 CTAs per SM 384 / 381 / 380 us, unroll 8 at 4 CTAs per SM (64 registers) 374 us
#endif
constexpr int FW_UNROLL = GSB_FWD_UNROLL;
constexpr int FW_CHUNK = 32;  // splats per private chunk of a warp

template <bool RGB_ONLY, bool EXACT_EXP, bool COUNT = false>
__global__ void __launch_bounds__(GSB_TILE_PIXELS, GSB_FWD_MIN_BLOCKS)
blend_forward_kernel(const BlendFwdParams p) {
    // double-buffered staging area: [buf][plane][splat]; planes: u v a b | c rescale opacity depth | r g b radius
    __shared__ float4 s_rec[2 * 3 * GSB_TILE_PIXELS];
    __shared__ unsigned int s_bits[2][8][8];        // [buf][consumer warp patch][loader warp] -> splats that can reach it
    __shared__ float4 s_chunk[8][3][FW_CHUNK];      // per warp: the records of the current chunk [plane][slot]; the unused
                                                    //   radius word carries the splat's sorted index + 1 ("last effective")
    __shared__ unsigned char s_list[8][GSB_TILE_PIXELS];  // per warp: elements of the current batch to visit, in order

    const int tile = blockIdx.x;
    const int tu = tile % p.tiles_x, tv = tile / p.tiles_x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // warp w covers the 8x4 patch at ((w & 1) * 8, (w >> 1) * 4)
    const int pu = tu * GSB_TILE_WIDTH + (warp & 1) * 8 + (lane & 7);
    const int pv = tv * GSB_TILE_HEIGHT + (warp >> 1) * 4 + (lane >> 3);
    const float px = (float)pu + 0.5f, py = (float)pv + 0.5f;  // GPCR:442 pixel centre
    const float tile_x0 = (float)(tu * GSB_TILE_WIDTH), tile_y0 = (float)(tv * GSB_TILE_HEIGHT);
    const int start = p.tile_start[tile], end = p.tile_end[tile];

    // T is the working transmittance; once the pixel has saturated it is <= 0 (exact path: 0, with Tlive keeping the value
    // to output; fast path: minus the last live value), which makes every later splat fail the T(1-a) >= 1e-4 test.
    float T = 1.0f, Tlive = 1.0f, C0 = 0.0f, C1 = 0.0f, C2 = 0.0f, D = 0.0f, Wt = 0.0f;
    int last = start, cnt = 0;
    unsigned int n_visits = 0, n_pairs = 0;  // COUNT only
    unsigned int n_p84 = 0, n_p88 = 0, n_p164 = 0, n_p44 = 0;
    float4 *const ck0 = s_chunk[warp][0], *const ck1 = s_chunk[warp][1], *const ck2 = s_chunk[warp][2];
    unsigned char *const list = s_list[warp];
    const unsigned int lt_mask = (1u << lane) - 1u;

    // One barrier per batch: batch k is staged into buffer k&1 while slower warps may still be copying chunks of
    // batch k-1 out of the other buffer; passing barrier k implies everybody is done with batch k-1.
    int buf = 0;
    for (int base = start; base < end; base += GSB_TILE_PIXELS, buf ^= 1) {
        float4 *const s_r0 = s_rec + buf * 3 * GSB_TILE_PIXELS;
        float4 *const s_r1 = s_r0 + GSB_TILE_PIXELS, *const s_r2 = s_r0 + 2 * GSB_TILE_PIXELS;
        const int idx = base + tid;
        unsigned int mask = 0;
        if (idx < end) {
            const int o = __ldg(&p.sorted_vals[idx]);
            const float4 *rec = p.records + 3 * (size_t)o;
            const float4 r0 = __ldg(rec), r1 = __ldg(rec + 1);
            if (EXACT_EXP) {
                s_r0[tid] = r0;
                s_r1[tid] = r1;
            } else {  // fast path: -1/2, log2(e) and rescale*opacity folded into the staged record (common.cuh)
                float4 f0, f1;
                fast_planes(r0, r1, f0, f1);
                s_r0[tid] = f0;
                s_r1[tid] = f1;
            }
            s_r2[tid] = __ldg(rec + 2);
            mask = splat_patch_mask(r0.x, r0.y, r0.z, r0.w, r1.x, r1.y * r1.z, tile_x0, tile_y0);
            // the backward walks the keys below each patch's deepest effective splat; all of them are staged here (the
            // early exit below comes after the staging of its batch)
            if (!RGB_ONLY) store_patch_mask(p.patch_masks, idx, mask);
            if (COUNT) {  // patch w sits at column (w & 1), row (w >> 1)
                n_p84 += __popc(mask);
                n_p88 += __popc((mask | (mask >> 2)) & 0x33u);   // rows 0|1 and 2|3 merged
                n_p164 += __popc((mask | (mask >> 1)) & 0x55u);  // the two columns merged
                // ... and with 4x4 sub-patches (one splat per half-warp): the 16 sub-rectangles of the tile
                const SplatReach rr = make_splat_reach(r0.z, r0.w, r1.x, r1.y * r1.z);
                if (rr.mode == 2) n_p44 += 16;
                else if (rr.mode == 1)
                    for (int q = 0; q < 16; ++q) {
                        const float X0 = tile_x0 + 4.0f * (q & 3) + 0.5f - r0.x, Y0 = tile_y0 + 4.0f * (q >> 2) + 0.5f - r0.y;
                        n_p44 += rect_reachable(rr, X0, X0 + 3.0f, Y0, Y0 + 3.0f) ? 1 : 0;
                    }
            }
        }
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            const unsigned int bits = __ballot_sync(0xffffffffu, (mask >> w) & 1u);
            if (lane == 0) s_bits[buf][w][warp] = bits;
        }
        if (__syncthreads_and(!(T > 0.0f))) break;  // staging visible + tile-level early exit
        if (__all_sync(0xffffffffu, !(T > 0.0f))) continue;  // whole patch saturated: only help with loads
        // ordered visit list of this patch: the set bits of its 8 words
        int count = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const unsigned int bits = s_bits[buf][warp][k];
            if ((bits >> lane) & 1u) list[count + __popc(bits & lt_mask)] = (unsigned char)(k * 32 + lane);
            count += __popc(bits);
        }
        __syncwarp();
#pragma unroll 1
        for (int pos = 0; pos < count; pos += FW_CHUNK) {
            const int n = min(FW_CHUNK, count - pos);
            if (lane < n) {
                const int j = list[pos + lane];
                ck0[lane] = s_r0[j];
                ck1[lane] = s_r1[j];
                float4 r2 = s_r2[j];
                r2.w = __int_as_float(base + j + 1);  // GPCR:462 offset_of_last_effective_point if this splat is blended
                ck2[lane] = r2;
            }
            __syncwarp();
            if (COUNT) n_visits += (lane == 0) ? (unsigned int)n : 0u;
            if (lane == 0) GSB_EMU_COUNT(EC_FW_VISITS, n);
#pragma unroll FW_UNROLL
            for (int i = 0; i < n; ++i) {
                const float4 r0 = ck0[i];  // u v a b               (fast: u v A B)
                const float4 r1 = ck1[i];  // c rescale opacity depth (fast: C ro - depth)
                const float4 r2 = ck2[i];  // r g b | sorted index + 1
                const float dx = px - r0.x, dy = py - r0.y;
                if (EXACT_EXP) {  // the reference's op order (UT:275-284, GPCR:451-469)
                    const float power = -0.5f * (dx * dx * r0.z + dy * dy * r1.x) - dx * dy * r0.w;
                    float alpha = expf(power) * r1.y * r1.z;
                    if (!(alpha < 1.0f / 255.0f)) {             // GPCR:451 (same comparison as the reference)
                        if (COUNT) n_pairs += T > 0.0f ? 1u : 0u;
                        GSB_EMU_COUNT(EC_FW_PAIRS, 1);
                        alpha = fminf(alpha, 0.99f);            // GPCR:453
                        const float nT = T * (1.0f - alpha);
                        if (nT >= 0.0001f) {
                            last = __float_as_int(r2.w);
                            C0 += r2.x * alpha * T;
                            C1 += r2.y * alpha * T;
                            C2 += r2.z * alpha * T;
                            if (!RGB_ONLY) {
                                D += r1.w * alpha * T;
                                Wt += alpha * T;
                                cnt += 1;
                            }
                            T = nT;
                            Tlive = nT;
                        } else {
                            T = 0.0f;  // GPCR:457-460: saturated; this splat is NOT blended
                        }
                    }
                } else {
                    // Branch-free: a pair that fails the alpha cut gets alpha = 0 (T, the sums and the counters are left
                    // as they are).  A pixel that saturates keeps the MAGNITUDE of its last transmittance with the sign
                    // flipped: T < 0 makes every later nT = T (1 - alpha) fail the 1e-4 test, so it gets zero weight without
                    // a separate flag, and |T| is the value to output (GPCR:457-460, 476).
                    float P = fast_alpha(dx, dy, r0.z, r0.w, r1.x, r1.y);
                    P = (P < 1.0f / 255.0f) ? 0.0f : P;        // GPCR:451 (same comparison as the reference)
                    const float alpha = fminf(P, 0.99f);        // GPCR:453
                    const float nT = T * (1.0f - alpha);
                    const bool ok = nT >= 0.0001f;              // GPCR:457
                    const float wgt = ok ? alpha * T : 0.0f;   // > 0 exactly for the blended pairs (alpha > 0 and T > 0)
                    if (COUNT) n_pairs += (P != 0.0f && T > 0.0f) ? 1u : 0u;
                    GSB_EMU_COUNT(EC_FW_PAIRS, (P != 0.0f && T > 0.0f) ? 1 : 0);
                    C0 = fmaf(r2.x, wgt, C0);
                    C1 = fmaf(r2.y, wgt, C1);
                    C2 = fmaf(r2.z, wgt, C2);
                    if (!RGB_ONLY) {
                        D = fmaf(r1.w, wgt, D);
                        Wt += wgt;
                        count_if_blended(wgt, __float_as_int(r2.w), cnt, last);
                    }
                    T = ok ? nT : -fabsf(T);
                }
            }
            __syncwarp();  // everybody has read the chunk before the next one overwrites it
            if (__all_sync(0xffffffffu, !(T > 0.0f))) break;
        }
    }
    const size_t pix = (size_t)pv * p.W + pu;
    p.image[3 * pix] = C0;
    p.image[3 * pix + 1] = C1;
    p.image[3 * pix + 2] = C2;
    if (!RGB_ONLY) {
        p.depth[pix] = D / fmaxf(Wt, 1e-6f);  // GPCR:479-480
        p.acc_alpha[pix] = 1.0f - (EXACT_EXP ? Tlive : fabsf(T));
        p.last_effective[pix] = last;
        p.valid_count[pix] = cnt;
    }
    if (COUNT) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            n_visits += __shfl_xor_sync(0xffffffffu, n_visits, d);
            n_pairs += __shfl_xor_sync(0xffffffffu, n_pairs, d);
            n_p84 += __shfl_xor_sync(0xffffffffu, n_p84, d);
            n_p88 += __shfl_xor_sync(0xffffffffu, n_p88, d);
            n_p164 += __shfl_xor_sync(0xffffffffu, n_p164, d);
            n_p44 += __shfl_xor_sync(0xffffffffu, n_p44, d);
        }
        if (lane == 0) {
            atomicAdd(p.work_counters, (unsigned long long)n_visits);
            atomicAdd(p.work_counters + 1, (unsigned long long)n_pairs);
            atomicAdd(p.work_counters + 2, (unsigned long long)n_p84);
            atomicAdd(p.work_counters + 3, (unsigned long long)n_p88);
            atomicAdd(p.work_counters + 4, (unsigned long long)n_p164);
            atomicAdd(p.work_counters + 5, (unsigned long long)n_p44);
        }
    }
}

#ifndef GSB_HOST_EMU
int launch_blend_forward(const GsbForwardArgs &a, const Workspace &ws, cudaStream_t stream) {
    BlendFwdParams p;
    p.H = a.camera_height;
    p.W = a.camera_width;
    p.tiles_x = a.camera_width / GSB_TILE_WIDTH;
    p.tile_start = ws.tile_start;
    p.tile_end = ws.tile_end;
    p.sorted_vals = ws.vals_b;  // the sort always ends in b
    p.records = ws.records;
    p.image = a.rasterized_image;
    p.depth = a.rasterized_depth;
    p.acc_alpha = a.pixel_accumulated_alpha;
    p.last_effective = a.pixel_offset_of_last_effective_point;
    p.valid_count = a.pixel_valid_point_count;
    p.patch_masks = ws.patch_masks;
    p.work_counters = nullptr;
    const int tiles = p.tiles_x * (a.camera_height / GSB_TILE_HEIGHT);
    if (tiles <= 0) return GSB_OK;
    const bool exact = (a.flags & GSB_FLAG_EXACT_EXP) != 0;
    if (a.rgb_only) {
        if (exact) blend_forward_kernel<true, true><<<tiles, GSB_TILE_PIXELS, 0, stream>>>(p);
        else blend_forward_kernel<true, false><<<tiles, GSB_TILE_PIXELS, 0, stream>>>(p);
    } else {
        if (exact) blend_forward_kernel<false, true><<<tiles, GSB_TILE_PIXELS, 0, stream>>>(p);
        else blend_forward_kernel<false, false><<<tiles, GSB_TILE_PIXELS, 0, stream>>>(p);
    }
    GSB_CUDA_CHECK(cudaGetLastError());
    return GSB_OK;
}

// Diagnostic: the forward blend of a frame whose earlier stages have run in this workspace, with GPU-side work counters
// (full outputs, default arithmetic): counters_dev[0] = (warp, splat) visits, [1] = (pixel, splat) evaluations that pass
// the alpha cut on a live pixel -- SURVEY 8(d)'s "E" measured on the device instead of estimated.
int launch_blend_forward_count(const GsbForwardArgs &a, const Workspace &ws, unsigned long long *counters_dev,
                               cudaStream_t stream) {
    BlendFwdParams p;
    p.H = a.camera_height;
    p.W = a.camera_width;
    p.tiles_x = a.camera_width / GSB_TILE_WIDTH;
    p.tile_start = ws.tile_start;
    p.tile_end = ws.tile_end;
    p.sorted_vals = ws.vals_b;  // the sort always ends in b
    p.records = ws.records;
    p.image = a.rasterized_image;
    p.depth = a.rasterized_depth;
    p.acc_alpha = a.pixel_accumulated_alpha;
    p.last_effective = a.pixel_offset_of_last_effective_point;
    p.valid_count = a.pixel_valid_point_count;
    p.patch_masks = ws.patch_masks;
    p.work_counters = counters_dev;
    const int tiles = p.tiles_x * (a.camera_height / GSB_TILE_HEIGHT);
    if (tiles <= 0) return GSB_OK;
    blend_forward_kernel<false, false, true><<<tiles, GSB_TILE_PIXELS, 0, stream>>>(p);
    GSB_CUDA_CHECK(cudaGetLastError());
    return GSB_OK;
}
#endif  // GSB_HOST_EMU

}  // namespace gsb
