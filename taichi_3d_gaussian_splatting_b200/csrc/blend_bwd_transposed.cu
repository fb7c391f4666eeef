// blend_bwd_transposed.cu -- loop A of the backward (GPCR:531-705); the DEFAULT implementation since round 2 (the round-1
// butterfly kernel of blend_bwd.cu stays selectable: backward_impl="butterfly").  Verified on the CPU under tests/simt (the
// kernel body compiled as host C++ and run by a lock-step SIMT emulator against the butterfly kernel and the oracle) and
// on the GPU by every backward parity test.
//
// blend_bwd.cu reduces the 11 per-splat partials of every (warp, splat) visit across the 32 pixels of the warp with a
// 13-shuffle butterfly: ~52 of the ~117 SASS instructions of a visit.  Here a warp copies the splats it has to visit,
// 16 at a time, into a private chunk buffer and works on a chunk in two phases:
//   phase 1 (lane = pixel, as before): the sequential part of GPCR:609-657 -- alpha, the transmittance recursion and
//     the colour recursion -- which leaves two numbers per (pixel, splat): G = dL/dalpha * alpha and alpha*T.  They go
//     to a 32 x 16 exchange buffer in shared memory (row stride 17: conflict-free both ways);
//   phase 2 (lane = splat; lanes 0..15 take pixels 0..15 of the patch, lanes 16..31 the same splats for pixels 16..31):
//     every lane re-derives d and conic*d for its splat, accumulates the 11 partials over its 16 pixels in registers,
//     the two halves are added with one shuffle per value, and the 16 finished rows leave through shared memory as
//     8 RED.ADD.F32 instructions of two contiguous rows each (same 2 sectors per (warp, splat) as the butterfly kernel).
// Per 32 (pixel, splat) pairs that is ~36 (phase 1) + ~36 (chunk fill, phase 2, epilogue) SASS instructions.
//
// Which splats a warp visits: the forward blend has recorded, per sorted key, the mask of the 8 patches of the tile the
// splat can reach (Workspace::patch_masks).  Each warp walks its tile's sorted list on its own, back to front from the
// deepest last_effective of its 32 pixels, in windows of 32 keys: one mask byte and one sorted_vals entry per lane, a
// ballot on the warp's bit, and the selected records go into the chunk with three 16-byte cp.async copies each (through
// L1, which the tile's 8 warps share).  The warps never wait for each other: there is no CTA barrier, and a warp with a
// short list finishes early.  Software pipeline: two chunk buffers per warp (the copies of chunk c+1 are in flight while
// chunk c is computed) and the next window's mask bytes and values are held in registers one window ahead.
// STATS = false (GSB_FLAG_NO_HOOK_STATS, the reference's need_extra_info = False, GPCR:521, 690-704) drops the |d/duv|
// magnitude, the affected-pixel count and the per-pixel magnitude image.
#include "blend_bwd.cuh"

namespace gsb {

constexpr int TB_CHUNK = 16;          // splats per chunk
constexpr int TB_ROW = TB_CHUNK + 1;  // row stride (floats) of the (pixel, splat) exchange buffers
constexpr int TB_TR_ROW = 13;         // row stride of the finished rows (12 accumulator words, odd stride)

struct TbShared {  // dynamic shared memory image, 52 KB -> 4 CTAs per SM
    float4 g[8][32];                      // dL/dimage of the warp's pixels
    float xg[8][32 * TB_ROW];             // G  per (pixel, splat of the chunk); reused for the finished rows
    float xa[8][32 * TB_ROW];             // alpha * T   (interleaving the two as float2 -- one 64-bit store / load instead of
                                          //   two 32-bit ones -- was measured SLOWER on a B200: 724 vs 718 us, profiles/r02_call20.log)
    float4 chunk[8][2][3][TB_CHUNK];      // per warp, two buffers: records of a chunk's splats [plane][slot]; once the copies
                                          //   have landed, the unused radius word of plane 2 carries the splat's sorted index
    int chunk_off[8][2][TB_CHUNK];        //   their accumulator row (set to -1 after phase 2 if nothing is to be added)
    int chunk_idx[8][2][TB_CHUNK];        //   their sorted index (moved into plane 2 after the copies have landed)
};
static_assert(32 * TB_ROW >= TB_CHUNK * TB_TR_ROW, "finished rows must fit into the exchange buffer");

#ifdef GSB_HOST_EMU
static inline unsigned char *tb_dynamic_smem() { return simt_emu::dynamic_smem(); }
#else
extern __shared__ __align__(16) unsigned char gsb_tb_dynamic_smem[];
__device__ __forceinline__ unsigned char *tb_dynamic_smem() { return gsb_tb_dynamic_smem; }
#endif

#ifndef GSB_TB_P1_UNROLL
#define GSB_TB_P1_UNROLL 4  // phase-1 splats per loop trip (measured: 1 -> 746, 2 -> 734, 4 -> 725 us at C3)
#endif
constexpr int TB_P1_UNROLL = GSB_TB_P1_UNROLL;
#ifndef GSB_TB_MIN_BLOCKS
#define GSB_TB_MIN_BLOCKS 4  // 64 registers, 4 x 52 KB of shared memory per SM; measured at C3: 3 CTAs (80 registers) 677 us,
                             //   4 CTAs 634 us.  Tuning knob (GSB200_DEFINES="-DGSB_TB_MIN_BLOCKS=3")
#endif
// CTAs per SM the register budget is set for: the exact path (expf, IEEE division) spills at 64 registers and keeps 3 (80)
constexpr int tb_min_blocks(bool exact_exp) { return exact_exp && GSB_TB_MIN_BLOCKS > 3 ? 3 : GSB_TB_MIN_BLOCKS; }
// P if (idx < last && P >= 1/255) else 0 -- the two tests folded into one predicate (ISETP, FSETP.AND, FSEL instead of
// the two selects the compiler makes of the && expression)
__device__ __forceinline__ float keep_if_contributing(float P, int idx, int last) {
#ifdef GSB_HOST_EMU
    return ((idx < last) && (P >= 1.0f / 255.0f)) ? P : 0.0f;
#else
    float r;
    asm("{\n"
        ".reg .pred p, q;\n"
        "setp.lt.s32 q, %2, %3;\n"
        "setp.ge.and.f32 p, %1, 0f3B808081, q;\n"   // 1.0f / 255.0f
        "selp.f32 %0, %1, 0f00000000, p;\n"
        "}\n"
        : "=f"(r)
        : "f"(P), "r"(idx), "r"(last));
    return r;
#endif
}

// The forward's reach mask of sorted key i (tile at tile_x0, tile_y0).
#ifdef GSB_HOST_EMU
// tests/simt: the entry points that run loop A without the emulated forward pass no mask array; the byte the forward would
// have written comes from the same splat_patch_mask on the same record
inline unsigned int load_patch_mask(const BlendBwdParams &p, int i, float tile_x0, float tile_y0) {
    if (p.patch_masks) return p.patch_masks[i];
    const float4 *r = p.records + 3 * (size_t)p.sorted_vals[i];
    return splat_patch_mask(r[0].x, r[0].y, r[0].z, r[0].w, r[1].x, r[1].y * r[1].z, tile_x0, tile_y0);
}
#else
__device__ __forceinline__ unsigned int load_patch_mask(const BlendBwdParams &p, int i, float, float) {
    return __ldg(p.patch_masks + i);
}
#endif

template <bool EXACT_EXP, bool STATS, bool COUNT = false>
__global__ void __launch_bounds__(GSB_TILE_PIXELS, tb_min_blocks(EXACT_EXP))
blend_backward_transposed_kernel(const BlendBwdParams p) {
    TbShared &S = *reinterpret_cast<TbShared *>(tb_dynamic_smem());
    constexpr int NV = STATS ? 11 : 9;

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
    unsigned int n_visits = 0, n_pairs = 0;  // COUNT only
    S.g[warp][lane] = make_float4(g0, g1, g2, 0.0f);

    // phase-2 role of this lane: splat `ci` of the chunk, pixels 16*half .. 16*half+15 of the patch (= rows 2*half, 2*half+1)
    const int ci = lane & (TB_CHUNK - 1), half = lane >> 4;
    const float pxb = tile_x0 + (float)((warp & 1) * 8) + 0.5f;
    const float pyb = tile_y0 + (float)((warp >> 1) * 4 + 2 * half) + 0.5f;
    float *const xg = S.xg[warp], *const xa = S.xa[warp];
    // flush role of this lane: word fl_word of the even (lanes 0..11) or odd (lanes 12..23) row of a row pair
    const int fl_row = lane >= GSB_ACCUM_FLOATS ? 1 : 0;
    const int fl_word = lane - GSB_ACCUM_FLOATS * fl_row;
    const bool fl_ok = lane < 2 * GSB_ACCUM_FLOATS && fl_word < NV;
    const float *const fl_val = xg + fl_row * TB_TR_ROW + (fl_ok ? fl_word : 0);
    int warp_last = last;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) warp_last = max(warp_last, __shfl_xor_sync(0xffffffffu, warp_last, d));

    // The walk: window w holds the keys top-1-lane for top = warp_last - 32 w (lane 0 the deepest).  `sel`: the keys of
    // the current window this patch can reach and that no chunk has taken yet; `val`: this lane's in-camera offset.
    const unsigned int bit = 1u << warp;
    const unsigned int lt_mask = (1u << lane) - 1u;
    int top = warp_last + 32;  // the current window (none yet)
    unsigned int sel = 0u;
    int val = 0;
    unsigned int next_mask = 0u;  // the next window, loaded one window ahead
    int next_val = 0;
    {
        const int i = warp_last - 1 - lane;
        if (i >= start) {
            next_mask = load_patch_mask(p, i, tile_x0, tile_y0);
            next_val = __ldg(p.sorted_vals + i);
        }
    }
    // Fills chunk buffer b with the next (up to) 16 splats of the walk and returns their number (warp-uniform); the records
    // arrive through cp.async (one group per call and lane).
    auto fill = [&](int b) -> int {
        float4 *const c0 = S.chunk[warp][b][0], *const c1 = S.chunk[warp][b][1], *const c2 = S.chunk[warp][b][2];
        int have = 0;
        while (have < TB_CHUNK) {
            if (sel == 0u) {  // next window
                top -= 32;
                if (top <= start) break;
                if (lane == 0) GSB_EMU_COUNT(EC_TB_WINDOWS, 1);
                const int i = top - 1 - lane;
                sel = __ballot_sync(0xffffffffu, i >= start && (next_mask & bit) != 0u);
                val = next_val;
                next_mask = 0u;
                if (i - 32 >= start) {
                    next_mask = load_patch_mask(p, i - 32, tile_x0, tile_y0);
                    next_val = __ldg(p.sorted_vals + i - 32);
                }
                continue;
            }
            const int take = min(__popc(sel), TB_CHUNK - have);
            const int rank = __popc(sel & lt_mask);
            const bool mine = (sel >> lane) & 1u;
            if (mine && rank < take) {
                const int slot = have + rank;
                const float4 *rec = p.records + 3 * (size_t)val;
                cp_async16(c0 + slot, rec);
                cp_async16(c1 + slot, rec + 1);
                cp_async16(c2 + slot, rec + 2);
                S.chunk_off[warp][b][slot] = val;
                S.chunk_idx[warp][b][slot] = top - 1 - lane;
            }
            // a full chunk leaves the rest of the window for the next one
            sel = take == TB_CHUNK - have ? __ballot_sync(0xffffffffu, mine && rank >= take) : 0u;
            have += take;
        }
        cp_async_commit();
        return have;
    };

    int buf = 0;
    int n = fill(0);
#pragma unroll 1
    while (n > 0) {
        const int n_next = fill(buf ^ 1);  // in flight while this chunk is computed
        cp_async_wait<1>();
        __syncwarp();
        float4 *const ck0 = S.chunk[warp][buf][0], *const ck1 = S.chunk[warp][buf][1], *const ck2 = S.chunk[warp][buf][2];
        int *const ck_off = S.chunk_off[warp][buf];
        const int *const fl_off = ck_off + fl_row;
        if (lane < n) {
            if (!EXACT_EXP) {  // the forward's staged planes (common.cuh): u v A B | C rescale*opacity 1-opacity depth
                float4 f0, f1;
                fast_planes(ck0[lane], ck1[lane], f0, f1);
                ck0[lane] = f0;
                ck1[lane] = f1;
            }
            ck2[lane].w = __int_as_float(S.chunk_idx[warp][buf][lane]);  // sorted index instead of the radius (unused here)
        }
        __syncwarp();
        if (COUNT) n_visits += (lane == 0) ? (unsigned int)n : 0u;
        if (lane == 0) {
            GSB_EMU_COUNT(EC_TB_SPLATS, n);
            GSB_EMU_COUNT(EC_TB_CHUNKS, 1);
        }
        // ---- phase 1: lane = pixel; sequential over the chunk's splats (back to front)
#pragma unroll TB_P1_UNROLL
        for (int i = 0; i < n; ++i) {
            const float4 r0 = ck0[i];  // u v a b                   (fast path: u v A B, conic scaled by -log2(e)/2)
            const float4 r1 = ck1[i];  // c rescale opacity depth   (fast path: C rescale*opacity 1-opacity depth)
            const float4 r2 = ck2[i];  // r g b | sorted index
            const int idx = __float_as_int(r2.w);
            const float d0 = px - r0.x, d1 = py - r0.y;
            float G, aT;
            if (EXACT_EXP) {
                const float q0 = r0.z * d0 + r0.w * d1;
                const float q1 = r0.w * d0 + r1.x * d1;
                const float gp = expf(-0.5f * (d0 * q0 + d1 * q1)) * r1.y;
                const float prod_alpha = gp * r1.z;
                const bool contributes = (idx < last) && (prod_alpha >= 1.0f / 255.0f);
                const float alpha = fminf(prod_alpha, 0.99f);
                const float inv = 1.0f / (1.0f - alpha);
                const float Tn = T * inv;
                aT = contributes ? alpha * Tn : 0.0f;
                const float a_grad = contributes ? (r2.x * Tn - w0 * inv) * g0 + (r2.y * Tn - w1 * inv) * g1 +
                                                       (r2.z * Tn - w2 * inv) * g2
                                                 : 0.0f;
                T = contributes ? Tn : T;
                w0 = fmaf(r2.x, aT, w0);
                w1 = fmaf(r2.y, aT, w1);
                w2 = fmaf(r2.z, aT, w2);
                G = a_grad * r1.z * gp;
                if (STATS) {
                    mag0 += fabsf(G * q0);
                    mag1 += fabsf(G * q1);
                }
            } else {
                // One-scalar colour recursion (see blend_bwd.cu); alpha is the FORWARD's expression on the forward's
                // staged values (fast_alpha, common.cuh), so both passes take the 1/255 decision on identical bits.
                // A pair that does not contribute gets P = 0: then alpha = 0, 1/(1-alpha) = 1, T and w0 keep their
                // values and G = aT = 0 -- no other select is needed.
                float P = fast_alpha(d0, d1, r0.z, r0.w, r1.x, r1.y);
                P = keep_if_contributing(P, idx, last);
                const float alpha = fminf(P, 0.99f);
                const float inv = rcp_approx(1.0f - alpha);
                T *= inv;                 // T_i = T_{i+1} / (1 - alpha), GPCR:640
                aT = alpha * T;
                const float cg = fmaf(r2.z, g2, fmaf(r2.y, g1, r2.x * g0));
                const float a_grad = fmaf(cg, T, -(w0 * inv));
                w0 = fmaf(cg, aT, w0);
                G = a_grad * P;
                if (STATS) {  // hook only: |d/duv| on the image needs conic * d  (A d0 + B/2 d1 = -log2(e)/2 q0)
                    const float q0 = (-2.0f / GSB_L2E) * fmaf(r0.z, d0, 0.5f * r0.w * d1);
                    const float q1 = (-2.0f / GSB_L2E) * fmaf(0.5f * r0.w, d0, r1.x * d1);
                    mag0 += fabsf(G * q0);
                    mag1 += fabsf(G * q1);
                }
            }
            if (COUNT) n_pairs += aT > 0.0f ? 1u : 0u;
            xg[lane * TB_ROW + i] = G;
            xa[lane * TB_ROW + i] = aT;
        }
        __syncwarp();

        // ---- phase 2: lane = splat ci of the chunk, over 16 pixels
        const bool active = ci < n;
        float4 s0 = ck0[active ? ci : 0];
        float4 s1 = ck1[active ? ci : 0];
        if (!EXACT_EXP) {  // back to the conic itself (the chunk holds it scaled by -log2(e)/2 for fast_alpha)
            s0.z *= -2.0f / GSB_L2E;
            s0.w *= -1.0f / GSB_L2E;
            s1.x *= -2.0f / GSB_L2E;
        }
        // conic * d at the first pixel of each of this lane's two rows; along a row d0 grows by exactly 1 per pixel, so
        // q0 += a, q1 += b (two FADD instead of two FMUL + two FFMA per pixel)
        const float dx0 = pxb - s0.x;
        float acc[11];
#pragma unroll
        for (int k = 0; k < 11; ++k) acc[k] = 0.0f;
        unsigned int nz = 0u;
#pragma unroll
        for (int row = 0; row < 2; ++row) {
            const float d1 = (pyb + (float)row) - s0.y;
            float q0 = s0.z * dx0 + s0.w * d1;
            float q1 = s0.w * dx0 + s1.x * d1;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int pp = 8 * row + k + 16 * half;  // the pixel = phase-1 lane
                const float G = xg[pp * TB_ROW + ci], aT = xa[pp * TB_ROW + ci];
                const float4 gp = S.g[warp][pp];
                const float vs0 = G * q0, vs1 = G * q1;
                acc[0] += vs0;
                acc[1] += vs1;
                acc[2] = fmaf(vs0, q0, acc[2]);  // the 1/2 of UT:345 is applied once per point in the epilogue kernel
                acc[3] = fmaf(vs0, q1, acc[3]);
                acc[4] = fmaf(vs1, q1, acc[4]);
                acc[5] = fmaf(aT, gp.x, acc[5]);
                acc[6] = fmaf(aT, gp.y, acc[6]);
                acc[7] = fmaf(aT, gp.z, acc[7]);
                acc[8] += G;
                if (STATS) {
                    const float m2 = vs0 * vs0 + vs1 * vs1;
                    acc[9] += EXACT_EXP ? sqrtf(m2) : sqrt_approx(m2);
                    acc[10] += aT > 0.0f ? 1.0f : 0.0f;  // alpha >= 1/255 and T > 0: alpha*T > 0 exactly for the contributing pixels
                }
                nz |= __float_as_uint(aT);
                q0 += s0.z;
                q1 += s0.w;
            }
        }
        // rows 0..1 + rows 2..3 of the patch
#pragma unroll
        for (int k = 0; k < NV; ++k) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], 16);
        nz |= __shfl_xor_sync(0xffffffffu, nz, 16);
        acc[8] *= EXACT_EXP ? (1.0f - s1.z) : s1.z;  // d alpha / d logit = alpha (1 - opacity)
        __syncwarp();  // every lane has consumed its xg / xa entries: xg now takes the finished rows
        if (lane < TB_CHUNK) {
            if (!(active && nz != 0u)) ck_off[ci] = -1;
            else GSB_EMU_COUNT(EC_TB_ROWS, 1);
#pragma unroll
            for (int k = 0; k < NV; ++k) xg[ci * TB_TR_ROW + k] = acc[k];
        }
        __syncwarp();
        // two rows per step: lanes 0..11 the words of row 2s, lanes 12..23 those of row 2s+1 (no index division)
#pragma unroll
        for (int step = 0; step < TB_CHUNK / 2; ++step) {
            const int o = fl_off[2 * step];
            const float v = fl_val[2 * step * TB_TR_ROW];
            if (fl_ok && o >= 0) atomicAdd(p.accum + (size_t)o * GSB_ACCUM_FLOATS + fl_word, v);
        }
        __syncwarp();  // the chunk after next overwrites this chunk buffer, and the next chunk xg
        buf ^= 1;
        n = n_next;
    }
    if (STATS) {
        p.mag_image[2 * pix] = mag0;  // GPCR:700-704
        p.mag_image[2 * pix + 1] = mag1;
    }
    if (COUNT) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            n_visits += __shfl_xor_sync(0xffffffffu, n_visits, d);
            n_pairs += __shfl_xor_sync(0xffffffffu, n_pairs, d);
        }
        if (lane == 0) {
            atomicAdd(p.work_counters, (unsigned long long)n_visits);
            atomicAdd(p.work_counters + 1, (unsigned long long)n_pairs);
        }
    }
}

#ifndef GSB_HOST_EMU
template <bool EXACT_EXP, bool STATS>
static int launch_tb(const BlendBwdParams &p, int tiles, cudaStream_t stream) {
    static bool configured = false;  // one device per process (one process per GPU)
    if (!configured) {
        GSB_CUDA_CHECK(cudaFuncSetAttribute(blend_backward_transposed_kernel<EXACT_EXP, STATS>,
                                            cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(TbShared)));
        configured = true;
    }
    blend_backward_transposed_kernel<EXACT_EXP, STATS><<<tiles, GSB_TILE_PIXELS, sizeof(TbShared), stream>>>(p);
    GSB_CUDA_CHECK(cudaGetLastError());
    return GSB_OK;
}

int launch_blend_backward_transposed(const BlendBwdParams &p, int tiles, bool exact_exp, bool stats,
                                     cudaStream_t stream) {
    if (exact_exp) return stats ? launch_tb<true, true>(p, tiles, stream) : launch_tb<true, false>(p, tiles, stream);
    return stats ? launch_tb<false, true>(p, tiles, stream) : launch_tb<false, false>(p, tiles, stream);
}

// Diagnostic: loop A with GPU-side work counters (default arithmetic, no hook statistics): counters[0] = (warp, splat)
// visits of phase 1, [1] = contributing (pixel, splat) pairs.  Adds into p.accum like the normal launch.
int launch_blend_backward_count(const BlendBwdParams &p, int tiles, cudaStream_t stream) {
    GSB_CUDA_CHECK(cudaFuncSetAttribute(blend_backward_transposed_kernel<false, false, true>,
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(TbShared)));
    blend_backward_transposed_kernel<false, false, true><<<tiles, GSB_TILE_PIXELS, sizeof(TbShared), stream>>>(p);
    GSB_CUDA_CHECK(cudaGetLastError());
    return GSB_OK;
}
#endif  // GSB_HOST_EMU

}  // namespace gsb
