// emu_patch_masks.cpp -- the forward blend and loop A of the backward compiled as host C++ under simt_emu.h, with the reach
// masks the forward records for the backward (BlendFwdParams / BlendBwdParams::patch_masks) passed in and out explicitly.
// TEST INFRASTRUCTURE, see simt_emu.h; built by tests/test_simt_patch_masks_cpu.py with g++.
#include "simt_emu.h"
// the kernel sources, unmodified (their launchers are compiled out under GSB_HOST_EMU)
#include "../../taichi_3d_gaussian_splatting_b200/csrc/blend_fwd.cu"
#include "../../taichi_3d_gaussian_splatting_b200/csrc/blend_bwd.cu"
#include "../../taichi_3d_gaussian_splatting_b200/csrc/blend_bwd_transposed.cu"

namespace gsb {
void set_error(const char *, ...) {}
}  // namespace gsb

// masks_out[k] = splat_patch_mask of sorted key k against its tile, for every key of every tile
extern "C" void emu_patch_masks(int H, int W, const int *tile_start, const int *tile_end, const int *sorted_vals,
                                const float *records, unsigned char *masks_out) {
    const int tiles_x = W / GSB_TILE_WIDTH, tiles = tiles_x * (H / GSB_TILE_HEIGHT);
    for (int t = 0; t < tiles; ++t) {
        const float x0 = (float)((t % tiles_x) * GSB_TILE_WIDTH), y0 = (float)((t / tiles_x) * GSB_TILE_HEIGHT);
        for (int i = tile_start[t]; i < tile_end[t]; ++i) {
            const float *r = records + 12 * (size_t)sorted_vals[i];
            masks_out[i] = (unsigned char)gsb::splat_patch_mask(r[0], r[1], r[2], r[3], r[4], r[5] * r[6], x0, y0);
        }
    }
}

// the forward blend; patch_masks (one byte per sorted key) receives the reach mask of every key it stages unless rgb_only
extern "C" long long emu_blend_forward_masks(int rgb_only, int exact_exp, int H, int W, const int *tile_start,
                                             const int *tile_end, const int *sorted_vals, const float *records, float *image,
                                             float *depth, float *acc_alpha, int *last_effective, int *valid_count,
                                             unsigned char *patch_masks) {
    using namespace gsb;
    BlendFwdParams p;
    p.H = H;
    p.W = W;
    p.tiles_x = W / GSB_TILE_WIDTH;
    p.tile_start = tile_start;
    p.tile_end = tile_end;
    p.sorted_vals = sorted_vals;
    p.records = reinterpret_cast<const float4 *>(records);
    p.image = image;
    p.depth = depth;
    p.acc_alpha = acc_alpha;
    p.last_effective = last_effective;
    p.valid_count = valid_count;
    p.patch_masks = patch_masks;
    const int tiles = p.tiles_x * (H / GSB_TILE_HEIGHT);
    simt_emu::M().switches = 0;
    if (rgb_only) {
        if (exact_exp) simt_emu::launch(blend_forward_kernel<true, true>, tiles, GSB_TILE_PIXELS, p);
        else simt_emu::launch(blend_forward_kernel<true, false>, tiles, GSB_TILE_PIXELS, p);
    } else {
        if (exact_exp) simt_emu::launch(blend_forward_kernel<false, true>, tiles, GSB_TILE_PIXELS, p);
        else simt_emu::launch(blend_forward_kernel<false, false>, tiles, GSB_TILE_PIXELS, p);
    }
    return simt_emu::M().switches;
}

// loop A of the backward (transposed: blend_bwd_transposed.cu, else the butterfly kernel of blend_bwd.cu, which runs its own
// reach tests) fed with the given reach masks, one byte per sorted key as the forward writes them
extern "C" long long emu_blend_backward_masks(int transposed, int exact_exp, int stats, int H, int W, const int *tile_start,
                                              const int *tile_end, const int *sorted_vals, const float *records,
                                              const unsigned char *patch_masks, const float *grad_image,
                                              const float *acc_alpha, const int *last_effective, float *accum,
                                              float *mag_image) {
    using namespace gsb;
    BlendBwdParams p;
    p.H = H;
    p.W = W;
    p.tiles_x = W / GSB_TILE_WIDTH;
    p.tile_start = tile_start;
    p.tile_end = tile_end;
    p.sorted_vals = sorted_vals;
    p.records = reinterpret_cast<const float4 *>(records);
    p.grad_image = grad_image;
    p.acc_alpha = acc_alpha;
    p.last_effective = last_effective;
    p.patch_masks = patch_masks;
    p.accum = accum;
    p.mag_image = mag_image;
    const int tiles = p.tiles_x * (H / GSB_TILE_HEIGHT);
    simt_emu::M().switches = 0;
    if (!transposed) {
        if (exact_exp && stats) simt_emu::launch(blend_backward_kernel<true, true>, tiles, GSB_TILE_PIXELS, p);
        else if (exact_exp) simt_emu::launch(blend_backward_kernel<true, false>, tiles, GSB_TILE_PIXELS, p);
        else if (stats) simt_emu::launch(blend_backward_kernel<false, true>, tiles, GSB_TILE_PIXELS, p);
        else simt_emu::launch(blend_backward_kernel<false, false>, tiles, GSB_TILE_PIXELS, p);
    } else if (exact_exp) {
        if (stats) simt_emu::launch(blend_backward_transposed_kernel<true, true>, tiles, GSB_TILE_PIXELS, p);
        else simt_emu::launch(blend_backward_transposed_kernel<true, false>, tiles, GSB_TILE_PIXELS, p);
    } else {
        if (stats) simt_emu::launch(blend_backward_transposed_kernel<false, true>, tiles, GSB_TILE_PIXELS, p);
        else simt_emu::launch(blend_backward_transposed_kernel<false, false>, tiles, GSB_TILE_PIXELS, p);
    }
    return simt_emu::M().switches;
}
