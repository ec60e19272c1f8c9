// Host build of the Layout part of arap_flow_b200/csrc/devmem.cuh for tests/test_devmem.py (g++, no CUDA): the carves
// of the library's device buffers, block for block in the order the .cu files take them.
#include "../arap_flow_b200/csrc/devmem.cuh"

#include <cstddef>

using arapb200::Layout;

extern "C" {

// pipeline.cu run(), a slot's extras: bflow, occ, bytes
void dm_extras(size_t N, size_t* o)
{
    Layout l;
    o[0] = l.take(8 * N);
    o[1] = l.take(N);
    o[2] = l.bytes();
}

// pipeline.cu run(), a slot's frames: pos, z, rgb, mask, flow, bflow, occ, flow0, bytes
void dm_frames(size_t N, size_t K, size_t* o)
{
    const size_t F = N * K;
    Layout l;
    o[0] = l.take(8 * F);
    o[1] = l.take(2 * 4 * N);
    o[2] = l.take(3 * F);
    o[3] = l.take(F);
    o[4] = l.take(8 * F);
    o[5] = l.take(8 * F);
    o[6] = l.take(F);
    o[7] = l.take(8 * F);
    o[8] = l.bytes();
}

// pipeline.cu SceneLayout, K frames after the pair: bg, rgb0, flow, rgb, mask, bflow, occ, bytes
void dm_scene(size_t W, size_t H, size_t bgW, size_t bgH, size_t K, int rgb0, size_t* o)
{
    const size_t N = W * H, F = N * (K + 1);
    Layout l;
    o[0] = l.take(3 * bgW * bgH);
    o[1] = l.take(rgb0 ? 3 * N : 0);
    o[2] = l.take(8 * F);
    o[3] = l.take(3 * F);
    o[4] = l.take(F);
    o[5] = l.take(8 * F);
    o[6] = l.take(F);
    o[7] = l.bytes();
}

// arapb200_api.cu warp_common: in, pos, z, rgb, orgb, m, om, bf, fl, occ, bytes
void dm_warp(size_t N, int ex, int occ, size_t* o)
{
    Layout l;
    o[0] = l.take(8 * N);
    o[1] = l.take(8 * N);
    o[2] = l.take(4 * N);
    o[3] = l.take(3 * N);
    o[4] = l.take(3 * N);
    o[5] = l.take(N);
    o[6] = l.take(N);
    o[7] = l.take(ex ? 8 * N : 0);
    o[8] = l.take(occ ? 8 * N : 0);
    o[9] = l.take(occ ? N : 0);
    o[10] = l.bytes();
}

// composite.cu flatten_common: per layer flow, rgb, mask, bflow, src; then bg, flow, rgb, mask, bflow, occ, bytes
void dm_flatten(size_t N, int n_layers, int background, int out_bflow, int out_occ, size_t* o)
{
    const bool ex = out_bflow || out_occ;
    Layout l;
    for (int s = 0; s < n_layers; ++s, o += 5) {
        o[0] = l.take(8 * N);
        o[1] = l.take(3 * N);
        o[2] = l.take(N);
        o[3] = l.take(ex ? 8 * N : 0);
        o[4] = l.take(out_occ ? N : 0);
    }
    o[0] = l.take(background ? 3 * N : 0);
    o[1] = l.take(8 * N);
    o[2] = l.take(3 * N);
    o[3] = l.take(N);
    o[4] = l.take(out_bflow ? 8 * N : 0);
    o[5] = l.take(out_occ ? N : 0);
    o[6] = l.bytes();
}

// composite.cu arapb200_composite: per layer flow, rgb, mask, src, bflow; then bg, flow, rgb, mask, bflow, occ, bytes
void dm_composite(size_t N, size_t NB, int n_layers, int ex, int out_occ, size_t* o)
{
    Layout l;
    for (int s = 0; s < n_layers; ++s, o += 5) {
        o[0] = l.take(8 * N);
        o[1] = l.take(3 * N);
        o[2] = l.take(N);
        o[3] = l.take(N);
        o[4] = l.take(ex ? 8 * N : 0);
    }
    o[0] = l.take(3 * NB);
    o[1] = l.take(8 * N);
    o[2] = l.take(3 * N);
    o[3] = l.take(N);
    o[4] = l.take(ex ? 8 * N : 0);
    o[5] = l.take(out_occ ? N : 0);
    o[6] = l.bytes();
}
}
