// Interface between conv2d_tc.cu (argument checks, tensor maps, dispatch) and the grouped 3x3 kernels: conv3x3_ring.cu (row ring)
// and gconv3x3_tapn.cu (horizontal taps stacked along N).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

struct RingP {
    int N, H, W, C;          // images, rows, columns (ring: multiple of 128; tapn: 64 or 128), channels (multiple of 64; Cin == Cout, grouped)
    int planes, wplanes;     // activation / weight bf16 planes (1 or 2)
    int relu;                // 0 none, 1 ReLU
    int segs, seg_rows;      // row segments per (image, column tile, channel block) strip and rows per segment (set by the launcher)
    int pdl;                 // launched with programmatic stream serialization (griddepcontrol.wait before the first global read)
    int dbg;                 // gconv3x3_tapn: HEAL_TC_DBG timing bits (results invalid): 1 no epilogue, 4 no activation loads, 16 no MMAs
    const float* bias;       // [C] or null
};

// tmA: activations {C, W, H, N, plane}, box {64, 130, 1, 1, planes}, 128B swizzle (the halo map of heal_conv2d_tc)
// tmB: packed diagonal weight sub-blocks, box {16, 16, wplanes, 4, 3}, 32B swizzle
// tmO: output {C, W, H, N, plane}, box {64, 128, 1, 1, planes}, 128B swizzle
int heal_conv3x3_ring_launch(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmO, RingP p, cudaStream_t st);

// W 64 or 128, split weights (wplanes 2).
// tmA: activations {C, W, H, N, plane}, box {64, W, 1, 1, 1}, 128B swizzle (one row of one plane per load)
// tmB: packed diagonal weight sub-blocks {16 ci, 16 co, 9 taps, plane, C / 16 sub-blocks}, box {16, 16, 3, 2, 4}, 32B swizzle
// tmO: output {C, W, H, N, plane}, box {64, W, 128 / W, 1, planes}, 128B swizzle
int heal_gconv3x3_tapn_launch(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmO, RingP p, cudaStream_t st);
