// Implicit-GEMM 2-D convolution on the 5th-generation tensor cores (tcgen05.mma, accumulators in TMEM),
// operands staged by TMA (cp.async.bulk.tensor) with the 128-byte swizzle, warp-specialised and persistent.
//
// Replaces the dense convolutions of the BEV backbones / ResNeXt pyramid / shrink header
// (reference: resblock.py:48-64,102-122; base_bev_backbone.py:40-86; base_bev_backbone_resnet.py:54-85;
//  downsample_conv.py:16-27) with BN folded, and ReLU / residual / bias in the epilogue.
//
// Precision ("split-bf16", fp32-equivalent): an fp32 value x is stored as two bf16 planes hi = bf16(x),
// lo = bf16(x - hi) (16 mantissa bits).  A product a*b is evaluated as a_hi*b_hi + a_hi*b_lo + a_lo*b_hi
// with fp32 accumulation in TMEM: three tcgen05.mma per K step into the same accumulator, relative
// error ~2^-16 per product, which keeps 70 stacked layers inside the 1e-3 fp32 parity tolerance that plain
// bf16 / tf32 tensor-core math cannot meet.  With planes == 1 the same kernel is a plain bf16 conv.
//
// GEMM view: M = output pixels (tile = TH x TW = 128 pixels of one image), N = output channels,
// K = taps x Cin in blocks of 64 channels.  A tile for tap (r,s) is ONE 5-D TMA box of the activation
// tensor {C, W, H, N, plane} at (c0, w0+s-pad, h0+r-pad, n, 0); out-of-bounds elements are zero-filled
// by the TMA unit, which implements the convolution padding.  B tiles come from the packed weights
// {Cin, taps*CoutPad, plane}.
//
// Roles (320 threads): warp 0 = TMA producer, warp 1 = MMA issuer + TMEM allocator (both loop as converged warps and issue
// under elect.sync so the tcgen05 / TMA instructions stay on the uniform datapath), warps 2..9 = epilogue, two warps per
// TMEM lane quarter (TMEM -> registers -> bias / residual / ReLU -> hi/lo split -> swizzled smem staging -> one
// cp.async.bulk.tensor store per 64-channel chunk; fp32 / transposed-conv outputs use direct stores).
// Two TMEM accumulator buffers let the epilogue of tile i overlap the MMAs of tile i+1.
// Modes: stride 2 through TMA element strides; grouped 3x3 as 16-channel sub-block MMAs on block-diagonal 64-channel
// tiles; "halo" (3x3, stride 1, one-row tiles, N = 64): one activation box of TW+2 pixels per kernel ROW, the three
// horizontal taps are row-shifted descriptors of the same smem tile (3x less L2->smem activation traffic).
// HEAL_TC_* environment switches are measurement hooks (profiles/tc_experiment.py), not product paths.
#include <cuda.h>
#include <stdlib.h>
#include "common.cuh"
#include "tc_prims.cuh"
#include "conv_ring.cuh"
#include "../../include/heal_b200.h"

namespace {

constexpr int TC_THREADS = 320;      // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue (2 per TMEM lane quarter)
constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;                 // bf16 elements = 128 B = one swizzle row
constexpr int A_TILE_BYTES = BLOCK_M * BLOCK_K * 2;   // 16 KiB per plane

struct TcP {
    int N, Ho, Wo, Cout;          // output grid (conv resolution) and real output channels
    int taps_w, taps, pad;        // kw, kh*kw, padding
    int stride;                   // conv stride (TMA element stride on W and H)
    int blockdiag;                // grouped conv as block-diagonal 64x64 channel blocks: n-tile nt reads channel block nt only
    int bdiag;                    // block-diagonal weights arrive packed: only the four 16x16 diagonal sub-blocks ([16 rows][32 B], 32B swizzle)
    int kc_blocks;                // Cin / 64
    int TH, TW, tiles_h, tiles_w; // pixel tile and tile grid per image
    int m_tiles, n_tiles;
    int planes;                   // ACTIVATION planes: 1 = bf16, 2 = split-bf16 (fp32-equivalent)
    int wplanes;                  // WEIGHT planes: 2 = split weights (hi + lo).  planes 1 + wplanes 2 = the 'bf16' engine mode:
                                  // bf16 activations x un-rounded (16-mantissa-bit) weights, a_hi x [b_hi | b_lo]
    int coutp;                    // padded Cout rows per tap in the weight matrix (multiple of BLOCK_N)
    int relu;                     // epilogue activation: 0 none, 1 ReLU, 2 GELU (erf)
    int up;                       // transposed conv (k == stride == up): n-tile -> (i,j) sub-position
    int pdl;                      // launched with programmatic stream serialization
    int bo_mode;                  // experiment: base-offset convention of the halo descriptors
    int halo;                     // 3x3 stride-1, one-row tiles: ONE activation load per kernel ROW (TW+2 pixels) serves the 3 horizontal taps
    int tma_out;                  // epilogue drains through shared memory + TMA tensor store (tmO valid)
    int res_tma;                  // STG >= 2: the residual chunk is TMA-loaded into the staging buffer one chunk ahead (tmR valid)
    int dbg;                      // HEAL_TC_DBG experiment bits (timing only, results invalid): 1 no stores, 2 no B loads, 4 no A loads, 8 no residual loads (TMA-store epilogue), 16 no MMAs
    const float* bias;            // [Cout]
    // residual (optional): split planes or fp32
    const __nv_bfloat16* res_split; size_t res_plane; const float* res_f32; int res_cs, res_co;
    // outputs (either or both)
    __nv_bfloat16* out_split; size_t out_plane; int out_cs, out_co;
    float* out_f32; int out32_cs, out32_co;
};

// STG = number of 64-channel output staging buffers in shared memory (0: the epilogue stores straight to global memory;
// >0: it writes the swizzled tile to smem and one elected thread issues a TMA tensor store, so every global write is a
// full coalesced line and the drain is asynchronous).
// GELU: the exact-erf GELU epilogue (ConvNeXt pwconv1) lives in its OWN instantiations: this kernel is sensitive to code size
// (an erff call inside every instantiation's epilogue cost the ReLU paths ~4 % of the C2 frame, A/B on the bench)
template <int BLOCK_N, int STAGES, int STG, bool GELU = false>
__global__ void __launch_bounds__(TC_THREADS, 1)
k_conv2d_tc(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
            const __grid_constant__ CUtensorMap tmO, const __grid_constant__ CUtensorMap tmR, const TcP p) {
    // 1024 B alignment for the 128B swizzle atoms: requested from the toolchain (no slack bytes to round up inside -- the halo +
    // two-staging-buffer configuration needs all 227 KiB) and checked once.  The pointer is laundered through an empty asm so
    // that shared-memory addresses stay run-time values: with compile-time-constant addresses ptxas emits a slower kernel
    // (measured A/B on one box: level-0 1x1 conv 51 -> 66 us).
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uintptr_t raw_addr = reinterpret_cast<uintptr_t>(smem_raw);
    asm volatile("" : "+l"(raw_addr));
    uint8_t* smem = reinterpret_cast<uint8_t*>(raw_addr);
    if (smem_u32(smem) & 1023u) __trap();
    // weight bytes per (tap, plane) in a stage: a BLOCK_N x 64 tile, or (grouped, packed) the four 16x16 diagonal sub-blocks
    const int B_TILE_BYTES = p.bdiag ? (BLOCK_N / 16) * 512 : BLOCK_N * BLOCK_K * 2;
    // halo mode: A = [plane][TW+2 rows][128 B] (padded to 1 KiB), B = [plane][3 taps][BLOCK_N rows][128 B]
    const int halo_a_plane = (p.TW + 2) * 128;
    const int halo_a_bytes = (p.planes * halo_a_plane + 1023) & ~1023;
    const int stage_bytes = p.halo ? (halo_a_bytes + p.wplanes * 3 * B_TILE_BYTES) : (p.planes * A_TILE_BYTES + p.wplanes * B_TILE_BYTES);
    const int stg_bytes = p.planes * A_TILE_BYTES;                        // one staging buffer: [plane][128 rows][128 B]
    uint8_t* stg = smem + (size_t)STAGES * stage_bytes;                   // 1024-aligned (stage_bytes is a multiple of 1024)
    uint64_t* bars = reinterpret_cast<uint64_t*>(stg + (size_t)STG * stg_bytes);
    // bars: full[STAGES], empty[STAGES], tmem_full[2], tmem_empty[2], (spare), residual_full[3]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 8);
    const uint32_t bar_res = smem_u32(bars + 2 * STAGES + 5);
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t bar_full = smem_u32(bars), bar_empty = smem_u32(bars + STAGES);
    const uint32_t bar_tfull = smem_u32(bars + 2 * STAGES), bar_tempty = smem_u32(bars + 2 * STAGES + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // Split-bf16 products a_hi*b_hi + a_hi*b_lo + a_lo*b_hi.  For BLOCK_N <= 64 the hi and lo weight planes sit next to each other
    // in shared memory, so ONE MMA with N' = 2N computes a_hi x [b_hi | b_lo] (main | aux accumulator columns) and a second
    // N-wide MMA adds a_lo x b_hi: 2 tensor-core instructions and 2 reads of the A slice per K step instead of 3 (these tile
    // shapes are bound by the A-operand shared-memory reads: a 128x16 N=16 MMA costs ~2/3 of an N=128 one).  The epilogue
    // adds aux to main.  BLOCK_N = 128 keeps 3 MMAs (N' = 256 would be the same tensor time and needs all of TMEM).
    constexpr bool NCAT = (BLOCK_N <= 64);
    constexpr int ACC_STRIDE = NCAT ? 2 * BLOCK_N : BLOCK_N;      // TMEM columns per accumulator buffer
    constexpr int TMEM_COLS = (2 * ACC_STRIDE < 32) ? 32 : 2 * ACC_STRIDE;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(bar_tfull + 8 * a, 1); mbar_init(bar_tempty + 8 * a, 256); }
        for (int a = 0; a < 3; ++a) mbar_init(bar_res + 8 * a, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // Programmatic dependent launch: everything above (barrier init, TMEM allocation) overlapped the tail of the previous
    // kernel in the stream / graph; from here on we touch memory it produced, so wait for it, and let the next kernel start
    // its own prologue as soon as our CTAs begin to drain.
    if (p.pdl) {
        asm volatile("griddepcontrol.wait;" ::: "memory");
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    }

    const int total_tiles = p.m_tiles * p.n_tiles;
    const int kcn = p.blockdiag ? 1 : p.kc_blocks;      // channel blocks per tap visited by one tile
    const int kblocks = (p.halo ? 3 : p.taps) * kcn;    // halo mode: one k-block per kernel ROW (3 taps each)

    if (warp == 0) {
        // ============================== TMA producer (whole warp loops, one elected lane issues) ==
        {
            int stage = 0; uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const int nt = tile % p.n_tiles, mt = tile / p.n_tiles;
                const int tw_i = mt % p.tiles_w; const int t2 = mt / p.tiles_w;
                const int th_i = t2 % p.tiles_h; const int img = t2 / p.tiles_h;
                const int h0 = th_i * p.TH, w0 = tw_i * p.TW;
                for (int kb = 0; kb < kblocks; ++kb) {
                    const int tap = kb / kcn, kc = p.blockdiag ? nt : kb % kcn;
                    const int r = tap / p.taps_w, s = tap % p.taps_w;
                    mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                    if (p.halo) {
                        // k-block = (kernel row tap, channel block): pixels [w0-1, w0+TW] of input row h0+tap-1, and the 3 taps' weights
                        const uint32_t sa = smem_base + stage * stage_bytes, sb = sa + halo_a_bytes;
                        if (elect_one()) {
                            mbar_expect_tx(bar_full + 8 * stage, (uint32_t)(p.planes * halo_a_plane + p.wplanes * 3 * B_TILE_BYTES));
                            tma_load_5d(sa, &tmA, bar_full + 8 * stage, kc * BLOCK_K, w0 - 1, h0 + tap - 1, img, 0);
                            // B lands as [tap][plane][rows] (dense) or [tap][16-row sub-block][plane][16 rows] (block-diagonal)
                            if (p.blockdiag) tma_load_5d(sb, &tmB, bar_full + 8 * stage, 0, 0, 0, nt * (BLOCK_N / 16), tap * 3);
                            else tma_load_4d(sb, &tmB, bar_full + 8 * stage, kc * BLOCK_K, nt * BLOCK_N, 0, tap * 3);
                        }
                        __syncwarp();
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                        continue;
                    }
                    const uint32_t sa = smem_base + stage * stage_bytes;
                    const uint32_t sb = sa + p.planes * A_TILE_BYTES;
                    const bool ldA = !(p.dbg & 4), ldB = !(p.dbg & 2);
                    if (elect_one()) {
                        mbar_expect_tx(bar_full + 8 * stage, (uint32_t)((ldA ? p.planes * A_TILE_BYTES : 0) + (ldB ? p.wplanes * B_TILE_BYTES : 0)));
                        if (ldA) tma_load_5d(sa, &tmA, bar_full + 8 * stage, kc * BLOCK_K, w0 * p.stride + s - p.pad, h0 * p.stride + r - p.pad, img, 0);
                        if (ldB) {
                            if (p.blockdiag) tma_load_4d(sb, &tmB, bar_full + 8 * stage, 0, 0, 0, (tap * p.coutp + nt * BLOCK_N) / 16);   // [sub-block][plane][16 rows]
                            else tma_load_3d(sb, &tmB, bar_full + 8 * stage, kc * BLOCK_K, tap * p.coutp + nt * BLOCK_N, 0);                // [plane][rows]
                        }
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ============================== MMA issuer (whole warp loops, one elected lane issues) ====
        {
            // instruction descriptor: D=f32, A=B=bf16, K-major both, N>>3 @17, M>>4 @24
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BLOCK_N >> 3) << 17) | ((uint32_t)(BLOCK_M >> 4) << 24);
            const uint32_t idesc16 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(16 >> 3) << 17) | ((uint32_t)(BLOCK_M >> 4) << 24);
            // N-concatenated forms (NCAT): N' = 2N
            const uint32_t idesc_cat = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)((2 * BLOCK_N) >> 3) << 17) | ((uint32_t)(BLOCK_M >> 4) << 24);
            const uint32_t idesc32 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(32 >> 3) << 17) | ((uint32_t)(BLOCK_M >> 4) << 24);
            const bool split = (p.planes == 2);                      // activations carry a lo plane
            const bool wsplit = (p.wplanes == 2);                    // weights carry a lo plane
            const int sub_cols = (NCAT && wsplit) ? 32 : 16;         // accumulator columns per 16-channel diagonal sub-block
            const int sub_bytes = p.wplanes * 2048;                  // smem bytes per sub-block: [plane][16 rows][128 B]
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                mbar_wait(bar_tempty + 8 * acc, acc_phase ^ 1);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + (uint32_t)(acc * ACC_STRIDE);
                for (int kb = 0; kb < kblocks; ++kb) {
                    mbar_wait(bar_full + 8 * stage, phase);
                    tc_fence_after();
                    // A: [plane][rows][128 B]; halo mode: tap s reads rows [s, s+128) of the (TW+2)-row tile (start address + s*128 B;
                    // the swizzle is a function of the absolute smem address, so no base offset)
                    const uint32_t sa = smem_base + stage * stage_bytes;
                    const uint32_t a_plane = p.halo ? (uint32_t)halo_a_plane : (uint32_t)A_TILE_BYTES;
                    const uint32_t sb = sa + (p.halo ? (uint32_t)halo_a_bytes : (uint32_t)(p.planes * A_TILE_BYTES));
                    const int ntap = p.halo ? 3 : 1;
                    if (elect_one()) {
                        if (!(p.dbg & 16))
                        for (int s = 0; s < ntap; ++s) {
                            const uint32_t ah = sa + s * 128, al = ah + a_plane;
                            const uint32_t bs = sb + s * p.wplanes * B_TILE_BYTES;
#pragma unroll
                            for (int k = 0; k < BLOCK_K / 16; ++k) {
                                const uint64_t a_hi = umma_desc_sw128_off(ah + k * 32, p.bo_mode), a_lo = umma_desc_sw128_off(al + k * 32, p.bo_mode);
                                if (p.blockdiag) {
                                    // Grouped conv: channels-per-group divides 16, so output channels [16k,16k+16) of this 64-block depend
                                    // only on input channels [16k,16k+16): one M128 x N16 x K16 product per 16-channel sub-block.
                                    // sub-block k: [plane][16 rows] of 128 B rows at K offset k*16 elements, or packed 32 B rows
                                    const uint32_t bk = p.bdiag ? bs + k * p.wplanes * 512 : bs + k * sub_bytes + k * 32;
                                    const uint64_t bd = p.bdiag ? umma_desc_sw32(bk) : umma_desc_sw128(bk);
                                    const uint32_t td = tmem_d + (uint32_t)(k * sub_cols);
                                    const uint32_t f0 = (kb == 0 && s == 0) ? 0u : 1u;
                                    if constexpr (NCAT) {
                                        if (wsplit) {
                                            umma_bf16(td, a_hi, bd, idesc32, f0);                 // [a_hi*b_hi | a_hi*b_lo]
                                            if (split) umma_bf16(td, a_lo, bd, idesc16, 1u);      // += a_lo*b_hi
                                        } else {
                                            umma_bf16(td, a_hi, bd, idesc16, f0);
                                        }
                                    }
                                } else {
                                    const uint32_t first = (kb == 0 && s == 0 && k == 0) ? 0u : 1u;
                                    const uint64_t b_hi = umma_desc_sw128(bs + k * 32);
                                    if (!wsplit) {
                                        umma_bf16(tmem_d, a_hi, b_hi, idesc, first);
                                    } else if constexpr (NCAT) {
                                        umma_bf16(tmem_d, a_hi, b_hi, idesc_cat, first);                // [a_hi*b_hi | a_hi*b_lo]
                                        if (split) umma_bf16(tmem_d, a_lo, b_hi, idesc, 1u);            // += a_lo*b_hi
                                    } else {
                                        const uint64_t b_lo = umma_desc_sw128(bs + B_TILE_BYTES + k * 32);
                                        umma_bf16(tmem_d, a_hi, b_lo, idesc, first);
                                        if (split) umma_bf16(tmem_d, a_lo, b_hi, idesc, 1u);
                                        umma_bf16(tmem_d, a_hi, b_hi, idesc, 1u);
                                    }
                                }
                            }
                        }
                        umma_commit(bar_empty + 8 * stage);       // smem slot free once these MMAs retire
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                if (elect_one()) umma_commit(bar_tfull + 8 * acc);   // accumulator ready for the epilogue
                __syncwarp();
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ============================== epilogue (warps 2..5) =====================
        const int quarter = warp & 3;                   // TMEM lane quarter this warp may access
        const int chalf = (warp - 2) >> 2;              // which half of the tile's column chunks this warp drains
        const int row = quarter * 32 + lane;            // accumulator row = pixel within the tile
        constexpr int CHUNK = (BLOCK_N >= 32) ? 32 : 16;
        int acc = 0; uint32_t acc_phase = 0;
        int stg_count = 0;
        // Residual prefetch (TMA-store epilogue, split/bf16 residual): the 2 x 4 x 16 B of this thread's row for the NEXT 64-channel
        // chunk are requested one chunk ahead, so their DRAM latency hides behind the current chunk (and the wait for the MMAs)
        // instead of stalling every 8-channel group (measured: level-0 conv3 105 -> 44 us with the loads removed).
        // CH logical accumulator columns [col0, col0+CH) of buffer `acc` -> raw (fp32 bits); with the N-concatenated split MMAs the
        // value is main + aux: dense = columns c and BLOCK_N + c, block-diagonal = per 16-channel sub-block [main16 | aux16].
        auto ld_acc = [&](int col0, uint32_t* raw) {
            const uint32_t tb = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * ACC_STRIDE);
            if (NCAT && p.wplanes == 2) {
                uint32_t y[CHUNK];
                if constexpr (CHUNK == 32) {
                    if (p.blockdiag) {
                        tmem_ld32(tb + (uint32_t)(2 * col0), raw); tmem_ld32(tb + (uint32_t)(2 * col0 + 32), y);
                        tmem_wait_ld();
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            raw[j] = __float_as_uint(__uint_as_float(raw[j]) + __uint_as_float(raw[16 + j]));
                            raw[16 + j] = __float_as_uint(__uint_as_float(y[j]) + __uint_as_float(y[16 + j]));
                        }
                        return;
                    }
                    tmem_ld32(tb + (uint32_t)col0, raw); tmem_ld32(tb + (uint32_t)(BLOCK_N + col0), y);
                } else {
                    tmem_ld16(tb + (uint32_t)col0, raw); tmem_ld16(tb + (uint32_t)(BLOCK_N + col0), y);
                }
                tmem_wait_ld();
#pragma unroll
                for (int j = 0; j < CHUNK; ++j) raw[j] = __float_as_uint(__uint_as_float(raw[j]) + __uint_as_float(y[j]));
            } else {
                if constexpr (CHUNK == 32) tmem_ld32(tb + (uint32_t)col0, raw); else tmem_ld16(tb + (uint32_t)col0, raw);
                tmem_wait_ld();
            }
        };
        uint4 rn_h[4], rn_l[4];
        // compiled only into the instantiations that are dispatched with a residual (<*,2,3> and the halo <64,2,2>): the extra
        // single-thread TMA issue path costs the others ~800 R2UR moves and 5-40 % of their speed (measured A/B on one box)
        constexpr bool RES_TMA_OK = (STG == 3) || (STG == 2 && BLOCK_N == 64 && STAGES == 2);
        const bool res_tma = RES_TMA_OK && p.res_tma && !(p.dbg & 8);
        constexpr bool RES_PF = (STG == 1 && BLOCK_N == 64);      // the halo configuration: no room for 3 staging buffers
        const bool res_pf = RES_PF && p.tma_out && p.res_split && !(p.dbg & 8);
        auto res_fetch = [&](int tile_, int c64_) {
            const int nt_ = tile_ % p.n_tiles, mt_ = tile_ / p.n_tiles;
            const int tw_ = mt_ % p.tiles_w; const int t2_ = mt_ / p.tiles_w;
            const int th_ = t2_ % p.tiles_h; const int img_ = t2_ / p.tiles_h;
            const int oh_ = th_ * p.TH + row / p.TW, ow_ = tw_ * p.TW + row % p.TW;
            const int ng_ = nt_ * BLOCK_N;
            const int q_ = ng_ / p.coutp, c0_ = ng_ % p.coutp + c64_ * 64 + chalf * 32;
            const size_t pix_ = ((size_t)img_ * (p.Ho * p.up) + (size_t)(oh_ * p.up + q_ / p.up)) * (size_t)(p.Wo * p.up) + (size_t)(ow_ * p.up + q_ % p.up);
            const bool ok_ = (oh_ < p.Ho) && (ow_ < p.Wo);
            const __nv_bfloat16* rp = p.res_split + pix_ * p.res_cs + p.res_co + c0_;
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                rn_h[g] = make_uint4(0u, 0u, 0u, 0u); rn_l[g] = make_uint4(0u, 0u, 0u, 0u);
                if (ok_ && c0_ + g * 8 + 8 <= p.Cout) {
                    rn_h[g] = __ldg(reinterpret_cast<const uint4*>(rp + g * 8));
                    if (p.planes == 2) rn_l[g] = __ldg(reinterpret_cast<const uint4*>(rp + p.res_plane + g * 8));
                }
            }
        };
        if (RES_PF && res_pf && (int)blockIdx.x < total_tiles) res_fetch(blockIdx.x, 0);
        // TMA variant (STG == 3): residual chunk i+1 lands in staging buffer (i+1) % 3 while chunk i is processed; the epilogue
        // then adds it IN PLACE (same swizzled 16 B slots it will overwrite with the output) -- fully coalesced, no registers.
        auto res_tma_issue = [&](int tile_, int c64_, int buf_) {
            const int nt_ = tile_ % p.n_tiles, mt_ = tile_ / p.n_tiles;
            const int tw_ = mt_ % p.tiles_w; const int t2_ = mt_ / p.tiles_w;
            const int th_ = t2_ % p.tiles_h; const int img_ = t2_ / p.tiles_h;
            mbar_expect_tx(bar_res + 8 * buf_, (uint32_t)stg_bytes);
            tma_load_5d(smem_u32(stg) + buf_ * stg_bytes, &tmR, bar_res + 8 * buf_, (nt_ * BLOCK_N) % p.coutp + c64_ * 64, tw_ * p.TW, th_ * p.TH, img_, 0);
        };
        if (res_tma && warp == 2 && lane == 0 && (int)blockIdx.x < total_tiles) res_tma_issue(blockIdx.x, 0, 0);
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            const int nt = tile % p.n_tiles, mt = tile / p.n_tiles;
            const int tw_i = mt % p.tiles_w; const int t2 = mt / p.tiles_w;
            const int th_i = t2 % p.tiles_h; const int img = t2 / p.tiles_h;
            const int oh = th_i * p.TH + row / p.TW, ow = tw_i * p.TW + row % p.TW;
            const bool valid = (oh < p.Ho) && (ow < p.Wo);
            const int n_glob = nt * BLOCK_N;
            const int q = n_glob / p.coutp, ch0 = n_glob % p.coutp;   // q = sub-position of a transposed conv (0 otherwise)
            const int ui = q / p.up, uj = q % p.up;
            const size_t pix = ((size_t)img * (p.Ho * p.up) + (size_t)(oh * p.up + ui)) * (size_t)(p.Wo * p.up) + (size_t)(ow * p.up + uj);
            mbar_wait(bar_tfull + 8 * acc, acc_phase);
            tc_fence_after();
            if constexpr (STG > 0 && BLOCK_N >= 64) {
              if (p.tma_out) {
                const uint32_t stg_base = smem_u32(stg);
#pragma unroll 1
                for (int c64 = 0; c64 < BLOCK_N / 64; ++c64) {
                    const int b = stg_count % STG;
                    if (res_tma) {
                        // (A') the store that last used buffer (i+1) % STG has been read out -> request residual(i+1) into it, then wait
                        // for residual(i) in buffer b (STG == 3: a full chunk of lead; STG == 2: the lead is the chunk minus the store drain)
                        if (warp == 2 && lane == 0) {
                            bulk_wait_read<(STG >= 2 ? STG - 2 : 0)>();
                            int ntile = tile, nc = c64 + 1;
                            if (nc == BLOCK_N / 64) { nc = 0; ntile = tile + (int)gridDim.x; }
                            if (ntile < total_tiles) res_tma_issue(ntile, nc, (stg_count + 1) % STG);
                        }
                        mbar_wait(bar_res + 8 * b, (uint32_t)((stg_count / STG) & 1));
                    } else {
                        // (A) buffer b is free once at most STG-1 store groups are still reading shared memory
                        if (warp == 2 && lane == 0) bulk_wait_read<STG - 1>();
                        epi_bar(1);
                    }
                    // (B) this warp's 32 columns of the 64-column chunk -> registers -> epilogue -> swizzled smem.  Loads first (bias:
                    // warp-uniform 16 B broadcasts; residual: this thread's eight 16 B slots of the staging buffer), then the
                    // arithmetic, then the eight 16 B stores back to back.
                    uint32_t raw[32];
                    const int col0 = c64 * 64 + chalf * 32;
                    float bv[32];
#pragma unroll
                    for (int g = 0; g < 8; ++g) {
                        float4 t = p.bias ? __ldg(reinterpret_cast<const float4*>(p.bias + ch0 + col0) + g) : make_float4(0.f, 0.f, 0.f, 0.f);
                        bv[4 * g] = t.x; bv[4 * g + 1] = t.y; bv[4 * g + 2] = t.z; bv[4 * g + 3] = t.w;
                    }
                    const uint32_t srow = stg_base + b * stg_bytes + row * 128;
                    uint4 rh[4], rl[4];
#pragma unroll
                    for (int g8 = 0; g8 < 4; ++g8) { rh[g8] = make_uint4(0u, 0u, 0u, 0u); rl[g8] = make_uint4(0u, 0u, 0u, 0u); }
                    bool have_res = false;
                    if (res_tma) {
                        have_res = true;
#pragma unroll
                        for (int g8 = 0; g8 < 4; ++g8) {
                            const uint32_t chunk16 = (uint32_t)(((chalf * 4 + g8) ^ (row & 7)) * 16);      // 128B swizzle
                            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(rh[g8].x), "=r"(rh[g8].y), "=r"(rh[g8].z), "=r"(rh[g8].w) : "r"(srow + chunk16));
                            if (p.planes == 2)
                                asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(rl[g8].x), "=r"(rl[g8].y), "=r"(rl[g8].z), "=r"(rl[g8].w) : "r"(srow + A_TILE_BYTES + chunk16));
                        }
                    } else if (RES_PF && res_pf) {
                        have_res = true;        // register-prefetched one chunk ago (rn_h / rn_l)
                    }
                    const uint4* res_h = RES_PF ? rn_h : rh;
                    const uint4* res_l = RES_PF ? rn_l : rl;
                    ld_acc(col0, raw);
                    uint32_t hw[4][4], lw[4][4];
#pragma unroll
                    for (int g8 = 0; g8 < 4; ++g8) {
                        const int c = ch0 + col0 + g8 * 8;
                        float v[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(raw[g8 * 8 + j]) + bv[g8 * 8 + j];
                        if (have_res) {
                            const __nv_bfloat16* hb = reinterpret_cast<const __nv_bfloat16*>(&res_h[g8]);
                            const __nv_bfloat16* lb = reinterpret_cast<const __nv_bfloat16*>(&res_l[g8]);
#pragma unroll
                            for (int j = 0; j < 8; ++j) v[j] += __bfloat162float(hb[j]);
                            if (p.planes == 2) {
#pragma unroll
                                for (int j = 0; j < 8; ++j) v[j] += __bfloat162float(lb[j]);
                            }
                        } else if (valid && p.res_f32 && !(p.dbg & 8)) {
                            const float* rp = p.res_f32 + pix * p.res_cs + p.res_co + c;
#pragma unroll
                            for (int j = 0; j < 8; ++j) v[j] += __ldg(rp + j);
                        }
                        if constexpr (GELU) {
#pragma unroll
                            for (int j = 0; j < 8; ++j) v[j] = heal_act_fn(v[j], 2);
                        } else if (p.relu) {
#pragma unroll
                            for (int j = 0; j < 8; ++j) v[j] = fmaxf(v[j], 0.f);
                        }
                        float lo[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) lo[j] = v[j] - __bfloat162float(__float2bfloat16_rn(v[j]));
#pragma unroll
                        for (int j = 0; j < 4; ++j) { hw[g8][j] = pack_bf16(v[2 * j], v[2 * j + 1]); lw[g8][j] = pack_bf16(lo[2 * j], lo[2 * j + 1]); }
                    }
                    if (RES_PF && res_pf) {      // registers consumed: request the next chunk's residual
                        if (c64 + 1 < BLOCK_N / 64) res_fetch(tile, c64 + 1);
                        else if (tile + (int)gridDim.x < total_tiles) res_fetch(tile + gridDim.x, 0);
                    }
#pragma unroll
                    for (int g8 = 0; g8 < 4; ++g8) {
                        const uint32_t chunk16 = (uint32_t)(((chalf * 4 + g8) ^ (row & 7)) * 16);      // 128B swizzle
                        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(srow + chunk16), "r"(hw[g8][0]), "r"(hw[g8][1]), "r"(hw[g8][2]), "r"(hw[g8][3]) : "memory");
                        if (p.planes == 2)
                            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(srow + A_TILE_BYTES + chunk16), "r"(lw[g8][0]), "r"(lw[g8][1]), "r"(lw[g8][2]), "r"(lw[g8][3]) : "memory");
                    }
                    fence_async_smem();
                    epi_bar(2);
                    // (C) one thread drains the buffer with a TMA tensor store (out-of-range pixels are clipped by the unit)
                    if (warp == 2 && lane == 0 && !(p.dbg & 1)) {
                        tma_store_5d(&tmO, stg_base + b * stg_bytes, ch0 + c64 * 64, tw_i * p.TW, th_i * p.TH, img, 0);
                        bulk_commit();
                    }
                    ++stg_count;
                }
                tc_fence_before();
                mbar_arrive(bar_tempty + 8 * acc);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                continue;
              }
            }
#pragma unroll 1
            for (int cc = chalf; cc < BLOCK_N / CHUNK; cc += 2) {
                uint32_t raw[CHUNK];
                ld_acc(cc * CHUNK, raw);
                const int c_first = ch0 + cc * CHUNK;
                if (valid && c_first < p.Cout) {
#pragma unroll
                    for (int g8 = 0; g8 < CHUNK / 8; ++g8) {
                        const int c = c_first + g8 * 8;
                        if (c >= p.Cout) break;
                        float v[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(raw[g8 * 8 + j]) + ((c + j < p.Cout && p.bias) ? __ldg(p.bias + c + j) : 0.f);
                        const bool full8 = (c + 8 <= p.Cout);
                        if (p.res_split) {
                            const __nv_bfloat16* rp = p.res_split + pix * p.res_cs + p.res_co + c;
                            if (full8 && (((p.res_cs | p.res_co) & 7) == 0)) {
                                uint4 h = __ldg(reinterpret_cast<const uint4*>(rp));
                                const __nv_bfloat16* hb = reinterpret_cast<const __nv_bfloat16*>(&h);
#pragma unroll
                                for (int j = 0; j < 8; ++j) v[j] += __bfloat162float(hb[j]);
                                if (p.planes == 2) {
                                    uint4 l = __ldg(reinterpret_cast<const uint4*>(rp + p.res_plane));
                                    const __nv_bfloat16* lb = reinterpret_cast<const __nv_bfloat16*>(&l);
#pragma unroll
                                    for (int j = 0; j < 8; ++j) v[j] += __bfloat162float(lb[j]);
                                }
                            } else {
                                for (int j = 0; j < 8 && c + j < p.Cout; ++j) {
                                    v[j] += __bfloat162float(rp[j]);
                                    if (p.planes == 2) v[j] += __bfloat162float(rp[p.res_plane + j]);
                                }
                            }
                        } else if (p.res_f32) {
                            const float* rp = p.res_f32 + pix * p.res_cs + p.res_co + c;
                            for (int j = 0; j < 8 && c + j < p.Cout; ++j) v[j] += __ldg(rp + j);
                        }
                        if constexpr (GELU) {
#pragma unroll
                            for (int j = 0; j < 8; ++j) v[j] = heal_act_fn(v[j], 2);
                        } else if (p.relu) {
#pragma unroll
                            for (int j = 0; j < 8; ++j) v[j] = fmaxf(v[j], 0.f);
                        }
                        if (p.out_split && !((p.dbg & 1) && v[0] != 1.2345e30f)) {
                            __nv_bfloat16* op = p.out_split + pix * p.out_cs + p.out_co + c;
                            float lo[8];
                            uint32_t hw[4], lw[4];
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                float h = __bfloat162float(__float2bfloat16_rn(v[j]));
                                lo[j] = v[j] - h;
                            }
#pragma unroll
                            for (int j = 0; j < 4; ++j) { hw[j] = pack_bf16(v[2 * j], v[2 * j + 1]); lw[j] = pack_bf16(lo[2 * j], lo[2 * j + 1]); }
                            if (full8 && (((p.out_cs | p.out_co) & 7) == 0)) {
                                *reinterpret_cast<uint4*>(op) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
                                if (p.planes == 2) *reinterpret_cast<uint4*>(op + p.out_plane) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
                            } else {
                                for (int j = 0; j < 8 && c + j < p.Cout; ++j) {
                                    op[j] = __float2bfloat16_rn(v[j]);
                                    if (p.planes == 2) op[p.out_plane + j] = __float2bfloat16_rn(lo[j]);
                                }
                            }
                        }
                        if (p.out_f32 && !((p.dbg & 1) && v[0] != 1.2345e30f)) {
                            float* op = p.out_f32 + pix * p.out32_cs + p.out32_co + c;
                            if (full8 && (((p.out32_cs | p.out32_co) & 3) == 0)) {
                                stg_f4(op, make_float4(v[0], v[1], v[2], v[3]));
                                stg_f4(op + 4, make_float4(v[4], v[5], v[6], v[7]));
                            } else {
                                for (int j = 0; j < 8 && c + j < p.Cout; ++j) op[j] = v[j];
                            }
                        }
                    }
                }
            }
            tc_fence_before();
            mbar_arrive(bar_tempty + 8 * acc);          // 128 arrivals release this accumulator buffer
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        if (STG > 0 && warp == 2 && lane == 0) bulk_wait_all();     // all output tiles have left shared memory
        (void)stg_count;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
    }
}

// HEAL_TC_* measurement hooks (profiles/tc_experiment.py), read once per process instead of six getenv calls per launch.
struct TcEnv {
    int dbg, pdl, halo, bo, tma_store, res_tma, ring, tapn, deep, l2promo;
    TcEnv() {
        auto geti = [](const char* n, int dflt) { const char* e = getenv(n); return e ? atoi(e) : dflt; };
        dbg = geti("HEAL_TC_DBG", 0); pdl = geti("HEAL_TC_PDL", 1); halo = geti("HEAL_TC_HALO", 1); bo = geti("HEAL_TC_BO", 0);
        tma_store = geti("HEAL_TC_TMA_STORE", 1); res_tma = geti("HEAL_TC_RES_TMA", 1); ring = geti("HEAL_TC_RING", 1); tapn = geti("HEAL_TC_TAPN", 1);
        deep = geti("HEAL_TC_DEEP", 0); l2promo = geti("HEAL_TC_L2PROMO", 128);
    }
};
const TcEnv& tc_env() { static const TcEnv e; return e; }

template <int BLOCK_N, int STAGES, int STG, bool GELU = false>
int launch_tc(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmO, const CUtensorMap& tmR, const TcP& p_in, cudaStream_t st) {
    TcP p = p_in;
    p.res_tma = ((STG == 3 || (STG == 2 && BLOCK_N == 64 && STAGES == 2)) && p.tma_out && p.res_split && p_in.res_tma) ? 1 : 0;
    const size_t b_tile = p.bdiag ? (size_t)(BLOCK_N / 16) * 512 : (size_t)BLOCK_N * BLOCK_K * 2;
    size_t stage_bytes = (size_t)p.planes * A_TILE_BYTES + (size_t)p.wplanes * b_tile;
    if (p.halo) stage_bytes = (((size_t)p.planes * (p.TW + 2) * 128 + 1023) & ~(size_t)1023) + (size_t)p.wplanes * 3 * b_tile;
    size_t smem = (size_t)STAGES * stage_bytes + (size_t)STG * p.planes * A_TILE_BYTES + 256;
    if (smem > 227 * 1024) return HEAL_ERR_UNSUPPORTED;
    static size_t attr_set[HEAL_MAX_DEVICES] = {};
    if (!heal_ensure_dyn_smem(k_conv2d_tc<BLOCK_N, STAGES, STG, GELU>, 227 * 1024, attr_set)) return HEAL_ERR_LAUNCH;
    int total = p.m_tiles * p.n_tiles;
    int grid = total < HEAL_NUM_SMS ? total : HEAL_NUM_SMS;
    if (grid < 1) return HEAL_ERR_UNSUPPORTED;
    if (p.pdl) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(grid); cfg.blockDim = dim3(TC_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        cudaError_t e = cudaLaunchKernelEx(&cfg, k_conv2d_tc<BLOCK_N, STAGES, STG, GELU>, tmA, tmB, tmO, tmR, p);
        heal_launch_counter_add(1);
        return e == cudaSuccess ? HEAL_OK : HEAL_ERR_LAUNCH;
    }
    k_conv2d_tc<BLOCK_N, STAGES, STG, GELU><<<grid, TC_THREADS, smem, st>>>(tmA, tmB, tmO, tmR, p);
    return heal_check_launch();
}

}  // namespace

extern "C" int heal_conv2d_tc(const void* in_split, size_t in_plane_stride, int N, int H, int W, int Cin, int in_cstride, int in_coffset,
                              const void* w_packed, const void* w_diag, int w_rows, int coutp, const float* bias,
                              int kh, int kw, int stride, int pad, int blockdiag, int planes, int w_planes,
                              const void* res_split, size_t res_plane_stride, const float* res_f32, int res_cstride, int res_coffset,
                              void* out_split, size_t out_plane_stride, int out_cstride, int out_coffset,
                              float* out_f32, int out32_cstride, int out32_coffset,
                              int Ho, int Wo, int Cout, int upsample, int relu, void* stream_) {
    if (!in_split || !w_packed || (!out_split && !out_f32)) return HEAL_ERR_ARG;
    if (planes != 1 && planes != 2) return HEAL_ERR_ARG;
    if (w_planes != 1 && w_planes != 2) return HEAL_ERR_ARG;
    if (planes == 2 && w_planes != 2) return HEAL_ERR_UNSUPPORTED;
    if ((Cin % BLOCK_K) || (in_cstride & 7) || (in_coffset & 7) || upsample < 1) return HEAL_ERR_UNSUPPORTED;
    if (stride < 1 || stride > 2) return HEAL_ERR_UNSUPPORTED;
    if (Ho != (H + 2 * pad - kh) / stride + 1 || Wo != (W + 2 * pad - kw) / stride + 1) return HEAL_ERR_ARG;
    if (blockdiag && (upsample > 1 || coutp != Cin || (coutp % 64))) return HEAL_ERR_UNSUPPORTED;
    if (upsample > 1 && (kh != 1 || kw != 1)) return HEAL_ERR_UNSUPPORTED;
    const int taps = kh * kw;
    const int block_n = blockdiag ? 64 : (coutp >= 128 ? 128 : coutp);
    if (!(block_n == 16 || block_n == 32 || block_n == 64 || block_n == 128) || (coutp % block_n)) return HEAL_ERR_UNSUPPORTED;
    if (w_rows != (upsample > 1 ? upsample * upsample : taps) * coutp) return HEAL_ERR_ARG;
    PFN_tmEncodeTiled enc = get_encode();
    if (!enc) return HEAL_ERR_DRIVER;

    TcP p;
    p.res_tma = 0; p.bdiag = 0;
    p.N = N; p.Ho = Ho; p.Wo = Wo; p.Cout = Cout;
    p.taps_w = kw; p.taps = taps; p.pad = pad; p.kc_blocks = Cin / BLOCK_K;
    int tw = 128; while (tw > Wo && tw > 8) tw >>= 1;
    p.TW = tw; p.TH = BLOCK_M / tw;
    p.tiles_w = (Wo + p.TW - 1) / p.TW; p.tiles_h = (Ho + p.TH - 1) / p.TH;
    p.m_tiles = N * p.tiles_h * p.tiles_w;
    p.n_tiles = w_rows / taps / block_n;
    p.stride = stride; p.blockdiag = blockdiag;
    if (upsample > 1) p.n_tiles = w_rows / block_n;
    p.planes = planes; p.wplanes = w_planes; p.coutp = coutp; p.relu = relu; p.up = upsample; p.bias = bias;
    const TcEnv& env = tc_env();
    p.dbg = env.dbg; p.pdl = env.pdl;
    p.res_split = (const __nv_bfloat16*)res_split; p.res_plane = res_plane_stride; p.res_f32 = res_f32;
    p.res_cs = res_cstride; p.res_co = res_coffset;
    p.out_split = (__nv_bfloat16*)out_split; p.out_plane = out_plane_stride; p.out_cs = out_cstride; p.out_co = out_coffset;
    p.out_f32 = out_f32; p.out32_cs = out32_cstride; p.out32_co = out32_coffset;

    {
        const bool want = env.halo != 0;
        p.bo_mode = env.bo;
        p.halo = (want && kh == 3 && kw == 3 && stride == 1 && pad == 1 && p.TH == 1 && block_n == 64 && upsample == 1) ? 1 : 0;
    }
    // L2 promotion of the activation / residual loads (HEAL_TC_L2PROMO=256: experiment)
    const CUtensorMapL2promotion act_promo = env.l2promo == 256 ? CU_TENSOR_MAP_L2_PROMOTION_L2_256B : CU_TENSOR_MAP_L2_PROMOTION_L2_128B;
    CUtensorMap tmA, tmB;
    {
        cuuint64_t dims[5] = {(cuuint64_t)Cin, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N, (cuuint64_t)planes};
        cuuint64_t strides[4] = {(cuuint64_t)in_cstride * 2, (cuuint64_t)W * in_cstride * 2, (cuuint64_t)H * W * in_cstride * 2,
                                 (cuuint64_t)in_plane_stride * 2};
        cuuint32_t box[5] = {(cuuint32_t)BLOCK_K, (cuuint32_t)(p.TW * stride), (cuuint32_t)(p.TH * stride), 1u, (cuuint32_t)planes};
        if (p.halo) box[1] = (cuuint32_t)(p.TW + 2);
        cuuint32_t es[5] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1, 1};
        void* base = (void*)((const __nv_bfloat16*)in_split + in_coffset);
        if (planes == 1) { strides[3] = strides[2] * N; }
        CUresult r = enc(&tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, act_promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return HEAL_ERR_DRIVER;
    }
    {
        // packed weights in global memory: [plane][taps * coutp rows][wk] bf16.  The box order decides the shared-memory layout:
        // hi and lo planes of the same rows must be adjacent for the N-concatenated MMAs (see NCAT in the kernel).
        const cuuint64_t wk = blockdiag ? 64 : Cin;      // K extent of the packed weight matrix
        const cuuint64_t row_b = wk * 2, plane_b = (cuuint64_t)w_rows * wk * 2;
        const cuuint32_t pl = (cuuint32_t)w_planes;
        cuuint32_t es[5] = {1, 1, 1, 1, 1};
        CUresult r;
        p.bdiag = (blockdiag && w_diag) ? 1 : 0;
        if (p.bdiag) {
            // packed diagonal sub-blocks in global memory: [plane][taps * coutp rows][16] bf16 (32 B rows) -> a quarter of the bytes
            const cuuint64_t pb = (cuuint64_t)w_rows * 32;
            if (p.halo) {                   // smem [3 taps][4 sub-blocks][plane][16 rows][32 B]
                cuuint64_t d[5] = {16, 16, (cuuint64_t)w_planes, (cuuint64_t)coutp / 16, (cuuint64_t)taps};
                cuuint64_t st[4] = {32, pb, 512, (cuuint64_t)coutp * 32};
                cuuint32_t b[5] = {16u, 16u, pl, (cuuint32_t)block_n / 16, 3u};
                r = enc(&tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, (void*)w_diag, d, st, b, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            } else {                        // smem [4 sub-blocks][plane][16 rows][32 B]
                cuuint64_t d[4] = {16, 16, (cuuint64_t)w_planes, (cuuint64_t)w_rows / 16};
                cuuint64_t st[3] = {32, pb, 512};
                cuuint32_t b[4] = {16u, 16u, pl, (cuuint32_t)block_n / 16};
                r = enc(&tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void*)w_diag, d, st, b, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            }
        } else if (blockdiag && p.halo) {   // smem [3 taps][4 sub-blocks][plane][16 rows]
            cuuint64_t d[5] = {wk, 16, (cuuint64_t)w_planes, (cuuint64_t)coutp / 16, (cuuint64_t)taps};
            cuuint64_t st[4] = {row_b, plane_b, 16 * row_b, (cuuint64_t)coutp * row_b};
            cuuint32_t b[5] = {(cuuint32_t)BLOCK_K, 16u, pl, (cuuint32_t)block_n / 16, 3u};
            r = enc(&tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, (void*)w_packed, d, st, b, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        } else if (blockdiag) {             // smem [4 sub-blocks][plane][16 rows]
            cuuint64_t d[4] = {wk, 16, (cuuint64_t)w_planes, (cuuint64_t)w_rows / 16};
            cuuint64_t st[3] = {row_b, plane_b, 16 * row_b};
            cuuint32_t b[4] = {(cuuint32_t)BLOCK_K, 16u, pl, (cuuint32_t)block_n / 16};
            r = enc(&tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void*)w_packed, d, st, b, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        } else if (p.halo) {                // smem [3 taps][plane][block_n rows]: one box brings the 3 horizontal taps of a kernel row
            cuuint64_t d[4] = {wk, (cuuint64_t)coutp, (cuuint64_t)w_planes, (cuuint64_t)taps};
            cuuint64_t st[3] = {row_b, plane_b, (cuuint64_t)coutp * row_b};
            cuuint32_t b[4] = {(cuuint32_t)BLOCK_K, (cuuint32_t)block_n, pl, 3u};
            r = enc(&tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void*)w_packed, d, st, b, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        } else {                            // smem [plane][block_n rows]
            cuuint64_t d[3] = {wk, (cuuint64_t)w_rows, (cuuint64_t)w_planes};
            cuuint64_t st[2] = {row_b, plane_b};
            cuuint32_t b[3] = {(cuuint32_t)BLOCK_K, (cuuint32_t)block_n, pl};
            r = enc(&tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, (void*)w_packed, d, st, b, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        }
        if (r != CUDA_SUCCESS) return HEAL_ERR_DRIVER;
    }
    // output tensor map for the TMA-store epilogue (split / bf16 output at conv resolution, 64-channel boxes)
    CUtensorMap tmO = tmA;
    p.tma_out = 0;
    {
        const bool want = env.tma_store != 0;
        if (want && out_split && upsample == 1 && block_n >= 64 && (Cout % 64) == 0 && !(out_cstride & 7) && !(out_coffset & 7) &&
            (!res_split || (!(res_cstride & 7) && !(res_coffset & 7)))) {
            cuuint64_t dims[5] = {(cuuint64_t)Cout, (cuuint64_t)Wo, (cuuint64_t)Ho, (cuuint64_t)N, (cuuint64_t)planes};
            cuuint64_t strides[4] = {(cuuint64_t)out_cstride * 2, (cuuint64_t)Wo * out_cstride * 2, (cuuint64_t)Ho * Wo * out_cstride * 2,
                                     (cuuint64_t)out_plane_stride * 2};
            if (planes == 1) strides[3] = strides[2] * N;
            cuuint32_t box[5] = {(cuuint32_t)BLOCK_K, (cuuint32_t)p.TW, (cuuint32_t)p.TH, 1u, (cuuint32_t)planes};
            cuuint32_t es[5] = {1, 1, 1, 1, 1};
            void* base = (void*)((__nv_bfloat16*)out_split + out_coffset);
            CUresult r = enc(&tmO, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                             CU_TENSOR_MAP_SWIZZLE_128B, act_promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (r != CUDA_SUCCESS) return HEAL_ERR_DRIVER;
            p.tma_out = out_f32 ? 0 : 1;
        }
    }
    // residual tensor map (same boxes as the output map): the residual chunk is TMA-loaded into the output staging buffer
    CUtensorMap tmR = tmO;
    bool res_tma_ok = false;
    {
        const bool want = env.res_tma != 0;
        if (want && p.tma_out && res_split) {
            cuuint64_t dims[5] = {(cuuint64_t)Cout, (cuuint64_t)Wo, (cuuint64_t)Ho, (cuuint64_t)N, (cuuint64_t)planes};
            cuuint64_t strides[4] = {(cuuint64_t)res_cstride * 2, (cuuint64_t)Wo * res_cstride * 2, (cuuint64_t)Ho * Wo * res_cstride * 2,
                                     (cuuint64_t)res_plane_stride * 2};
            if (planes == 1) strides[3] = strides[2] * N;
            cuuint32_t box[5] = {(cuuint32_t)BLOCK_K, (cuuint32_t)p.TW, (cuuint32_t)p.TH, 1u, (cuuint32_t)planes};
            cuuint32_t es[5] = {1, 1, 1, 1, 1};
            void* base = (void*)((const __nv_bfloat16*)res_split + res_coffset);
            CUresult r = enc(&tmR, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                             CU_TENSOR_MAP_SWIZZLE_128B, act_promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (r != CUDA_SUCCESS) return HEAL_ERR_DRIVER;
            res_tma_ok = true;
            p.res_tma = 1;
        }
    }
    // a split residual under the TMA-store epilogue is either TMA-loaded (STG == 3) or register-prefetched (halo, <64,2,1>)
    if (p.tma_out && res_split && !res_tma_ok && !p.halo) p.tma_out = 0;
    if (p.halo && p.bdiag) p.res_tma = 0;      // <64,4,1>: register prefetch
    cudaStream_t st = (cudaStream_t)stream_;
    const int kblocks = (blockdiag ? 1 : p.kc_blocks) * taps;
    // grouped 3x3 on maps 64 or 128 pixels wide with split weights: the horizontal taps stacked along N (gconv3x3_tapn.cu), 24 MMAs
    // per 128-pixel x 64-channel unit instead of 72.  It needs its own activation box (one row, one plane, no halo) and weight box
    // (the 3 taps of a kernel row per sub-block); the output map above already has the unit's shape.
    if (env.tapn && p.bdiag && p.tma_out && !res_split && !res_f32 && kh == 3 && kw == 3 && stride == 1 && pad == 1 &&
        (Wo == 64 || Wo == 128) && relu != 2 && Cin == Cout && coutp == Cout && w_planes == 2) {
        {
            cuuint64_t dims[5] = {(cuuint64_t)Cin, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N, (cuuint64_t)planes};
            cuuint64_t strides[4] = {(cuuint64_t)in_cstride * 2, (cuuint64_t)W * in_cstride * 2, (cuuint64_t)H * W * in_cstride * 2,
                                     (cuuint64_t)in_plane_stride * 2};
            if (planes == 1) strides[3] = strides[2] * N;
            cuuint32_t box[5] = {(cuuint32_t)BLOCK_K, (cuuint32_t)W, 1u, 1u, 1u};
            cuuint32_t es[5] = {1, 1, 1, 1, 1};
            void* base = (void*)((const __nv_bfloat16*)in_split + in_coffset);
            if (enc(&tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, act_promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) return HEAL_ERR_DRIVER;
        }
        {
            // [plane][tap * C + co][16 ci]: the box {16 ci, 16 co, 3 taps, 2 planes, 4 sub-blocks} lands as [sub-block][plane][tap][co]
            cuuint64_t d[5] = {16, 16, 9, 2, (cuuint64_t)Cout / 16};
            cuuint64_t st_[4] = {32, (cuuint64_t)Cout * 32, (cuuint64_t)w_rows * 32, 512};
            cuuint32_t b[5] = {16u, 16u, 3u, 2u, 4u};
            cuuint32_t es[5] = {1, 1, 1, 1, 1};
            if (enc(&tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, (void*)w_diag, d, st_, b, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
                return HEAL_ERR_DRIVER;
        }
        RingP rp;
        rp.N = N; rp.H = Ho; rp.W = Wo; rp.C = Cout; rp.planes = planes; rp.wplanes = w_planes; rp.relu = relu; rp.bias = bias;
        rp.segs = 1; rp.seg_rows = Ho; rp.pdl = env.pdl; rp.dbg = p.dbg;
        return heal_gconv3x3_tapn_launch(tmA, tmB, tmO, rp, st);
    }
    // grouped 3x3 on maps at least 128 pixels wide: the row-ring kernel (conv3x3_ring.cu) reads every input row and the weights
    // once per CTA instead of three times / once per tile; it shares the three tensor maps built above
    if (env.ring && p.halo && p.bdiag && p.tma_out && !res_split && !res_f32 && (Wo % 128) == 0 && relu != 2 && Cin == Cout &&
        coutp == Cout && !p.dbg) {
        RingP rp;
        rp.N = N; rp.H = Ho; rp.W = Wo; rp.C = Cout; rp.planes = planes; rp.wplanes = w_planes; rp.relu = relu; rp.bias = bias;
        rp.segs = 1; rp.seg_rows = Ho; rp.pdl = env.pdl; rp.dbg = 0;
        return heal_conv3x3_ring_launch(tmA, tmB, tmO, rp, st);
    }
    if (relu == 2) {        // GELU: 1x1 / 3x3 convs with >= 128 output channels and no residual (ConvNeXt pwconv1: dim -> 4 dim)
        if (block_n != 128 || res_split || res_f32) return HEAL_ERR_UNSUPPORTED;
        if (!p.tma_out) return launch_tc<128, 3, 0, true>(tmA, tmB, tmO, tmR, p, st);
        return kblocks <= 4 ? launch_tc<128, 2, 2, true>(tmA, tmB, tmO, tmR, p, st) : launch_tc<128, 3, 1, true>(tmA, tmB, tmO, tmR, p, st);
    }
    switch (block_n) {
        case 16: return launch_tc<16, 4, 0>(tmA, tmB, tmO, tmR, p, st);
        case 32: return launch_tc<32, 4, 0>(tmA, tmB, tmO, tmR, p, st);
        case 64:
            if (p.halo && res_tma_ok && !p.bdiag) return launch_tc<64, 2, 2>(tmA, tmB, tmO, tmR, p, st);   // 81 KiB stages + 2 x 32 KiB: all of shared memory
            if (p.halo && p.bdiag && p.tma_out) return launch_tc<64, 4, 1>(tmA, tmB, tmO, tmR, p, st);     // 45 KiB stages
            if (p.halo) return p.tma_out ? launch_tc<64, 2, 1>(tmA, tmB, tmO, tmR, p, st) : launch_tc<64, 2, 0>(tmA, tmB, tmO, tmR, p, st);
            if (p.bdiag && p.tma_out && !res_tma_ok) return launch_tc<64, 4, 2>(tmA, tmB, tmO, tmR, p, st);   // 36 KiB stages
            if (res_tma_ok) return launch_tc<64, 2, 3>(tmA, tmB, tmO, tmR, p, st);
            return p.tma_out ? launch_tc<64, 3, 2>(tmA, tmB, tmO, tmR, p, st) : launch_tc<64, 4, 0>(tmA, tmB, tmO, tmR, p, st);
        default:
            if (!p.tma_out) return launch_tc<128, 3, 0>(tmA, tmB, tmO, tmR, p, st);
            if (res_tma_ok) return launch_tc<128, 2, 3>(tmA, tmB, tmO, tmR, p, st);
            // HEAL_TC_DEEP=1 (experiment): 3 stages + 1 staging buffer also for the short-K layers
            return (kblocks <= 4 && env.deep != 1) ? launch_tc<128, 2, 2>(tmA, tmB, tmO, tmR, p, st) : launch_tc<128, 3, 1>(tmA, tmB, tmO, tmR, p, st);
    }
}
