// Grouped 3x3 convolution (stride 1, pad 1, split weights) on maps 64 or 128 pixels wide, with the three horizontal taps of a
// kernel row STACKED ALONG N: one MMA per (kernel row, 16-channel sub-block) computes all three taps.
//
// Why: the row ring (conv3x3_ring.cu) issues 9 taps x 4 sub-blocks x 2 = 72 tcgen05.mma per (128 px x 64 ch) unit at N = 16 / 32,
// and a small-N MMA costs mostly the re-read of its 4 KB A slice (DESIGN §10).  The horizontal taps multiply the SAME input
// pixels; only the output pixel they land on differs.  So here A is the unit's 128 input pixels with no halo, B is the three
// taps of one kernel row stacked as N = 48 rows [s][16 co] (per weight plane), and the one-pixel shift moves to the epilogue:
//   Z_s[p] = sum_r in[row(p) + r - 1][col(p)] . w[r][s]        (TMEM, accumulated over r)
//   out[q] = Z_0[q-1] + Z_1[q] + Z_2[q+1]                     (fp32, this order; Z_0 dropped at col 0, Z_2 at col W-1)
// MMA forms per (kernel row, sub-block): a_hi x [b_hi | b_lo] at N = 96, plus a_lo x b_hi at N = 48 when the activations carry a
// lo plane: 24 MMAs per unit (tc32) or 12 (bf16) instead of 72 / 36.
//
// A unit is 128 output pixels: one row at W = 128, two consecutive rows (contiguous in NHWC) at W = 64.  A CTA owns
// (image, 64-channel block) x a range of units.  Shared memory holds
//   * a ring of input rows laid out [plane][slot][W pixels][64 channels] bf16 (one TMA box per row and plane; rows outside the
//     image are zero-filled = the vertical padding).  At W = 64 the A window of kernel row r spans two consecutive slots, so slot
//     0 is also written after the last slot and every window is contiguous;
//   * the 3 x 4 x [plane][3 taps][16 co] packed diagonal weight blocks, loaded once;
//   * one output staging tile for the TMA store and a small exchange buffer for the shift across the 32-lane quarters.
// TMEM: 4 sub-blocks x 96 columns do not double-buffer in 512 columns, so each unit is drained in two 32-channel halves, one per
// accumulator buffer: the epilogue of one half overlaps the MMAs of the other.
// Roles: warp 0 TMA producer, warp 1 MMA issuer, warps 2..9 epilogue (warp = TMEM lane quarter x 16-channel sub-block of the half).
#include <cuda.h>
#include "common.cuh"
#include "tc_prims.cuh"
#include "conv_ring.cuh"

namespace {

constexpr int TN_THREADS = 320;
constexpr int TN_M = 128;                           // output pixels per unit = MMA M
constexpr int TN_STG_PLANE = TN_M * 128;            // one plane of the output staging tile
constexpr int TN_WBLK = 2 * 48 * 32;                // one (kernel row, sub-block) weight block: [plane][3 taps][16 co][32 B]
constexpr int TN_W_BYTES = 3 * 4 * TN_WBLK;
constexpr int TN_XCH_BYTES = 2 * 2 * 4 * 32 * 4;    // [half][sub-block][quarter][Z_0 of lane 31 | Z_2 of lane 0] fp32
constexpr int TN_MAX_SLOTS = 8;
constexpr int TN_ACC_COLS = 256;                    // one accumulator buffer: 2 sub-blocks x 96 columns, 128 apart
constexpr int TN_TMEM_COLS = 512;                   // fine: shared memory already forces one CTA per SM
constexpr int TN_SMEM_LIMIT = 227 * 1024;

__host__ __device__ inline int tn_row_bytes(int W) { return W * 128; }

__global__ void __launch_bounds__(TN_THREADS, 1)
k_gconv3x3_tapn(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                const __grid_constant__ CUtensorMap tmO, const RingP p, const int slots) {
    const int R = TN_M / p.W;                           // image rows per unit
    const int CB = p.C / 64;
    const int seg = blockIdx.x % p.segs;
    const int strip = blockIdx.x / p.segs;
    const int cb = strip % CB, img = strip / CB;
    const int h_begin = seg * p.seg_rows;               // seg_rows is a multiple of R
    const int rows = min(p.seg_rows, p.H - h_begin);
    if (rows <= 0) return;
    const int units = (rows + R - 1) / R;

    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uintptr_t raw_addr = reinterpret_cast<uintptr_t>(smem_raw);
    asm volatile("" : "+l"(raw_addr));                    // keep shared-memory addresses run-time values (see conv2d_tc.cu)
    uint8_t* smem = reinterpret_cast<uint8_t*>(raw_addr);
    if (smem_u32(smem) & 1023u) __trap();
    const int row_bytes = tn_row_bytes(p.W);
    const bool dup = (R == 2);
    const int plane_bytes = (slots + (dup ? 1 : 0)) * row_bytes;
    const int stg_bytes = p.planes * TN_STG_PLANE;
    const uint32_t ring = smem_u32(smem);
    const uint32_t wbase = ring + (uint32_t)(p.planes * plane_bytes);
    const uint32_t stg = wbase + (uint32_t)TN_W_BYTES;
    float* xch = reinterpret_cast<float*>(smem + (size_t)p.planes * plane_bytes + TN_W_BYTES + stg_bytes);
    uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(xch) + TN_XCH_BYTES);
    // bars: full[8], empty[8], wfull, tfull[2], tempty[2]
    const uint32_t bar_full = smem_u32(bars), bar_empty = smem_u32(bars + TN_MAX_SLOTS), bar_w = smem_u32(bars + 2 * TN_MAX_SLOTS);
    const uint32_t bar_tfull = smem_u32(bars + 2 * TN_MAX_SLOTS + 1), bar_tempty = smem_u32(bars + 2 * TN_MAX_SLOTS + 3);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * TN_MAX_SLOTS + 6);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < TN_MAX_SLOTS; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        mbar_init(bar_w, 1);
        for (int a = 0; a < 2; ++a) { mbar_init(bar_tfull + 8 * a, 1); mbar_init(bar_tempty + 8 * a, 256); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TN_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // programmatic dependent launch: barrier init / TMEM allocation above overlapped the previous kernel's tail; nothing it
    // produced has been touched yet
    if (p.pdl) {
        asm volatile("griddepcontrol.wait;" ::: "memory");
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    }

    if (warp == 0) {
        // ============================== TMA producer ==============================
        if (elect_one()) {
            mbar_expect_tx(bar_w, (uint32_t)TN_W_BYTES);
            for (int r = 0; r < 3; ++r) tma_load_5d(wbase + r * 4 * TN_WBLK, &tmB, bar_w, 0, 0, 3 * r, 0, cb * 4);
        }
        __syncwarp();
        const int n_in = R * units + 2;                  // input rows h_begin-1 .. h_begin+R*units
        for (int j = 0; j < n_in; ++j) {
            const int slot = j % slots, use = j / slots;
            const bool copy2 = dup && slot == 0;         // slot 0 is mirrored after the last slot
            mbar_wait(bar_empty + 8 * slot, (uint32_t)((use & 1) ^ 1));
            if (elect_one()) {
                const bool ld = !(p.dbg & 4);
                mbar_expect_tx(bar_full + 8 * slot, ld ? (uint32_t)(p.planes * row_bytes * (copy2 ? 2 : 1)) : 0u);
                for (int pl = 0; pl < (ld ? p.planes : 0); ++pl) {
                    const uint32_t dst = ring + (uint32_t)(pl * plane_bytes + slot * row_bytes);
                    tma_load_5d(dst, &tmA, bar_full + 8 * slot, cb * 64, 0, h_begin - 1 + j, img, pl);
                    if (copy2) tma_load_5d(dst + (uint32_t)(slots * row_bytes), &tmA, bar_full + 8 * slot, cb * 64, 0, h_begin - 1 + j, img, pl);
                }
            }
            __syncwarp();
        }
    } else if (warp == 1) {
        // ============================== MMA issuer ================================
        const uint32_t idesc48 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(48 >> 3) << 17) | ((uint32_t)(TN_M >> 4) << 24);
        const uint32_t idesc96 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(96 >> 3) << 17) | ((uint32_t)(TN_M >> 4) << 24);
        const bool split = (p.planes == 2);
        mbar_wait(bar_w, 0);
        int waited = 0; uint32_t acc_phase = 0;
        for (int t = 0; t < units; ++t) {
            while (waited < R * t + R + 2) { mbar_wait(bar_full + 8 * (waited % slots), (uint32_t)((waited / slots) & 1)); ++waited; }
            for (int half = 0; half < 2; ++half) {
                mbar_wait(bar_tempty + 8 * half, acc_phase ^ 1);
                tc_fence_after();
                if (elect_one()) {
                    if (!(p.dbg & 16))
#pragma unroll
                    for (int r = 0; r < 3; ++r) {
                        // window of kernel row r: input rows R*t + r .. R*t + r + R - 1 (ring-relative), contiguous in the ring
                        const uint32_t ah = ring + (uint32_t)(((R * t + r) % slots) * row_bytes), al = ah + (uint32_t)plane_bytes;
#pragma unroll
                        for (int kk = 0; kk < 2; ++kk) {
                            const int k = half * 2 + kk;
                            const uint64_t bd = umma_desc_sw32(wbase + (uint32_t)((r * 4 + k) * TN_WBLK));
                            const uint32_t td = tmem_base + (uint32_t)(half * TN_ACC_COLS + kk * 128);
                            umma_bf16(td, umma_desc_sw128(ah + k * 32), bd, idesc96, r > 0 ? 1u : 0u);    // [a_hi*b_hi | a_hi*b_lo]
                            if (split) umma_bf16(td, umma_desc_sw128(al + k * 32), bd, idesc48, 1u);     // += a_lo*b_hi
                        }
                    }
                    if (half == 1)                       // input rows R*t .. R*t+R-1 are not needed by any later unit
                        for (int i = 0; i < R; ++i) umma_commit(bar_empty + 8 * ((R * t + i) % slots));
                    umma_commit(bar_tfull + 8 * half);
                }
                __syncwarp();
            }
            acc_phase ^= 1;
        }
    } else {
        // ============================== epilogue (warps 2..9) =====================
        const int quarter = warp & 3;                   // TMEM lane quarter this warp may access
        const int sub = (warp - 2) >> 2;                // which 16-channel sub-block of the half this warp drains
        const int px = quarter * 32 + lane;             // pixel within the unit
        const int col = px % p.W;
        const bool has_l = col != 0, has_r = col != p.W - 1;
        const uint32_t srow = stg + (uint32_t)(px * 128);
        float bv[2][16];
#pragma unroll
        for (int half = 0; half < 2; ++half)
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                float4 b4 = p.bias ? __ldg(reinterpret_cast<const float4*>(p.bias + cb * 64 + (half * 2 + sub) * 16) + g) : make_float4(0.f, 0.f, 0.f, 0.f);
                bv[half][4 * g] = b4.x; bv[half][4 * g + 1] = b4.y; bv[half][4 * g + 2] = b4.z; bv[half][4 * g + 3] = b4.w;
            }
        uint32_t acc_phase = 0;
        for (int t = 0; t < units; ++t) {
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                mbar_wait(bar_tfull + 8 * half, acc_phase);
                tc_fence_after();
                if (p.dbg & 1) { tc_fence_before(); mbar_arrive(bar_tempty + 8 * half); continue; }
                // columns of this sub-block: [Z_0 Z_1 Z_2 (hi weights) | Z_0 Z_1 Z_2 (lo weights)], 16 each
                const uint32_t tb = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(half * TN_ACC_COLS + sub * 128);
                float z0[16], z1[16], z2[16];
                {
                    uint32_t a[32], b[16], c[16], d[32];
                    tmem_ld32(tb, a); tmem_ld16(tb + 32, b); tmem_ld16(tb + 48, c); tmem_ld32(tb + 64, d);
                    tmem_wait_ld();
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        z0[j] = __uint_as_float(a[j]) + __uint_as_float(c[j]);
                        z1[j] = __uint_as_float(a[16 + j]) + __uint_as_float(d[j]);
                        z2[j] = __uint_as_float(b[j]) + __uint_as_float(d[16 + j]);
                    }
                }
                // accumulator consumed: hand the buffer back before the shift and the stores
                tc_fence_before();
                mbar_arrive(bar_tempty + 8 * half);
                // the 32-lane quarter boundaries: publish Z_0 of lane 31 and Z_2 of lane 0 to the neighbouring warps
                float* xq = xch + ((half * 2 + sub) * 4 + quarter) * 32;
                if (lane == 31) {
#pragma unroll
                    for (int c = 0; c < 16; c += 4) *reinterpret_cast<float4*>(xq + c) = make_float4(z0[c], z0[c + 1], z0[c + 2], z0[c + 3]);
                }
                if (lane == 0) {
#pragma unroll
                    for (int c = 0; c < 16; c += 4) *reinterpret_cast<float4*>(xq + 16 + c) = make_float4(z2[c], z2[c + 1], z2[c + 2], z2[c + 3]);
                }
                // the previous unit's TMA store has finished reading the staging tile
                if (half == 0 && warp == 2 && lane == 0) bulk_wait_read<0>();
                epi_bar(1);
                float zl[16], zr[16];
#pragma unroll
                for (int c = 0; c < 16; ++c) {
                    zl[c] = __shfl_up_sync(0xffffffffu, z0[c], 1);
                    zr[c] = __shfl_down_sync(0xffffffffu, z2[c], 1);
                }
                if (lane == 0 && quarter > 0) {
#pragma unroll
                    for (int c = 0; c < 16; ++c) zl[c] = xq[-32 + c];
                }
                if (lane == 31 && quarter < 3) {
#pragma unroll
                    for (int c = 0; c < 16; ++c) zr[c] = xq[32 + 16 + c];
                }
                uint32_t hw[8], lw[8];
#pragma unroll
                for (int c = 0; c < 16; c += 2) {
                    float v[2], lo[2];
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        v[j] = (has_l ? zl[c + j] : 0.f) + z1[c + j];
                        v[j] = v[j] + (has_r ? zr[c + j] : 0.f);
                        v[j] += bv[half][c + j];
                        if (p.relu) v[j] = fmaxf(v[j], 0.f);
                        lo[j] = v[j] - __bfloat162float(__float2bfloat16_rn(v[j]));
                    }
                    hw[c / 2] = pack_bf16(v[0], v[1]); lw[c / 2] = pack_bf16(lo[0], lo[1]);
                }
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const uint32_t chunk16 = (uint32_t)((((half * 2 + sub) * 2 + i) ^ (px & 7)) * 16);      // 128B swizzle
                    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(srow + chunk16), "r"(hw[4 * i]), "r"(hw[4 * i + 1]), "r"(hw[4 * i + 2]), "r"(hw[4 * i + 3]) : "memory");
                    if (p.planes == 2)
                        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(srow + TN_STG_PLANE + chunk16), "r"(lw[4 * i]), "r"(lw[4 * i + 1]), "r"(lw[4 * i + 2]), "r"(lw[4 * i + 3]) : "memory");
                }
            }
            fence_async_smem();
            epi_bar(2);
            if (warp == 2 && lane == 0 && !(p.dbg & 1)) {                // rows below the image (odd H at W = 64) are clipped by the TMA unit
                tma_store_5d(&tmO, stg, cb * 64, 0, h_begin + R * t, img, 0);
                bulk_commit();
            }
            acc_phase ^= 1;
        }
        if (warp == 2 && lane == 0) bulk_wait_all();     // the last tile has left shared memory
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TN_TMEM_COLS) : "memory");
    }
}

}  // namespace

int heal_gconv3x3_tapn_launch(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmO, RingP p, cudaStream_t st) {
    if ((p.W != 64 && p.W != 128) || (p.C % 64) || p.wplanes != 2 || p.N < 1 || p.H < 1) return HEAL_ERR_UNSUPPORTED;
    const int R = TN_M / p.W;
    const int row_bytes = tn_row_bytes(p.W), stg_bytes = p.planes * TN_STG_PLANE;
    const int fixed = TN_W_BYTES + stg_bytes + TN_XCH_BYTES + 256;
    int slots = (TN_SMEM_LIMIT - fixed) / (p.planes * row_bytes) - (R == 2 ? 1 : 0);
    if (slots > TN_MAX_SLOTS) slots = TN_MAX_SLOTS;
    if (slots < R + 3) return HEAL_ERR_UNSUPPORTED;
    const size_t smem = (size_t)p.planes * (slots + (R == 2 ? 1 : 0)) * row_bytes + fixed;
    // strips x segments of units: one wave of CTAs when the strips alone do not fill the SMs
    const int strips = p.N * (p.C / 64);
    const int units = (p.H + R - 1) / R;
    int segs = strips >= HEAL_NUM_SMS ? 1 : HEAL_NUM_SMS / strips;
    if (segs > units / 4) segs = units / 4 > 0 ? units / 4 : 1;
    const int seg_units = (units + segs - 1) / segs;
    p.seg_rows = seg_units * R;
    p.segs = (units + seg_units - 1) / seg_units;
    static size_t attr_set[HEAL_MAX_DEVICES] = {};
    if (!heal_ensure_dyn_smem(k_gconv3x3_tapn, TN_SMEM_LIMIT, attr_set)) return HEAL_ERR_LAUNCH;
    if (p.pdl) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(strips * p.segs); cfg.blockDim = dim3(TN_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        cudaError_t e = cudaLaunchKernelEx(&cfg, k_gconv3x3_tapn, tmA, tmB, tmO, p, slots);
        heal_launch_counter_add(1);
        return e == cudaSuccess ? HEAL_OK : HEAL_ERR_LAUNCH;
    }
    k_gconv3x3_tapn<<<strips * p.segs, TN_THREADS, smem, st>>>(tmA, tmB, tmO, p, slots);
    return heal_check_launch();
}
