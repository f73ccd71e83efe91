// Tensor-core super-resolution path for sm_100a: the modulated 3x3 convolutions of SuperresolutionHybrid8XDC (197.6 GFLOP/frame,
// SURVEY.md §8d) and the plain convolutions of the torso head as TMA-fed tcgen05 implicit GEMMs.
//
//   activations  NHWC fp16, channels padded to a multiple of 64 (one 128-byte swizzle row = 64 channels)
//   weights      per-sample folded (modulated+demodulated) fp16, packed [n][tap][Cout][Cin_pad]  (K-major B operand)
//   accumulate   fp32 in TMEM; epilogue in fp32 (bias, lrelu*sqrt2, ToRGB + skip) then fp16 / fp32 stores
//
// The conv kernel (conv_tc3_kernel): persistent CTA PAIRS (cta_group::2): M256 x N128 x K16 MMAs, half weight tile per CTA, A row strips
// reused by the horizontal taps through row-shifted descriptors, double-buffered TMEM accumulators, 8 epilogue warps.  (Its two
// predecessors - one tile per CTA, and the same persistent design on single CTAs - were removed in round 2; see git history.)
// The im2col is done by TMA itself: every (tap, 64-channel chunk) of the K loop is a box load at the tap's shifted
// coordinates, zero-filled outside the image (= the conv's zero padding); one elected lane issues the MMAs.
//
// The stride-2 transposed convolution of the up layers (conv2d_resample.py:116-133) keeps the reference's operation order for large Cin:
// four output-parity phases (4/2/2/1 taps) as units of ONE launch -> (2H+1)x(2W+1) fp16 result -> fir_tma_kernel (TMA-staged 4x4 FIR +
// bias + lrelu) + upconv_edge_kernel (last column).  For small Cin (block0.conv0) the FIR is composed into the weights instead.
#include "common.cuh"
#include "tc_prims.cuh"
#include <mutex>
#include <vector>
#include <type_traits>
#include <stdlib.h>

#ifndef R3DP_TC_DEBUG_TIMING
#define R3DP_TC_DEBUG_TIMING 0
#endif
namespace r3dp {
namespace tc {

constexpr int BM = 128, BN = 128, BK = 64, UMMA_K = 16;
constexpr float kSplitWeightScale = 1024.0f;       // split-fp16 weights are stored x 2^10: their lo halves (|w| 2^-11) stay normal fp16 numbers

// kind::f16 instruction descriptor: D=f32 (bit 4), A=B=f16 (0), both K-major, N>>3 at [17,23), M>>4 at [24,29)
constexpr uint32_t kIdesc = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

struct Taps {
    int n;
    int dy[9], dx[9], widx[9];
};
enum Mode { kStoreAct = 0, kStoreRaw = 1, kToRgbFinal = 2 };
struct ConvArgs {
    Taps taps;
    int k_chunks;            // Cin_pad / 64
    int tiles_x, rows;       // grid of M tiles: rows x tiles_x (each tile = 128 consecutive grid columns of one row)
    int w_shared;            // 1: all samples use weight set 0
    int mode;
    // output (fp16 NHWC) for kStoreAct / kStoreRaw: pixel (row*oy_mul+oy_off, col*ox_mul+ox_off) of an out_H x out_W x out_C image
    __half* out; int out_H, out_W, out_C, oy_mul, oy_off, ox_mul, ox_off;
    const float* bias;       // [Cout] conv bias (kStoreAct, kToRgbFinal)
    // kToRgbFinal: img_out[n][3][out_H][out_W] = upsample2d(img_prev[n][3][out_H/2][out_W/2]) + torgb(act) + brgb
    const float* wrgb;       // [Nw][3][128] folded ToRGB weights (fp32)
    const float* brgb;       // [3]
    const float* img_prev;
    float* img_out;
    int out_clamp; uint8_t* img_out_u8;
    int split;               // fp32-grade [hi | lo] operands (see Conv2Args)
};

// =====================================================================================================================
// Persistent implicit-GEMM conv design (shared by conv_tc3_kernel<R>): R output rows (R x 128 pixels) x 128 couts per tile.
//
// Why: ncu on the first one-tile-per-CTA kernel showed 58 % tensor-pipe activity on the largest layer, L2 at 65 % / 92 % hits: not L2-bound, but
// with 128x128 tiles the two smem operands cost 128 B/clk of shared-memory reads per MMA, the same port TMA fills.  This design cuts the
// fill traffic and the per-tile overheads:
//   * an input ROW STRIP {64 ch, 130 px} is loaded once per 64-channel chunk and serves all horizontal taps (the UMMA smem
//     descriptor starts 128 B x shift later; the 128-byte swizzle is a function of the ABSOLUTE smem address, so the descriptor's
//     base_offset stays 0 - verified on B200) and the R output rows that touch it vertically;
//   * every weight tile {64 ch, 128 couts} of a tap is used by R MMA groups before it is released;
//   * persistent CTAs, accumulators double-buffered in TMEM (R x 128 columns x 2), so the epilogue of tile i overlaps tile i+1;
//   * the four output-parity phases of a transposed conv are units of ONE launch;
//   * a unit = (image, phase, row group, x block); the CTA loops over the cout blocks of its unit so that ToRGB partial sums of a
//     256-channel layer stay in registers (block0's ToRGB is fused like the last layer's).
// Two mbarrier rings (A strips, B taps) are filled by one TMA lane in exactly the order the MMA lane consumes them.
// =====================================================================================================================
constexpr int A2_ROWS = 130, A2_BYTES = A2_ROWS * 128, A2_SLOT = 17408;       // 17 x 1024: every slot keeps the swizzle alignment
struct Taps2 {
    int n, ngroups;                 // taps sorted by (dy, dx); group = taps sharing dy
    int dyi[9], shift[9], widx[9];  // group index, horizontal shift (dx + 1, in pixels: strips start at x0 - 1), weight tap index
    int gstart[4];                  // first tap of each group (+ sentinel)
    int dy_min;
};
struct Phase2 {
    Taps2 taps;
    int rows, oy_off, ox_off;       // valid grid rows of this phase; output pixel = (row*oy_mul + oy_off, col*ox_mul + ox_off)
};
enum Mode2 { kActRgb = 3 };         // kStoreAct + ToRGB/skip accumulated over the cout blocks (in addition to Mode)
struct Conv2Args {
    Phase2 ph[4];
    int n_phases, k_chunks, tiles_x, row_groups, n_blocks, n_images, total_units;
    int w_shared, mode;
    __half* out; int out_H, out_W, out_C, oy_mul, ox_mul;
    const float* bias; const float* wrgb; const float* brgb; const float* img_prev; float* img_out; int img_H, img_W;
    float act_slope, act_gain;      // epilogue activation: v < 0 ? v*slope : v, then * gain  (0.2, sqrt2 = bias_act lrelu; 0.01, 1 = nn.LeakyReLU; 1, 1 = linear)
    int skip_same_res;              // ToRGB skip image has the output resolution (SynthesisBlockNoUp) instead of half (FIR-upsampled)
    const __half* residual;         // non-null: added to the activated output before the store (ResBlock2d of large_sr)
    int out_clamp;                  // final image clamped to [-1, 1] (the caller-side imgs.clamp(-1,1), inference/real3d_infer.py:515)
    uint8_t* img_out_u8;            // non-null: final image as uint8 HWC frames [N][H][W][3] = int((clamp(x)+1)/2*255) (real3d_infer.py:519) instead of fp32 NCHW
    int split;                      // fp32-grade operands: activations [hi | lo] (2 x Cin_pad channels), weights [hi | lo]; K loop = hi*hi + lo*hi + hi*lo
    int lo_off;                     // split: channel offset of the lo half in the OUTPUT tensor (= logical output channels); out_C is the physical pixel stride
    int phase_mix;                  // interleave the phases of a multi-phase launch over the units (see decode)
    float acc_scale;                // accumulator scale applied before the bias (split weights are stored x 2^10 so their lo halves stay normal fp16)
    unsigned long long* debug;      // R3DP_TC_DEBUG_TIMING builds: [acc wait, strip wait, tap wait, issue, total, #CTAs] clock sums of the MMA warp
};


// FIR-upsampled skip image (upsample2d, upfirdn2d.py:317-354) at output pixel (Y,X): zero-insert x2, pad (2,1,2,1), [1,3,3,1]^2/64 * 4
__device__ __forceinline__ float upsampled_skip(const float* __restrict__ ip, int h, int w, int Y, int X) {
    const float k4[4] = {0.25f, 0.75f, 0.75f, 0.25f};
    float acc = 0.f;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int zy = Y + u - 2;
        if (zy < 0 || (zy & 1) || (zy >> 1) >= h) continue;
        float rowv = 0.f;
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            const int zx = X + v - 2;
            if (zx < 0 || (zx & 1) || (zx >> 1) >= w) continue;
            rowv = fmaf(k4[v], __ldg(ip + (size_t)(zy >> 1) * w + (zx >> 1)), rowv);
        }
        acc = fmaf(k4[u], rowv, acc);
    }
    return acc;
}

// the same sum as upsampled_skip without branches: the two rows / columns of the half-resolution image that reach (Y, X) are (Y-1)>>1
// and its successor with weights (.25,.75) for even Y and (.75,.25) for odd Y; out-of-range taps get weight 0 and a clamped address, so
// the four loads are independent (one L2 round trip) and the fma order - hence the bits - are those of the loop above.
__device__ __forceinline__ float upsampled_skip_bf(const float* __restrict__ ip, int h, int w, int Y, int X) {
    const int y0 = (Y - 1) >> 1, x0 = (X - 1) >> 1;
    const float ky0 = (y0 >= 0 && y0 < h) ? ((Y & 1) ? 0.75f : 0.25f) : 0.f, ky1 = (y0 + 1 < h) ? ((Y & 1) ? 0.25f : 0.75f) : 0.f;
    const float kx0 = (x0 >= 0 && x0 < w) ? ((X & 1) ? 0.75f : 0.25f) : 0.f, kx1 = (x0 + 1 < w) ? ((X & 1) ? 0.25f : 0.75f) : 0.f;
    const int ya = min(max(y0, 0), h - 1), yb = min(y0 + 1, h - 1), xa = min(max(x0, 0), w - 1), xb = min(x0 + 1, w - 1);
    const float v00 = __ldg(ip + (size_t)ya * w + xa), v01 = __ldg(ip + (size_t)ya * w + xb);
    const float v10 = __ldg(ip + (size_t)yb * w + xa), v11 = __ldg(ip + (size_t)yb * w + xb);
    const float r0 = fmaf(kx1, v01, fmaf(kx0, v00, 0.f)), r1 = fmaf(kx1, v11, fmaf(kx0, v10, 0.f));
    return fmaf(ky1, r1, fmaf(ky0, r0, 0.f));
}

// packed 2 x fp32 arithmetic (sm_100 f32x2): one issue slot for two lanes of the epilogue's bias / lrelu / ToRGB work
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rc;\n\t"
        "mov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
        "fma.rn.f32x2 rc, ra, rb, rc;\n\t"
        "mov.b64 {%0, %1}, rc;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
    return d;
}
__device__ __forceinline__ float2 mul2(float2 a, float2 b) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rc;\n\t"
        "mov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
        "mul.rn.f32x2 rc, ra, rb;\n\t"
        "mov.b64 {%0, %1}, rc;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
}
__device__ __forceinline__ float2 add2(float2 a, float2 b) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rc;\n\t"
        "mov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
        "add.rn.f32x2 rc, ra, rb;\n\t"
        "mov.b64 {%0, %1}, rc;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
}

__device__ __forceinline__ uint4 pack_half8(const float* f) {
    __half2 h0 = __floats2half2_rn(f[0], f[1]), h1 = __floats2half2_rn(f[2], f[3]);
    __half2 h2 = __floats2half2_rn(f[4], f[5]), h3 = __floats2half2_rn(f[6], f[7]);
    uint4 pk;
    pk.x = *reinterpret_cast<uint32_t*>(&h0); pk.y = *reinterpret_cast<uint32_t*>(&h1);
    pk.z = *reinterpret_cast<uint32_t*>(&h2); pk.w = *reinterpret_cast<uint32_t*>(&h3);
    return pk;
}

__device__ __forceinline__ void store_half32(__half* dst, const float* f) {
    uint4* d4 = reinterpret_cast<uint4*>(dst);
#pragma unroll
    for (int v = 0; v < 4; ++v) {
        __half2 h0 = __floats2half2_rn(f[8 * v + 0], f[8 * v + 1]), h1 = __floats2half2_rn(f[8 * v + 2], f[8 * v + 3]);
        __half2 h2 = __floats2half2_rn(f[8 * v + 4], f[8 * v + 5]), h3 = __floats2half2_rn(f[8 * v + 6], f[8 * v + 7]);
        uint4 pk;
        pk.x = *reinterpret_cast<uint32_t*>(&h0); pk.y = *reinterpret_cast<uint32_t*>(&h1);
        pk.z = *reinterpret_cast<uint32_t*>(&h2); pk.w = *reinterpret_cast<uint32_t*>(&h3);
        d4[v] = pk;
    }
}

// =====================================================================================================================
// conv_tc3_kernel<R>: the v2 kernel on CTA PAIRS (thread-block cluster of 2 = one TPC, tcgen05 cta_group::2).
// ncu on v1/v2: with 128x128 single-CTA tiles every MMA pulls 4 KB (A) + 4 KB (B) from shared memory per 64 clk = 128 B/clk, the
// whole smem port, which TMA also needs for the fills -> tensor pipe stuck at ~58 %.  A pair computes M = 256 pixels (each CTA's
// own 128-pixel strips) x N = 128 couts per instruction and each CTA keeps only HALF of the weight tile (64 couts): 6 KB per 64 clk
// per SM.  Protocol: both CTAs run the same producer/epilogue loops on neighbouring units; all "full" barriers live in the leader
// (rank 0) and receive the TMA bytes of both CTAs (cp.async.bulk.tensor.cta_group::2, peer bit cleared in the barrier address);
// the leader's MMA lane issues tcgen05.mma.cta_group::2 and releases ring slots / publishes accumulators in BOTH CTAs with
// multicast tcgen05.commit; the epilogue warps of both CTAs arrive on the leader's accumulator-empty barrier.
// =====================================================================================================================
constexpr int kThreads3 = 64 + 256;                                          // TMA warp, MMA warp, 8 epilogue warps
constexpr int B3_BYTES = (BN / 2) * BK * 2;                                  // 64 couts x 64 ch fp16 = 8 KB per CTA
constexpr uint32_t kIdesc3 = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);    // M = 256 across the pair
template <int R> struct Cfg3 {
    static constexpr int NA = (R > 2) ? 7 : 8, NB = 8;   // R = 4 gives up one strip slot so the staging buffer fits in 227 KB
    static constexpr int NACC = (R * BN * 2 <= 512) ? 2 : 1;
    static constexpr int TMEM_COLS = (R * BN * NACC <= 128) ? 128 : (R * BN * NACC <= 256 ? 256 : 512);
    static constexpr int TAIL = (R > 2 ? 12288 : 8192);                      // barriers, bias, ToRGB weights, [R][128][3] partial sums
    static constexpr int STAGE = 8 * 32 * 64;                                // fp16 store staging: 8 epilogue warps x 32 px x 64 B
    static constexpr int SMEM = NA * A2_SLOT + NB * B3_BYTES + 1024 + TAIL + STAGE;
};
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_load_4d_2sm(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tc_commit_2sm(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void tc_mma_f16_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}

template <int R, bool SPLIT>
__global__ void __launch_bounds__(kThreads3, 1) conv_tc3_kernel(const __grid_constant__ CUtensorMap tmA,
                                                               const __grid_constant__ CUtensorMap tmB, const Conv2Args a) {
    using C = Cfg3<R>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = align_smem_1024(smem_raw);
    uint8_t* a_ring = smem;
    uint8_t* b_ring = smem + C::NA * A2_SLOT;
    uint8_t* tail = b_ring + C::NB * B3_BYTES;
    uint64_t* a_full = reinterpret_cast<uint64_t*>(tail);
    uint64_t* a_empty = a_full + C::NA;
    uint64_t* b_full = a_empty + C::NA;
    uint64_t* b_empty = b_full + C::NB;
    uint64_t* acc_full = b_empty + C::NB;
    uint64_t* acc_empty = acc_full + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
    float* s_bias = reinterpret_cast<float*>(tail + 512);                    // [256]
    float* s_wrgb = s_bias + 256;                                            // [3][n_blocks*128]
    float* s_part = s_wrgb + 768;                                            // [R][128][3] ToRGB partial sums of the second column group
    uint4* s_stage = reinterpret_cast<uint4*>(tail + C::TAIL);               // [8 warps][32 px][4 x 16 B] fp16 store staging (XOR-swizzled)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t cta_rank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(cta_rank));
    const bool leader = cta_rank == 0;
    const int units_per_image = a.n_phases * a.row_groups * a.tiles_x;

    if (warp == 0 && lane == 0) {
        for (int i = 0; i < C::NA; ++i) { mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 1); }
        for (int i = 0; i < C::NB; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 16); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(C::TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    if (warp >= 2) {
        const int t = threadIdx.x - 64;
        for (int e = t; e < a.n_blocks * BN && e < 256; e += 256) s_bias[e] = a.bias ? a.bias[e] : 0.f;
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // unit index -> (image n, phase, row group, x block); x fastest so neighbouring CTAs share strips in L2
    // Multi-phase launches with an even number of x blocks (the 4/2/2/1-tap phases of a transposed conv at W = 256): phases are interleaved,
    // slot = rg * n_phases + p' with ph = (p' + rg) mod n_phases, so that at any moment the CTA pairs are spread over all phases (the 1- and
    // 2-tap phases need 60-80 B/clk/SM of operands, above the L2 share of an SM, the 4-tap phase 40) and every pair sees every phase.
    const bool mix = a.phase_mix && a.n_phases > 1 && (a.tiles_x & 1) == 0;
    auto decode = [&](int unit, int& n, int& ph, int& row0, int& col0) {
        n = unit / units_per_image; int r = unit - n * units_per_image;
        const int xb = r % a.tiles_x; r /= a.tiles_x;
        int rg;
        if (mix) { rg = r / a.n_phases; ph = (r - rg * a.n_phases + rg) % a.n_phases; }
        else { rg = r % a.row_groups; ph = r / a.row_groups; }
        row0 = rg * R; col0 = xb * BM;
    };

    if (warp == 0) {
        // ===== TMA producer (one lane): strips and taps in consumption order =====
        if (lane == 0) {
            uint32_t aq = 0, bq = 0;                                         // running strip / tap sequence numbers
            for (int unit = (blockIdx.x & ~1) + (int)cta_rank; unit < a.total_units; unit += gridDim.x) {
                int n, ph, row0, col0; decode(unit, n, ph, row0, col0);
                const Taps2& tp = a.ph[ph].taps;
                const int DY = tp.ngroups;
                const int wn = a.w_shared ? 0 : n;
                const int K3 = SPLIT ? 3 * a.k_chunks : a.k_chunks;               // split: [x_hi w_hi | x_lo w_hi | x_hi w_lo] over the channel chunks
                for (int nblk = 0; nblk < a.n_blocks; ++nblk)
                    for (int kq = 0; kq < K3; ++kq) {
                        const int kc = kq < 2 * a.k_chunks ? kq : kq - 2 * a.k_chunks;    // activation chunk: hi, lo (at k_chunks + c), hi again
                        const int kb = kq < a.k_chunks ? kq : kq - a.k_chunks;            // weight chunk: hi, hi, lo (at k_chunks + c)
                        for (int d = 0; d < DY; ++d) {
                            const int s_lo = d == 0 ? 0 : R - 1 + d, s_hi = R - 1 + d;
                            for (int s = s_lo; s <= s_hi; ++s, ++aq) {
                                const int slot = aq % C::NA;
                                mbar_wait(&a_empty[slot], ((aq / C::NA) & 1) ^ 1);
                                if (leader) mbar_expect_tx(&a_full[slot], 2 * A2_BYTES);
                                tma_load_4d_2sm(a_ring + slot * A2_SLOT, &tmA, &a_full[slot], kc * BK, col0 - 1, row0 + tp.dy_min + s, n);
                            }
                            for (int t = tp.gstart[d]; t < tp.gstart[d + 1]; ++t, ++bq) {
                                const int slot = bq % C::NB;
                                mbar_wait(&b_empty[slot], ((bq / C::NB) & 1) ^ 1);
                                if (leader) mbar_expect_tx(&b_full[slot], 2 * B3_BYTES);
                                tma_load_4d_2sm(b_ring + slot * B3_BYTES, &tmB, &b_full[slot], kb * BK, nblk * BN + (int)cta_rank * (BN / 2), tp.widx[t], wn);
                            }
                        }
                    }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: the leader CTA issues for the pair (M = 256: rows 0-127 from CTA0's strips, 128-255 from CTA1's) =====
        if (leader) {
        uint32_t aq = 0, bq = 0, it = 0;
#if R3DP_TC_DEBUG_TIMING
        long long t_acc = 0, t_a = 0, t_b = 0, t_issue = 0, t_tot0 = clock64(), tt; unsigned long long ns0, ns1; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns0));
#define DT_BEGIN() tt = clock64()
#define DT_END(x) x += clock64() - tt
#else
#define DT_BEGIN()
#define DT_END(x)
#endif
        for (int unit = (blockIdx.x & ~1) + (int)cta_rank; unit < a.total_units; unit += gridDim.x) {
            int n, ph, row0, col0; decode(unit, n, ph, row0, col0);
            const Taps2& tp = a.ph[ph].taps;
            const int DY = tp.ngroups, NS = R + DY - 1;
            for (int nblk = 0; nblk < a.n_blocks; ++nblk, ++it) {
                const int buf = it % C::NACC;
                DT_BEGIN();
                mbar_wait(&acc_empty[buf], (((it / C::NACC) & 1) ^ 1));
                tc_fence_after();
                DT_END(t_acc);
                const uint32_t acc0 = tmem_base + buf * (R * BN);
                const int K3 = SPLIT ? 3 * a.k_chunks : a.k_chunks;
                for (int kc = 0; kc < K3; ++kc) {
                    const uint32_t a_base = aq;                               // sequence number of strip 0 of this chunk
                    for (int d = 0; d < DY; ++d) {
                        const int s_lo = d == 0 ? 0 : R - 1 + d, s_hi = R - 1 + d;
                        DT_BEGIN();
                        for (int s = s_lo; s <= s_hi; ++s, ++aq) mbar_wait(&a_full[aq % C::NA], (aq / C::NA) & 1);
                        DT_END(t_a);
                        for (int t = tp.gstart[d]; t < tp.gstart[d + 1]; ++t, ++bq) {
                            const int bslot = bq % C::NB;
                            DT_BEGIN();
                            mbar_wait(&b_full[bslot], (bq / C::NB) & 1);
                            tc_fence_after();
                            DT_END(t_b);
                            DT_BEGIN();
                            {
                                const uint64_t db = umma_desc_sw128(smem_u32(b_ring + bslot * B3_BYTES));
                                const int sh = tp.shift[t];
                                const uint32_t first = (uint32_t)(kc | t);
                                uint64_t da[R];
#pragma unroll
                                for (int j = 0; j < R; ++j) da[j] = umma_desc_sw128(smem_u32(a_ring + ((a_base + j + d) % C::NA) * A2_SLOT) + 128 * sh);
                                if (elect_one()) {
                                    // k-step outer, row inner: consecutive MMAs accumulate into DIFFERENT TMEM tiles
#pragma unroll
                                    for (int k = 0; k < BK / UMMA_K; ++k) {
#pragma unroll
                                        for (int j = 0; j < R; ++j)
                                            tc_mma_f16_2sm(acc0 + j * BN, da[j] + (uint64_t)(2 * k), db + (uint64_t)(2 * k), kIdesc3, first | (uint32_t)k);
                                    }
                                    tc_commit_2sm(&b_empty[bslot]);
                                }
                            }
                            __syncwarp();
                            DT_END(t_issue);
                        }
                        // strips no later group needs: strip d after group d; everything left after the last group
                        if (d < DY - 1) {
                            if (elect_one()) tc_commit_2sm(&a_empty[(a_base + d) % C::NA]);
                        } else {
                            for (int s = DY - 1; s < NS; ++s) { if (elect_one()) tc_commit_2sm(&a_empty[(a_base + s) % C::NA]); }
                        }
                        __syncwarp();
                    }
                }
                if (elect_one()) tc_commit_2sm(&acc_full[buf]);
                __syncwarp();
            }
        }
#if R3DP_TC_DEBUG_TIMING
        if (lane == 0 && a.debug) {
            atomicAdd((unsigned long long*)a.debug + 0, (unsigned long long)t_acc); atomicAdd((unsigned long long*)a.debug + 1, (unsigned long long)t_a);
            atomicAdd((unsigned long long*)a.debug + 2, (unsigned long long)t_b); atomicAdd((unsigned long long*)a.debug + 3, (unsigned long long)t_issue);
            atomicAdd((unsigned long long*)a.debug + 4, (unsigned long long)(clock64() - t_tot0)); atomicAdd((unsigned long long*)a.debug + 5, 1ull);
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns1)); atomicAdd((unsigned long long*)a.debug + 6, ns1 - ns0); atomicAdd((unsigned long long*)a.debug + 7, (unsigned long long)it);
        }
#endif
        }
    } else {
        // ===== epilogue: warps 2..9; warp w reads TMEM lanes [32*(w%4), +32); warps 2-5 take columns 0-63 of each accumulator, 6-9 columns 64-127 =====
        const int q = warp & 3, m = q * 32 + lane;
        const int cg = (warp - 2) >> 2;                                       // column group
        const bool want_rgb = (a.mode == kToRgbFinal) || (a.mode == kActRgb);
        const int CW = a.n_blocks * BN;                                      // channels ToRGB sums over
        float brgb[3] = {0.f, 0.f, 0.f};
        if (want_rgb) { brgb[0] = a.brgb[0]; brgb[1] = a.brgb[1]; brgb[2] = a.brgb[2]; }
        uint32_t it = 0;
        int n_loaded = -1;
#if R3DP_TC_DEBUG_TIMING
        long long e_full = 0, e_ld = 0, e_math = 0, e_xchg = 0, e_fin = 0, e_pre = 0, e_tot0 = clock64(), et;
#define ET_BEGIN() et = clock64()
#define ET_END(x) x += clock64() - et
#else
#define ET_BEGIN()
#define ET_END(x)
#endif
        for (int unit = (blockIdx.x & ~1) + (int)cta_rank; unit < a.total_units; unit += gridDim.x) {
            int n, ph, row0, col0; decode(unit, n, ph, row0, col0);
            const Phase2& P = a.ph[ph];
            const int wn = a.w_shared ? 0 : n;
            if (want_rgb && wn != n_loaded) {
                asm volatile("bar.sync 1, 256;" ::: "memory");               // all eight epilogue warps are done with the old weights
                for (int e = threadIdx.x - 64; e < 3 * CW; e += 256) s_wrgb[e] = a.wrgb[(size_t)wn * 3 * CW + e];
                asm volatile("bar.sync 1, 256;" ::: "memory");
                n_loaded = wn;
            }
            const int gcol = col0 + m, X = gcol * a.ox_mul + P.ox_off;
            float2 rgb2[R][3];                                               // ToRGB sums, even / odd channels in the two halves
#pragma unroll
            for (int j = 0; j < R; ++j) { rgb2[j][0] = make_float2(0.f, 0.f); rgb2[j][1] = make_float2(0.f, 0.f); rgb2[j][2] = make_float2(0.f, 0.f); }
            ET_BEGIN();
            // skip-image taps of this thread's pixels, fetched by the SECOND column group (it idles at the exchange barrier anyway) and
            // added to its partial sums.  Issued before the accumulator wait, all loads in one basic block (clamped addresses, zero
            // weights outside the image), so their L2 latency overlaps and hides behind the MMAs.
            float skipv[R][3];
#pragma unroll
            for (int j = 0; j < R; ++j) { skipv[j][0] = 0.f; skipv[j][1] = 0.f; skipv[j][2] = 0.f; }
            if (want_rgb && cg == 1 && a.img_prev) {
                if (a.skip_same_res) {
                    const int Xc = min(X, a.img_W - 1);
#pragma unroll
                    for (int j = 0; j < R; ++j) {
                        const int Yc = min((row0 + j) * a.oy_mul + P.oy_off, a.img_H - 1);
#pragma unroll
                        for (int c = 0; c < 3; ++c) skipv[j][c] = __ldg(a.img_prev + (((size_t)n * 3 + c) * a.img_H + Yc) * a.img_W + Xc);
                    }
                } else {
                    const int h = a.img_H / 2, w = a.img_W / 2;
                    const int x0 = (X - 1) >> 1;
                    const float kx0 = (x0 >= 0 && x0 < w) ? ((X & 1) ? 0.75f : 0.25f) : 0.f, kx1 = (x0 + 1 < w) ? ((X & 1) ? 0.25f : 0.75f) : 0.f;
                    const int xa = min(max(x0, 0), w - 1), xb = min(max(x0 + 1, 0), w - 1);
                    float v[R][3][4], ky0[R], ky1[R];
#pragma unroll
                    for (int j = 0; j < R; ++j) {
                        const int Y = (row0 + j) * a.oy_mul + P.oy_off, y0 = (Y - 1) >> 1;
                        ky0[j] = (y0 >= 0 && y0 < h) ? ((Y & 1) ? 0.75f : 0.25f) : 0.f;
                        ky1[j] = (y0 + 1 < h) ? ((Y & 1) ? 0.25f : 0.75f) : 0.f;
                        const int ya = min(max(y0, 0), h - 1), yb = min(max(y0 + 1, 0), h - 1);
#pragma unroll
                        for (int c = 0; c < 3; ++c) {
                            const float* ip = a.img_prev + ((size_t)n * 3 + c) * h * w;
                            v[j][c][0] = __ldg(ip + ya * w + xa); v[j][c][1] = __ldg(ip + ya * w + xb);
                            v[j][c][2] = __ldg(ip + yb * w + xa); v[j][c][3] = __ldg(ip + yb * w + xb);
                        }
                    }
#pragma unroll
                    for (int j = 0; j < R; ++j)
#pragma unroll
                        for (int c = 0; c < 3; ++c) {                        // the fma order of upsampled_skip
                            const float r0 = fmaf(kx1, v[j][c][1], fmaf(kx0, v[j][c][0], 0.f)), r1 = fmaf(kx1, v[j][c][3], fmaf(kx0, v[j][c][2], 0.f));
                            skipv[j][c] = fmaf(ky1[j], r1, fmaf(ky0[j], r0, 0.f));
                        }
                }
            }
            ET_END(e_pre);
            for (int nblk = 0; nblk < a.n_blocks; ++nblk, ++it) {
                const int buf = it % C::NACC;
                ET_BEGIN();
                mbar_wait(&acc_full[buf], (it / C::NACC) & 1);
                tc_fence_after();
                ET_END(e_full);
#pragma unroll
                for (int j = 0; j < R; ++j) {
                    const int row = row0 + j;
                    const int Y = row * a.oy_mul + P.oy_off;
                    const bool row_ok = (row < P.rows) && (Y < a.out_H);
                    const bool in_img = row_ok && (X < a.out_W);
                    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + buf * (R * BN) + j * BN;
#pragma unroll 1
                    for (int c0 = cg * (BN / 2); c0 < (cg + 1) * (BN / 2); c0 += 32) {
                        uint32_t r[32];
                        ET_BEGIN();
                        tc_ld32(taddr + c0, r);
                        ET_END(e_ld);
                        ET_BEGIN();
                        float2 f2[16];
                        const float2 sc2 = make_float2(a.acc_scale, a.acc_scale);
                        if (a.mode == kStoreRaw) {
#pragma unroll
                            for (int i = 0; i < 16; ++i) {
                                f2[i] = make_float2(__uint_as_float(r[2 * i]), __uint_as_float(r[2 * i + 1]));
                                if (SPLIT) f2[i] = mul2(f2[i], sc2);
                            }
                        } else {
                            // bias, leaky relu as max(v, v*slope) (slope <= 1), gain: bias_act lrelu*sqrt2 | nn.LeakyReLU | linear
                            const float2* b2 = reinterpret_cast<const float2*>(s_bias + nblk * BN + c0);
                            const float2 sl2 = make_float2(a.act_slope, a.act_slope), g2 = make_float2(a.act_gain, a.act_gain);
#pragma unroll
                            for (int i = 0; i < 16; ++i) {
                                const float2 acc2 = make_float2(__uint_as_float(r[2 * i]), __uint_as_float(r[2 * i + 1]));
                                const float2 v = SPLIT ? fma2(acc2, sc2, b2[i]) : add2(acc2, b2[i]);
                                const float2 t = mul2(v, sl2);
                                f2[i] = mul2(make_float2(fmaxf(v.x, t.x), fmaxf(v.y, t.y)), g2);
                            }
                        }
                        const float* f = reinterpret_cast<const float*>(f2);
                        if (a.mode != kToRgbFinal) {
                            // NHWC fp16 store through smem: the thread owns a pixel (32 channels = 64 B); written directly, every
                            // STG.128 of the warp would touch 32 different lines.  Staged, 4 lanes write one pixel's 64 contiguous bytes.
                            // Split mode: a second pass stores the fp16 remainders (v - fp16(v)) lo_off channels further.
                            uint4* st = s_stage + (warp - 2) * 128;
                            const int sw = (lane >> 1) & 3;
                            constexpr int passes = SPLIT ? 2 : 1;
#pragma unroll
                            for (int pass = 0; pass < passes; ++pass) {
                                if (pass == 0) {
#pragma unroll
                                    for (int v = 0; v < 4; ++v) st[lane * 4 + (v ^ sw)] = pack_half8(f + 8 * v);
                                } else {
#pragma unroll
                                    for (int v = 0; v < 4; ++v) {
                                        float lo[8];
#pragma unroll
                                        for (int e = 0; e < 8; ++e) lo[e] = f[8 * v + e] - __half2float(__float2half_rn(f[8 * v + e]));
                                        st[lane * 4 + (v ^ sw)] = pack_half8(lo);
                                    }
                                }
                                __syncwarp();
#pragma unroll
                                for (int i = 0; i < 4; ++i) {
                                    const int p = i * 8 + (lane >> 2), cch = lane & 3;
                                    uint4 pk = st[p * 4 + (cch ^ ((p >> 1) & 3))];
                                    const int Xp = (col0 + q * 32 + p) * a.ox_mul + P.ox_off;
                                    if (row_ok && Xp < a.out_W) {
                                        const size_t eo = ((size_t)n * a.out_H + Y) * a.out_W * a.out_C + nblk * BN + (size_t)Xp * a.out_C + c0 + cch * 8 + pass * a.lo_off;
                                        if (a.residual) {          // ResBlock2d: out = act(conv) + x (superresolution.py:283-288), same NHWC fp16 layout as the output
                                            const uint4 rv = __ldg(reinterpret_cast<const uint4*>(a.residual + eo));
                                            __half2* ph = reinterpret_cast<__half2*>(&pk); const __half2* rh = reinterpret_cast<const __half2*>(&rv);
#pragma unroll
                                            for (int e = 0; e < 4; ++e) { const float2 x = __half22float2(ph[e]), r = __half22float2(rh[e]); ph[e] = __floats2half2_rn(x.x + r.x, x.y + r.y); }
                                        }
                                        *reinterpret_cast<uint4*>(a.out + eo) = pk;
                                    }
                                }
                                __syncwarp();
                            }
                        }
                        if (want_rgb) {
#pragma unroll
                            for (int c = 0; c < 3; ++c) {
                                const float4* w4 = reinterpret_cast<const float4*>(s_wrgb + c * CW + nblk * BN + c0);
                                float2 acc = rgb2[j][c];
#pragma unroll
                                for (int j4 = 0; j4 < 8; ++j4) {
                                    const float4 w = w4[j4];
                                    acc = fma2(f2[2 * j4], make_float2(w.x, w.y), acc);
                                    acc = fma2(f2[2 * j4 + 1], make_float2(w.z, w.w), acc);
                                }
                                rgb2[j][c] = acc;
                            }
                        }
                        ET_END(e_math);
                    }
                    ET_BEGIN();
                    if (want_rgb && nblk == a.n_blocks - 1) {
                        // the two column groups hold partial ToRGB sums of the same pixel: group 1 hands its sums to group 0 through smem
                        if (cg == 1) {
#pragma unroll
                            for (int c = 0; c < 3; ++c) s_part[(j * BM + m) * 3 + c] = (rgb2[j][c].x + rgb2[j][c].y) + skipv[j][c];
                        }
                        asm volatile("bar.sync 2, 256;" ::: "memory");
                        if (cg == 0) {
#pragma unroll
                            for (int c = 0; c < 3; ++c) rgb2[j][c].x = (rgb2[j][c].x + rgb2[j][c].y) + s_part[(j * BM + m) * 3 + c];
                        }
                        asm volatile("bar.sync 3, 256;" ::: "memory");
                    }
                    ET_END(e_xchg);
                    ET_BEGIN();
                    if (want_rgb && nblk == a.n_blocks - 1 && in_img && cg == 0) {
#pragma unroll
                        for (int c = 0; c < 3; ++c) {
                            float v = rgb2[j][c].x + brgb[c];
                            if (a.out_clamp) v = fminf(fmaxf(v, -1.0f), 1.0f);
                            if (a.img_out_u8)          // torch: ((x + 1) / 2 * 255.).int() -> uint8, every step rounded in fp32, truncation
                                a.img_out_u8[(((size_t)n * a.img_H + Y) * a.img_W + X) * 3 + c] =
                                    (uint8_t)(int)__fmul_rn(__fmul_rn(__fadd_rn(v, 1.0f), 0.5f), 255.0f);
                            else
                                a.img_out[(((size_t)n * 3 + c) * a.img_H + Y) * a.img_W + X] = v;
                        }
                    }
                    ET_END(e_fin);
                }
                // this warp is done reading the accumulator buffer
                tc_fence_before();
                __syncwarp();
                if (lane == 0) asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(&acc_empty[buf]) & 0xFEFFFFFFu) : "memory");
            }
        }
#if R3DP_TC_DEBUG_TIMING
        if (lane == 0 && a.debug && (warp == 2 || warp == 6) && cta_rank == 0) {
            unsigned long long* d = a.debug + 8 + (warp == 6 ? 8 : 0);
            atomicAdd(d + 0, (unsigned long long)e_full); atomicAdd(d + 1, (unsigned long long)e_ld); atomicAdd(d + 2, (unsigned long long)e_math);
            atomicAdd(d + 3, (unsigned long long)e_xchg); atomicAdd(d + 4, (unsigned long long)e_fin); atomicAdd(d + 5, (unsigned long long)(clock64() - e_tot0));
            atomicAdd(d + 6, (unsigned long long)it); atomicAdd(d + 7, (unsigned long long)e_pre);
        }
#endif
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                     // the peer's smem/TMEM must stay alive until every MMA that reads it has retired
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(C::TMEM_COLS) : "memory");
    }
}

// ---- helpers around the GEMMs ---------------------------------------------------------------------------------------
// fp16 pair of a fp32 value: hi = fp16(v), lo = fp16(v - hi)  (v = hi + lo to ~2^-22 |v| while lo is a normal fp16 number)
__device__ __forceinline__ void split_half(float v, __half& hi, __half& lo) {
    hi = __float2half_rn(v);
    lo = __float2half_rn(v - __half2float(hi));
}

// wf fp32 [Nw][O][I][3][3] -> packed fp16 [Nw][9][O][Ip]  (zero for i >= I); split: [Nw][9][O][2*Ip] = [hi | lo] of wf * 2^10
__global__ void pack_weights_kernel(const float* __restrict__ wf, int Nw, int O, int I, int Ip, int split, __half* __restrict__ out) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)Nw * 9 * O * Ip;
    if (idx >= total) return;
    const int i = (int)(idx % Ip); const int o = (int)((idx / Ip) % O); const int t = (int)((idx / ((long long)Ip * O)) % 9);
    const int nw = (int)(idx / ((long long)Ip * O * 9));
    const float v = i < I ? wf[(((size_t)nw * O + o) * I + i) * 9 + t] : 0.f;
    if (!split) { out[idx] = __float2half_rn(v); return; }
    __half hi, lo;
    split_half(v * kSplitWeightScale, hi, lo);
    const size_t row = (idx / Ip) * (size_t)(2 * Ip);
    out[row + i] = hi; out[row + Ip + i] = lo;
}

// bilinear up-resize (or copy when size == h) of NCHW fp32 -> NHWC fp16 with channel padding to Cp
__global__ void resize_to_nhwc_f16_kernel(const float* __restrict__ x, int N, int C, int h, int w, int size, int Cp, int split, __half* __restrict__ y) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)N * size * size * Cp) return;
    const int c = (int)(idx % Cp); const int ox = (int)((idx / Cp) % size); const int oy = (int)((idx / ((long long)Cp * size)) % size);
    const int n = (int)(idx / ((long long)Cp * size * size));
    float v = 0.f;
    if (c < C) {
        const float sy = fmaxf(((float)oy + 0.5f) * ((float)h / (float)size) - 0.5f, 0.f);
        const float sx = fmaxf(((float)ox + 0.5f) * ((float)w / (float)size) - 0.5f, 0.f);
        const int y0 = min((int)sy, h - 1), x0 = min((int)sx, w - 1), y1 = min(y0 + 1, h - 1), x1 = min(x0 + 1, w - 1);
        const float ty = sy - (float)y0, tx = sx - (float)x0;
        const float* p = x + ((size_t)n * C + c) * h * w;
        const float r0 = p[y0 * w + x0] * (1.f - ty) + p[y1 * w + x0] * ty;
        const float r1 = p[y0 * w + x1] * (1.f - ty) + p[y1 * w + x1] * ty;
        v = r0 * (1.f - tx) + r1 * tx;
    }
    if (!split) { y[idx] = __float2half_rn(v); return; }
    __half hi, lo;
    split_half(v, hi, lo);
    const size_t pix = (idx / Cp) * (size_t)(2 * Cp);
    y[pix + c] = hi; y[pix + Cp + c] = lo;
}

// last column X = 2W of the transposed-conv result (the only part of the (2H+1)x(2W+1) grid the 128-wide GEMM tiles do not
// cover): yb[n][Y][2W][co] = sum_{ci, ky == Y (mod 2)} x[(Y-ky)/2][W-1][ci] * w[ky*3+2][co][ci].
// CTA = 32 couts x 16 rows of one image.  The kx = 2 column of the kernel for these couts ([3][32][Cp] fp16) and the <= 10 input
// pixels are staged in smem; thread (co, row pair) then runs plain dot products - no cross-lane reductions.  Cp <= 256.
constexpr int kEdgeRows = 16, kEdgeRowsSplit = 16, kEdgeCo = 32;      // (64 rows per CTA - the weight column staged 9 instead of 33 times per image - measured slower: 28.3 vs 25.3 us, 144 CTAs are too few)
__global__ void __launch_bounds__(256) upconv_edge_kernel(const __half* __restrict__ x, const __half* __restrict__ wp, int H, int W, int Cp, int O,
                                                          int w_shared, __half* __restrict__ yb) {
    extern __shared__ __align__(16) uint8_t edge_smem[];
    __half* s_x = reinterpret_cast<__half*>(edge_smem);                      // [10][Cp]
    __half* s_w = s_x + (kEdgeRows / 2 + 2) * Cp;                            // [3][32][Cp + 8]   (+8 halfs: rows land in different banks)
    const int WS = Cp + 8;
    const int n = blockIdx.z, Y0 = blockIdx.x * kEdgeRows, co0 = blockIdx.y * kEdgeCo;
    const int BH = 2 * H + 1, BW = 2 * W + 1;
    const int wn = w_shared ? 0 : n;
    const int iy0 = Y0 / 2 - 1;                                              // first input row any of these Y can touch
    const int vec = Cp / 8;
    for (int e = threadIdx.x; e < (kEdgeRows / 2 + 2) * vec; e += 256) {
        const int r = e / vec, c8 = e - r * vec, iy = iy0 + r;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (iy >= 0 && iy < H) v = __ldg(reinterpret_cast<const uint4*>(x + (((size_t)n * H + iy) * W + (W - 1)) * Cp) + c8);
        *reinterpret_cast<uint4*>(s_x + r * Cp + c8 * 8) = v;
    }
    for (int e = threadIdx.x; e < 3 * kEdgeCo * vec; e += 256) {
        const int c8 = e % vec, co = (e / vec) % kEdgeCo, ky = e / (vec * kEdgeCo);
        uint4 v = make_uint4(0, 0, 0, 0);
        if (co0 + co < O) v = __ldg(reinterpret_cast<const uint4*>(wp + (((size_t)wn * 9 + ky * 3 + 2) * O + co0 + co) * Cp) + c8);
        *reinterpret_cast<uint4*>(s_w + (ky * kEdgeCo + co) * WS + c8 * 8) = v;
    }
    __syncthreads();
    const int co = threadIdx.x & 31, yp = threadIdx.x >> 5;                  // 8 warps x 2 rows each; lanes = couts
    if (co0 + co >= O) return;
    constexpr int RPW = kEdgeRows / 8;                                        // rows per warp
#pragma unroll 2
    for (int hh = 0; hh < RPW; ++hh) {
        const int yy = yp * RPW + hh, Y = Y0 + yy;
        if (Y >= BH) continue;
        float acc = 0.f;
        for (int ky = (yy & 1); ky < 3; ky += 2) {                           // Y0 is even: parity of Y == parity of yy
            const int r = ((yy - ky) >> 1) + 1;                              // == (Y-ky)/2 - iy0 ; rows outside the image hold zeros
            const uint4* xr = reinterpret_cast<const uint4*>(s_x + r * Cp);
            const uint4* wr = reinterpret_cast<const uint4*>(s_w + (ky * kEdgeCo + co) * WS);
            for (int c8 = 0; c8 < vec; ++c8) {
                const uint4 xv = xr[c8], wv = wr[c8];
                const __half2* xh = reinterpret_cast<const __half2*>(&xv);
                const __half2* wh = reinterpret_cast<const __half2*>(&wv);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float2 a = __half22float2(xh[j]), b = __half22float2(wh[j]);
                    acc = fmaf(a.x, b.x, acc); acc = fmaf(a.y, b.y, acc);
                }
            }
        }
        yb[(((size_t)n * BH + Y) * BW + 2 * W) * O + co0 + co] = __float2half_rn(acc);
    }
}

// FIR 4x4 (pad 1, gain 4) + bias + lrelu*sqrt2 on the transposed-conv result: yb [N][2H+1][2W+1][C] fp16 -> y [N][2H][2W][C] fp16.
// HBM-bound stencil (read 1x + write 1x), done the Blackwell way: a persistent CTA streams {64 ch, 35 px, 11 rows} boxes of yb
// into shared memory with ONE TMA instruction each (double-buffered on mbarriers; the box is zero-filled outside the image,
// which IS the FIR's zero padding), then 256 threads (32 px x 8 channel-vectors) march down the tile: 4 swizzled LDS.128 per
// input row -> horizontal taps -> 4-row register window -> vertical taps, bias, lrelu -> one 16-byte store per output row.
constexpr int FIR_TW = 32, FIR_TH = 8, FIR_SEG = 32, FIR_BW = FIR_TW + 3, FIR_BH = FIR_TH + 3;
constexpr int FIR_BOX8_BYTES = FIR_BW * FIR_TH * 128;
constexpr int FIR_BOX_BYTES = FIR_BW * FIR_BH * 128, FIR_SLOT = (FIR_BOX_BYTES + 1023) / 1024 * 1024;
constexpr int FIR_SMEM = 2 * FIR_SLOT + 1024 + 64;
// packed 2 x fp32 FMA (sm_100 fma.rn.f32x2): (d0,d1) += (a0,a1) * (b0,b1)
__device__ __forceinline__ void ffma2(float& d0, float& d1, float a0, float a1, float b0, float b1) {
    asm("{\n\t.reg .b64 ra, rb, rc;\n\t"
        "mov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%0, %1};\n\t"
        "fma.rn.f32x2 rc, ra, rb, rc;\n\t"
        "mov.b64 {%0, %1}, rc;\n\t}"
        : "+f"(d0), "+f"(d1) : "f"(a0), "f"(a1), "f"(b0), "f"(b1));
}
// Work item = a strip of FIR_TW px x FIR_SEG output rows of one 64-channel group, streamed as FIR_SEG / FIR_TH chunks: the first box has the
// 3 halo rows (35 px x 11 rows), the following boxes only new rows (35 x 8) - the 4-row register window simply keeps rolling across the
// chunks, so only 35 input rows are loaded and converted per 32 output rows (ncu on the one-box-per-tile form: 386 MB read for 270 MB of
// input, the vertical halo rows came from DRAM twice).  A two-output-pixels-per-thread variant (2.5 LDS.128 and 20 converts per output vector
// instead of 4 and 32) was measured at 122-124 us against 124.5-126 us and dropped: the pass is not bound by instruction issue alone.
template <bool SPLIT>
__global__ void __launch_bounds__(256) fir_tma_kernel(const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmY8,
                                                      const float* __restrict__ bias, int N, int OH, int OW, int C, __half* __restrict__ y) {
    // SPLIT: yb and y hold [hi | lo] fp16 halves of C channels each (fp32-grade path): both halves of a tile are loaded, summed in fp32,
    // filtered, and the result is split again
    constexpr int NSL = SPLIT ? 2 : 1;
    constexpr int NCH = FIR_SEG / FIR_TH;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = align_smem_1024(smem_raw);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + 2 * NSL * FIR_SLOT);
    const int tid = threadIdx.x, px = tid >> 3, c8 = tid & 7;
    const int tiles_x = OW / FIR_TW, segs = (OH + FIR_SEG - 1) / FIR_SEG, cgs = C / 64;
    const int total = N * cgs * segs * tiles_x;
    const int my_items = (int)blockIdx.x < total ? (total - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    const int nseq = my_items * NCH;
    const int CS = SPLIT ? 2 * C : C;                                      // physical channels per pixel
    if (tid == 0) {
        mbar_init(&full[0], 1); mbar_init(&full[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmY) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmY8) : "memory");
    }
    __syncthreads();
    auto item_of = [&](int s, int& tx, int& sg, int& cg, int& n) {
        int r = blockIdx.x + (s / NCH) * gridDim.x;
        tx = r % tiles_x; r /= tiles_x;
        sg = r % segs; r /= segs;
        cg = r % cgs; n = r / cgs;
    };
    auto issue = [&](int s, int buf) {
        int tx, sg, cg, n; item_of(s, tx, sg, cg, n);
        const int c = s % NCH;
        const int y0 = sg * FIR_SEG - 1 + (c == 0 ? 0 : FIR_BH + FIR_TH * (c - 1));
        const CUtensorMap* map = c == 0 ? &tmY : &tmY8;
        mbar_expect_tx(&full[buf], NSL * (c == 0 ? FIR_BOX_BYTES : FIR_BOX8_BYTES));
        tma_load_4d(smem + buf * NSL * FIR_SLOT, map, &full[buf], cg * 64, tx * FIR_TW - 1, y0, n);
        if (SPLIT) tma_load_4d(smem + (buf * NSL + 1) * FIR_SLOT, map, &full[buf], C + cg * 64, tx * FIR_TW - 1, y0, n);
    };
    if (tid == 0) {
        if (nseq > 0) issue(0, 0);
        if (nseq > 1) issue(1, 1);
    }
    const float k4[4] = {0.25f, 0.75f, 0.75f, 0.25f};
    float win[4][8];
    float b[8];
    for (int s = 0; s < nseq; ++s) {
        const int buf = s & 1, c = s % NCH;
        int tx, sg, cg, n; item_of(s, tx, sg, cg, n);
        if (c == 0) {
#pragma unroll
            for (int j = 0; j < 8; ++j) b[j] = bias[cg * 64 + c8 * 8 + j];
#pragma unroll
            for (int rr = 0; rr < 4; ++rr)
#pragma unroll
                for (int j = 0; j < 8; ++j) win[rr][j] = 0.f;
        }
        mbar_wait(&full[buf], (s >> 1) & 1);
        const uint8_t* sb = smem + buf * NSL * FIR_SLOT;
        const int ox = tx * FIR_TW + px;
        const int gy0 = c == 0 ? 0 : FIR_BH + FIR_TH * (c - 1);            // index of this box's first row inside the item's 35 input rows
        auto rows = [&](auto nrows_tag) {
            constexpr int NROWS = decltype(nrows_tag)::value;
#pragma unroll
            for (int ry = 0; ry < NROWS; ++ry) {
#pragma unroll
                for (int j = 0; j < 8; ++j) { win[0][j] = win[1][j]; win[1][j] = win[2][j]; win[2][j] = win[3][j]; win[3][j] = 0.f; }
#pragma unroll
                for (int v = 0; v < 4; ++v) {
                    const int row = ry * FIR_BW + px + v;                        // 128-byte row of the box; swizzle = chunk ^ (row & 7)
                    const uint4 raw = *reinterpret_cast<const uint4*>(sb + row * 128 + ((c8 ^ (row & 7)) << 4));
                    const __half2* h = reinterpret_cast<const __half2*>(&raw);
                    uint4 rawl = make_uint4(0, 0, 0, 0);
                    if (SPLIT) rawl = *reinterpret_cast<const uint4*>(sb + FIR_SLOT + row * 128 + ((c8 ^ (row & 7)) << 4));
                    const __half2* hl = reinterpret_cast<const __half2*>(&rawl);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        float2 f = __half22float2(h[j]);
                        if (SPLIT) { const float2 g = __half22float2(hl[j]); f.x += g.x; f.y += g.y; }
                        ffma2(win[3][2 * j], win[3][2 * j + 1], k4[v], k4[v], f.x, f.y);  // packed f32x2: the kernel is issue-bound
                    }
                }
                const int gy = gy0 + ry;
                if (gy >= 3) {
                    const int oy = sg * FIR_SEG + gy - 3;
                    if (oy < OH) {
                        uint4 pk; __half2* ph = reinterpret_cast<__half2*>(&pk);
                        uint4 pl; __half2* pq = reinterpret_cast<__half2*>(&pl);
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            float a0 = b[2 * j], a1 = b[2 * j + 1];
#pragma unroll
                            for (int u = 0; u < 4; ++u) ffma2(a0, a1, k4[u], k4[u], win[u][2 * j], win[u][2 * j + 1]);
                            a0 = (a0 < 0.f ? a0 * 0.2f : a0) * 1.4142135623730951f; a1 = (a1 < 0.f ? a1 * 0.2f : a1) * 1.4142135623730951f;
                            ph[j] = __floats2half2_rn(a0, a1);
                            if (SPLIT) { const float2 hf = __half22float2(ph[j]); pq[j] = __floats2half2_rn(a0 - hf.x, a1 - hf.y); }
                        }
                        __half* dst = y + (((size_t)n * OH + oy) * OW + ox) * CS + cg * 64 + c8 * 8;
                        *reinterpret_cast<uint4*>(dst) = pk;
                        if (SPLIT) *reinterpret_cast<uint4*>(dst + C) = pl;
                    }
                }
            }
        };
        if (c == 0) rows(std::integral_constant<int, FIR_BH>{}); else rows(std::integral_constant<int, FIR_TH>{});
        __syncthreads();                                                      // everyone is done reading this buffer
        if (tid == 0 && s + 2 < nseq) issue(s + 2, buf);
    }
}

// split-operand version of upconv_edge_kernel (fp32-grade path): x [N][H][W][2*Cp] and the packed weights [..][2*Cp] hold [hi | lo] halves, the
// weights x 2^10; both are summed to fp32 while they are staged, the dot products run in fp32, the result is written as [hi | lo] of O channels.
__global__ void __launch_bounds__(256) upconv_edge_split_kernel(const __half* __restrict__ x, const __half* __restrict__ wp, int H, int W, int Cp, int O,
                                                                int w_shared, __half* __restrict__ yb) {
    extern __shared__ __align__(16) uint8_t edge_smem[];
    float* s_x = reinterpret_cast<float*>(edge_smem);                        // [10][Cp]
    float* s_w = s_x + (kEdgeRowsSplit / 2 + 2) * Cp;                             // [3][32][Cp + 4]
    const int WS = Cp + 4;
    const int n = blockIdx.z, Y0 = blockIdx.x * kEdgeRowsSplit, co0 = blockIdx.y * kEdgeCo;
    const int BH = 2 * H + 1, BW = 2 * W + 1;
    const int wn = w_shared ? 0 : n;
    const int iy0 = Y0 / 2 - 1;
    for (int e = threadIdx.x; e < (kEdgeRowsSplit / 2 + 2) * Cp; e += 256) {
        const int r = e / Cp, c = e - r * Cp, iy = iy0 + r;
        float v = 0.f;
        if (iy >= 0 && iy < H) { const __half* px = x + (((size_t)n * H + iy) * W + (W - 1)) * 2 * Cp; v = __half2float(px[c]) + __half2float(px[Cp + c]); }
        s_x[r * Cp + c] = v;
    }
    for (int e = threadIdx.x; e < 3 * kEdgeCo * Cp; e += 256) {
        const int c = e % Cp, co = (e / Cp) % kEdgeCo, ky = e / (Cp * kEdgeCo);
        float v = 0.f;
        if (co0 + co < O) { const __half* pw = wp + (((size_t)wn * 9 + ky * 3 + 2) * O + co0 + co) * 2 * Cp; v = __half2float(pw[c]) + __half2float(pw[Cp + c]); }
        s_w[(ky * kEdgeCo + co) * WS + c] = v;
    }
    __syncthreads();
    const int co = threadIdx.x & 31, yp = threadIdx.x >> 5;
    if (co0 + co >= O) return;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int yy = yp * 2 + half, Y = Y0 + yy;
        if (Y >= BH) continue;
        float acc = 0.f;
        for (int ky = (yy & 1); ky < 3; ky += 2) {
            const int r = ((yy - ky) >> 1) + 1;
            const float4* xr = reinterpret_cast<const float4*>(s_x + r * Cp);
            const float4* wr = reinterpret_cast<const float4*>(s_w + (ky * kEdgeCo + co) * WS);
            for (int c4 = 0; c4 < Cp / 4; ++c4) {
                const float4 a = xr[c4], b = wr[c4];
                acc = fmaf(a.x, b.x, acc); acc = fmaf(a.y, b.y, acc); acc = fmaf(a.z, b.z, acc); acc = fmaf(a.w, b.w, acc);
            }
        }
        acc *= 1.0f / kSplitWeightScale;
        __half hi, lo;
        split_half(acc, hi, lo);
        __half* dst = yb + (((size_t)n * BH + Y) * BW + 2 * W) * 2 * O + co0 + co;
        dst[0] = hi; dst[O] = lo;
    }
}

// ToRGB for the first block: x NHWC fp16 [N][H][W][C] -> img_out NCHW fp32 = upsample2d(img_prev) + conv1x1 + bias.  One warp per
// 32 consecutive pixels is wasteful on loads, so: one thread per pixel, 16-byte channel vectors, weights in smem.
__global__ void __launch_bounds__(256) torgb_f16_kernel(const __half* __restrict__ x, const float* __restrict__ wrgb, const float* __restrict__ brgb,
                                                        const float* __restrict__ img_prev, int H, int W, int C, int w_shared, int same_res,
                                                        float* __restrict__ img_out) {
    extern __shared__ float s_w[];                               // [3][C]
    const int n = blockIdx.y;
    const int wn = w_shared ? 0 : n;
    for (int e = threadIdx.x; e < 3 * C; e += blockDim.x) s_w[e] = wrgb[(size_t)wn * 3 * C + e];
    __syncthreads();
    const int pix = blockIdx.x * blockDim.x + threadIdx.x;
    if (pix >= H * W) return;
    const int Y = pix / W, X = pix - Y * W;
    const uint4* xp = reinterpret_cast<const uint4*>(x + ((size_t)n * H * W + pix) * C);
    float r = 0.f, g = 0.f, b = 0.f;
    for (int c8 = 0; c8 < C / 8; ++c8) {
        const uint4 raw = __ldg(xp + c8);
        const __half2* h = reinterpret_cast<const __half2*>(&raw);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float2 f = __half22float2(h[j]);
            const int c = c8 * 8 + 2 * j;
            r = fmaf(f.x, s_w[c], r); r = fmaf(f.y, s_w[c + 1], r);
            g = fmaf(f.x, s_w[C + c], g); g = fmaf(f.y, s_w[C + c + 1], g);
            b = fmaf(f.x, s_w[2 * C + c], b); b = fmaf(f.y, s_w[2 * C + c + 1], b);
        }
    }
    float out[3] = {r + brgb[0], g + brgb[1], b + brgb[2]};
    if (img_prev && same_res) {                                  // rgb = rgb + to_rgb(x) (LargeSynthesisBlock, superresolution.py:311,328)
#pragma unroll
        for (int c = 0; c < 3; ++c) out[c] += img_prev[((size_t)n * 3 + c) * H * W + pix];
    } else if (img_prev) {
        const int h = H / 2, w = W / 2;
#pragma unroll
        for (int c = 0; c < 3; ++c) out[c] += upsampled_skip(img_prev + ((size_t)n * 3 + c) * h * w, h, w, Y, X);
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) img_out[((size_t)n * 3 + c) * H * W + pix] = out[c];
}

// ---- host side: tensor maps -----------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    });
    return fn;
}

// fp16 tensor [d3][d2][d1][d0] (d0 innermost, dense), box {64, box1, 1, 1}, 128-byte swizzle, zero fill outside
static int make_map_4d_box(CUtensorMap* m, const void* ptr, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t d3, uint32_t box1);
static int make_map_4d(CUtensorMap* m, const void* ptr, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t d3, uint32_t box1) {
    return make_map_4d_box(m, ptr, d0, d1, d2, d3, box1);
}
static int make_map_4d_box(CUtensorMap* m, const void* ptr, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t d3, uint32_t box1) {
    EncodeTiledFn fn = encode_fn();
    R3DP_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled is not available from the driver");
    cuuint64_t dims[4] = {d0, d1, d2, d3};
    cuuint64_t strides[3] = {d0 * 2, d0 * d1 * 2, d0 * d1 * d2 * 2};
    cuuint32_t box[4] = {64, box1, 1, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    R3DP_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with CUresult %d (dims %llu x %llu x %llu x %llu)", (int)r,
                 (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2, (unsigned long long)d3);
    return 0;
}

static int make_map_fir(CUtensorMap* m, const void* ptr, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t d3, uint32_t box_rows) {
    EncodeTiledFn fn = encode_fn();
    R3DP_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled is not available from the driver");
    cuuint64_t dims[4] = {d0, d1, d2, d3};
    cuuint64_t strides[3] = {d0 * 2, d0 * d1 * 2, d0 * d1 * d2 * 2};
    cuuint32_t box[4] = {64, (cuuint32_t)FIR_BW, box_rows, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    R3DP_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (FIR) failed with CUresult %d", (int)r);
    return 0;
}

static int launch_conv2(const void* x, int N, int H, int W, int Cp, const void* wp, int Nw, int O, const ConvArgs& a1, cudaStream_t st);
static int launch_upconv2(const void* x, int N, int H, int W, int Cp, const void* wp, int Nw, int O, __half* yb, const float* bias, int split, cudaStream_t st);
static int launch_conv(const void* x, int N, int H, int W, int Cp, const void* wp, int Nw, int O, ConvArgs a, cudaStream_t st) {
    return launch_conv2(x, N, H, W, Cp, wp, Nw, O, a, st);
}

// ---- optional in-library timing of the conv launches (bench.py's roofline): CUDA events on the launching stream around each launch --------
struct ConvProf { bool on = false; std::vector<cudaEvent_t> ev; size_t used = 0; };
static ConvProf g_prof;
static void prof_mark(cudaStream_t st) {
    if (!g_prof.on) return;
    if (g_prof.used == g_prof.ev.size()) { cudaEvent_t e; if (cudaEventCreate(&e) != cudaSuccess) return; g_prof.ev.push_back(e); }
    cudaEventRecord(g_prof.ev[g_prof.used++], st);
}

static unsigned long long* g_debug_buf = nullptr;
static int g_debug_launch = 0;
static int tc_rows() {                         // R3DP_TC_ROWS = 1 | 2 | 4 output rows per tile (default 2: double-buffered accumulators)
    static int v = -1;
    if (v < 0) { const char* e = getenv("R3DP_TC_ROWS"); v = e ? atoi(e) : 2; if (v != 1 && v != 2 && v != 4) v = 2; }
    return v;
}

template <int R, bool SPLIT>
static int launch_conv3_rs(const CUtensorMap& tmA, const CUtensorMap& tmB, Conv2Args a, int max_rows, cudaStream_t st) {
    using C = Cfg3<R>;
    R3DP_CUDA(cudaFuncSetAttribute(conv_tc3_kernel<R, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM));
    a.debug = g_debug_buf ? g_debug_buf + 24 * (g_debug_launch++ % 32) : nullptr;
    a.row_groups = (max_rows + R - 1) / R;
    if ((a.row_groups * a.tiles_x) & 1) a.row_groups += 1;       // the two CTAs of a pair must work on units of the same (image, phase)
    a.total_units = a.n_images * a.n_phases * a.row_groups * a.tiles_x;
    int grid = a.total_units < sm_count() ? a.total_units : sm_count();
    grid &= ~1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kThreads3); cfg.dynamicSmemBytes = C::SMEM; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    prof_mark(st);
    R3DP_CUDA(cudaLaunchKernelEx(&cfg, conv_tc3_kernel<R, SPLIT>, tmA, tmB, a));
    prof_mark(st);
    count_launches(1);
    return 0;
}
template <int R>
static int launch_conv3_r(const CUtensorMap& tmA, const CUtensorMap& tmB, const Conv2Args& a, int max_rows, cudaStream_t st) {
    return a.split ? launch_conv3_rs<R, true>(tmA, tmB, a, max_rows, st) : launch_conv3_rs<R, false>(tmA, tmB, a, max_rows, st);
}

// taps given as (dy, dx, widx) lists -> sorted/grouped Taps2 (dy groups are contiguous for 3x3 and every transposed-conv phase)
static void fill_taps2(Taps2& t2, const Taps& t) {
    int order[9], n = t.n;
    for (int i = 0; i < n; ++i) order[i] = i;
    for (int i = 0; i < n; ++i)
        for (int j = i + 1; j < n; ++j) {
            const int a = order[i], b = order[j];
            if (t.dy[b] < t.dy[a] || (t.dy[b] == t.dy[a] && t.dx[b] < t.dx[a])) { order[i] = b; order[j] = a; }
        }
    int dy_min = 99;
    for (int i = 0; i < n; ++i) if (t.dy[i] < dy_min) dy_min = t.dy[i];
    t2.n = n; t2.dy_min = dy_min; t2.ngroups = 0;
    int last = -99;
    for (int i = 0; i < n; ++i) {
        const int o = order[i];
        if (t.dy[o] != last) { t2.gstart[t2.ngroups++] = i; last = t.dy[o]; }
        t2.dyi[i] = t.dy[o] - dy_min; t2.shift[i] = t.dx[o] + 1; t2.widx[i] = t.widx[o];      // strip box starts at x0 - 1
    }
    t2.gstart[t2.ngroups] = n;
}

static int run_conv2(const void* x, int N, int H, int W, int Cp, const void* wp, int Nw, int O, Conv2Args& a, int max_rows, cudaStream_t st, int n_taps = 9) {
    CUtensorMap tmA, tmB;
    const uint64_t Cphys = (uint64_t)Cp * (a.split ? 2 : 1);                      // split: [hi | lo] halves of Cp channels each
    if (make_map_4d_box(&tmA, x, Cphys, (uint64_t)W, (uint64_t)H, (uint64_t)N, A2_ROWS)) return 1;
    if (make_map_4d_box(&tmB, wp, Cphys, (uint64_t)O, (uint64_t)n_taps, (uint64_t)Nw, BN / 2)) return 1;
    if (a.split) { R3DP_REQUIRE(a.residual == nullptr, "conv_tc3: the residual epilogue is not built for split operands"); a.acc_scale = 1.0f / kSplitWeightScale; a.lo_off = a.out_C; a.out_C *= 2; }
    else { a.acc_scale = 1.0f; a.lo_off = 0; }
    a.k_chunks = Cp / BK; a.tiles_x = W / BM; a.n_blocks = O / BN; a.n_images = N; a.w_shared = (Nw == 1);
    { static int mixv = -1; if (mixv < 0) { const char* e = getenv("R3DP_TC_MIX"); mixv = (e && e[0] == '0') ? 0 : 1; } a.phase_mix = mixv; }      // A/B knob
    if (a.act_gain == 0.f) { a.act_slope = 0.2f; a.act_gain = 1.4142135623730951f; }      // default: bias_act lrelu
    R3DP_REQUIRE(a.n_blocks >= 1 && a.n_blocks <= 2, "conv_tc3: needs Cout == 128 or Cout == 256 (got Cout=%d)", O);
    return tc_rows() == 1 ? launch_conv3_r<1>(tmA, tmB, a, max_rows, st) : (tc_rows() == 4 ? launch_conv3_r<4>(tmA, tmB, a, max_rows, st) : launch_conv3_r<2>(tmA, tmB, a, max_rows, st));
}

// v1-style single-phase description -> v2 launch
static int launch_conv2(const void* x, int N, int H, int W, int Cp, const void* wp, int Nw, int O, const ConvArgs& a1, cudaStream_t st) {
    Conv2Args a = {};
    a.n_phases = 1;
    fill_taps2(a.ph[0].taps, a1.taps);
    a.ph[0].rows = a1.rows; a.ph[0].oy_off = a1.oy_off; a.ph[0].ox_off = a1.ox_off;
    a.mode = a1.mode; a.out = a1.out; a.out_H = a1.out_H; a.out_W = a1.out_W; a.out_C = a1.out_C; a.oy_mul = a1.oy_mul; a.ox_mul = a1.ox_mul;
    a.bias = a1.bias; a.wrgb = a1.wrgb; a.brgb = a1.brgb; a.img_prev = a1.img_prev; a.img_out = a1.img_out; a.img_H = a1.out_H; a.img_W = a1.out_W;
    a.out_clamp = a1.out_clamp; a.img_out_u8 = a1.img_out_u8; a.split = a1.split;
    return run_conv2(x, N, H, W, Cp, wp, Nw, O, a, a1.rows, st);
}

// all four output-parity phases of the stride-2 transposed conv in ONE persistent launch (raw fp16 result on the (2H+1)x(2W+1) grid)
static int launch_upconv2(const void* x, int N, int H, int W, int Cp, const void* wp, int Nw, int O, __half* yb, const float* bias, int split, cudaStream_t st) {
    Conv2Args a = {};
    a.n_phases = 4; a.split = split;
    for (int pa = 0; pa < 2; ++pa)
        for (int pb = 0; pb < 2; ++pb) {
            Taps t = {};
            for (int ky = pa; ky < 3; ky += 2)
                for (int kx = pb; kx < 3; kx += 2) { const int i = t.n++; t.dy[i] = -(ky >> 1); t.dx[i] = -(kx >> 1); t.widx[i] = ky * 3 + kx; }
            Phase2& P = a.ph[pa * 2 + pb];
            fill_taps2(P.taps, t);
            P.rows = pa ? H : H + 1; P.oy_off = pa; P.ox_off = pb;
        }
    a.mode = kStoreRaw; a.out = yb; a.out_H = 2 * H + 1; a.out_W = 2 * W + 1; a.out_C = O; a.oy_mul = a.ox_mul = 2; a.bias = bias;
    return run_conv2(x, N, H, W, Cp, wp, Nw, O, a, H + 1, st);
}

}  // namespace tc
}  // namespace r3dp

using namespace r3dp;
using namespace r3dp::tc;

static int pack_weights_impl(const float* wf, int Nw, int O, int I, void* packed_f16, int split, r3dp_stream_t stream) {
    R3DP_REQUIRE(wf && packed_f16, "sr_tc_pack_weights: null pointer");
    R3DP_REQUIRE(Nw > 0 && O > 0 && I > 0, "sr_tc_pack_weights: bad shape");
    const int Ip = (I + 63) / 64 * 64;
    const long long total = (long long)Nw * 9 * O * Ip;
    pack_weights_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(wf, Nw, O, I, Ip, split, reinterpret_cast<__half*>(packed_f16));
    R3DP_LAUNCH_CHECK();
    count_launches(1);
    return 0;
}
extern "C" int r3dp_sr_tc_pack_weights(const float* wf, int Nw, int O, int I, void* packed_f16, r3dp_stream_t stream) { return pack_weights_impl(wf, Nw, O, I, packed_f16, 0, stream); }
extern "C" int r3dp_sr_tcx_pack_weights(const float* wf, int Nw, int O, int I, void* packed_f16, r3dp_stream_t stream) { return pack_weights_impl(wf, Nw, O, I, packed_f16, 1, stream); }

static int input_impl(const float* x, int N, int C, int h, int w, int size, void* y_f16, int split, r3dp_stream_t stream) {
    R3DP_REQUIRE(x && y_f16, "sr_tc_input: null pointer");
    R3DP_REQUIRE(N > 0 && C > 0 && h > 0 && w > 0 && size >= h && size >= w, "sr_tc_input: up-scaling (or copy) only");
    const int Cp = (C + 63) / 64 * 64;
    const long long total = (long long)N * size * size * Cp;
    resize_to_nhwc_f16_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(x, N, C, h, w, size, Cp, split, reinterpret_cast<__half*>(y_f16));
    R3DP_LAUNCH_CHECK();
    count_launches(1);
    return 0;
}
extern "C" int r3dp_sr_tc_input(const float* x, int N, int C, int h, int w, int size, void* y_f16, r3dp_stream_t stream) { return input_impl(x, N, C, h, w, size, y_f16, 0, stream); }
extern "C" int r3dp_sr_tcx_input(const float* x, int N, int C, int h, int w, int size, void* y_f16, r3dp_stream_t stream) { return input_impl(x, N, C, h, w, size, y_f16, 1, stream); }

extern "C" size_t r3dp_sr_tc_scratch_bytes(int N, int O, int H, int W) { return (size_t)N * (2 * H + 1) * (2 * W + 1) * O * sizeof(__half); }
extern "C" size_t r3dp_sr_tcx_scratch_bytes(int N, int O, int H, int W) { return 2 * r3dp_sr_tc_scratch_bytes(N, O, H, W); }

// SynthesisLayer on tensor cores.  x [N][H][W][Ip] fp16 NHWC (Ip = I rounded up to 64), wp packed weights [Nw][9][O][Ip] fp16
// (Nw == N per-sample, or 1 shared), bias [O] fp32.  up == 1: y [N][H][W][O]; up == 2: y [N][2H][2W][O], scratch >= r3dp_sr_tc_scratch_bytes.
static int layer_impl(const void* x_f16, const void* wp_f16, const float* bias, int N, int Nw, int I, int O, int H, int W, int up,
                      void* y_f16, void* scratch, int split, r3dp_stream_t stream) {
    R3DP_REQUIRE(x_f16 && wp_f16 && bias && y_f16, "sr_tc_layer: null pointer");
    R3DP_REQUIRE(N > 0 && (Nw == N || Nw == 1) && I > 0 && H > 0, "sr_tc_layer: bad shape (needs N, I, H > 0 and Nw == N or Nw == 1; got N=%d, Nw=%d, I=%d, H=%d)",
                 N, Nw, I, H);
    R3DP_REQUIRE(W % BM == 0 && O % BN == 0, "sr_tc_layer: needs W %% 128 == 0 and Cout %% 128 == 0 (got W=%d, Cout=%d)", W, O);
    R3DP_REQUIRE(up == 1 || up == 2, "sr_tc_layer: up must be 1 or 2 (got up=%d)", up);
    const int Ip = (I + 63) / 64 * 64;
    cudaStream_t st = as_stream(stream);
    ConvArgs a = {};
    a.bias = bias; a.split = split;
    if (up == 1) {
        a.taps.n = 9;
        for (int t = 0; t < 9; ++t) { a.taps.dy[t] = t / 3 - 1; a.taps.dx[t] = t % 3 - 1; a.taps.widx[t] = t; }
        a.tiles_x = W / BM; a.rows = H; a.mode = kStoreAct;
        a.out = reinterpret_cast<__half*>(y_f16); a.out_H = H; a.out_W = W; a.out_C = O; a.oy_mul = a.ox_mul = 1;
        return launch_conv(x_f16, N, H, W, Ip, wp_f16, Nw, O, a, st);
    }
    // every check of the up=2 path runs before its first launch: a rejected call enqueues nothing and leaves the scratch untouched
    R3DP_REQUIRE(scratch, "sr_tc_layer: up=2 needs scratch");
    R3DP_REQUIRE(Ip <= 256, "sr_tc_layer: up=2 supports at most 256 input channels");
    R3DP_REQUIRE((2 * W) % FIR_TW == 0 && O % 64 == 0, "sr_tc_layer: FIR needs 2W %% 32 == 0 and Cout %% 64 == 0");
    __half* yb = reinterpret_cast<__half*>(scratch);
    CUtensorMap tmY, tmY8;
    if (make_map_fir(&tmY, yb, (uint64_t)O * (split ? 2 : 1), (uint64_t)(2 * W + 1), (uint64_t)(2 * H + 1), (uint64_t)N, FIR_BH)) return 1;
    if (make_map_fir(&tmY8, yb, (uint64_t)O * (split ? 2 : 1), (uint64_t)(2 * W + 1), (uint64_t)(2 * H + 1), (uint64_t)N, FIR_TH)) return 1;
    if (launch_upconv2(x_f16, N, H, W, Ip, wp_f16, Nw, O, yb, bias, split, st)) return 1;
    {
        const int erows = split ? kEdgeRowsSplit : kEdgeRows;
        dim3 grid((2 * H + 1 + erows - 1) / erows, (O + kEdgeCo - 1) / kEdgeCo, N);
        const size_t esmem = ((size_t)(kEdgeRows / 2 + 2) * Ip + 3 * (size_t)kEdgeCo * (Ip + 8)) * sizeof(__half);
        if (split) {
            const size_t ssmem = ((size_t)(kEdgeRowsSplit / 2 + 2) * Ip + 3 * (size_t)kEdgeCo * (Ip + 4)) * sizeof(float);
            R3DP_CUDA(cudaFuncSetAttribute(upconv_edge_split_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024));
            upconv_edge_split_kernel<<<grid, 256, ssmem, st>>>(reinterpret_cast<const __half*>(x_f16), reinterpret_cast<const __half*>(wp_f16), H, W, Ip, O,
                                                           Nw == 1, yb);
        } else {
        R3DP_CUDA(cudaFuncSetAttribute(upconv_edge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024));
        upconv_edge_kernel<<<grid, 256, esmem, st>>>(reinterpret_cast<const __half*>(x_f16), reinterpret_cast<const __half*>(wp_f16), H, W, Ip, O,
                                                 Nw == 1, yb);
        }
    }
    {
        const int total = N * (O / 64) * ((2 * H + FIR_SEG - 1) / FIR_SEG) * (2 * W / FIR_TW);
        if (split) {
            const int smem = 4 * FIR_SLOT + 1024 + 64;
            R3DP_CUDA(cudaFuncSetAttribute(fir_tma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
            const int grid = total < sm_count() ? total : sm_count();
            fir_tma_kernel<true><<<grid, 256, smem, st>>>(tmY, tmY8, bias, N, 2 * H, 2 * W, O, reinterpret_cast<__half*>(y_f16));
        } else {
            R3DP_CUDA(cudaFuncSetAttribute(fir_tma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, FIR_SMEM));
            const int grid = total < 2 * sm_count() ? total : 2 * sm_count();
            fir_tma_kernel<false><<<grid, 256, FIR_SMEM, st>>>(tmY, tmY8, bias, N, 2 * H, 2 * W, O, reinterpret_cast<__half*>(y_f16));
        }
    }
    R3DP_LAUNCH_CHECK();
    count_launches(2);
    return 0;
}
extern "C" int r3dp_sr_tc_layer(const void* x_f16, const void* wp_f16, const float* bias, int N, int Nw, int I, int O, int H, int W, int up,
                                void* y_f16, void* scratch, r3dp_stream_t stream) {
    return layer_impl(x_f16, wp_f16, bias, N, Nw, I, O, H, W, up, y_f16, scratch, 0, stream);
}
extern "C" int r3dp_sr_tcx_layer(const void* x_f16, const void* wp_f16, const float* bias, int N, int Nw, int I, int O, int H, int W, int up,
                                 void* y_f16, void* scratch, r3dp_stream_t stream) {
    return layer_impl(x_f16, wp_f16, bias, N, Nw, I, O, H, W, up, y_f16, scratch, 1, stream);
}

// Last layer fused with ToRGB: conv3x3 (I -> 128) + bias + lrelu, then img_out = upsample2d(img_prev) + torgb + brgb; the 128-channel
// activation itself is never written (SynthesisBlock is_last: only the image leaves the block).
static int last_layer_impl(const void* x_f16, const void* wp_f16, const float* bias, const float* wrgb, const float* brgb,
                           const float* img_prev, int N, int Nw, int I, int H, int W, float* img_out, uint8_t* img_out_u8, int clamp, int split,
                           r3dp_stream_t stream) {
    R3DP_REQUIRE(x_f16 && wp_f16 && bias && wrgb && brgb && (img_out || img_out_u8), "sr_tc_last_layer: null pointer");
    R3DP_REQUIRE(N > 0 && (Nw == N || Nw == 1) && W % BM == 0 && H % 2 == 0,
                 "sr_tc_last_layer: bad shape (needs N > 0, Nw == N or Nw == 1, W %% 128 == 0, H %% 2 == 0; got N=%d, Nw=%d, H=%d, W=%d)", N, Nw, H, W);
    const int Ip = (I + 63) / 64 * 64;
    ConvArgs a = {};
    a.bias = bias; a.wrgb = wrgb; a.brgb = brgb; a.img_prev = img_prev; a.img_out = img_out; a.img_out_u8 = img_out_u8; a.out_clamp = clamp || img_out_u8;
    a.split = split;
    a.taps.n = 9;
    for (int t = 0; t < 9; ++t) { a.taps.dy[t] = t / 3 - 1; a.taps.dx[t] = t % 3 - 1; a.taps.widx[t] = t; }
    a.tiles_x = W / BM; a.rows = H; a.mode = kToRgbFinal; a.out_H = H; a.out_W = W; a.out_C = BN; a.oy_mul = a.ox_mul = 1;
    return launch_conv(x_f16, N, H, W, Ip, wp_f16, Nw, BN, a, as_stream(stream));
}
extern "C" int r3dp_sr_tc_last_layer_ex(const void* x_f16, const void* wp_f16, const float* bias, const float* wrgb, const float* brgb,
                                        const float* img_prev, int N, int Nw, int I, int H, int W, float* img_out, uint8_t* img_out_u8, int clamp,
                                        r3dp_stream_t stream) {
    return last_layer_impl(x_f16, wp_f16, bias, wrgb, brgb, img_prev, N, Nw, I, H, W, img_out, img_out_u8, clamp, 0, stream);
}
extern "C" int r3dp_sr_tcx_last_layer(const void* x_f16, const void* wp_f16, const float* bias, const float* wrgb, const float* brgb,
                                      const float* img_prev, int N, int Nw, int I, int H, int W, float* img_out, uint8_t* img_out_u8, int clamp,
                                      r3dp_stream_t stream) {
    return last_layer_impl(x_f16, wp_f16, bias, wrgb, brgb, img_prev, N, Nw, I, H, W, img_out, img_out_u8, clamp, 1, stream);
}
extern "C" int r3dp_sr_tc_last_layer(const void* x_f16, const void* wp_f16, const float* bias, const float* wrgb, const float* brgb,
                                     const float* img_prev, int N, int Nw, int I, int H, int W, float* img_out, r3dp_stream_t stream) {
    return r3dp_sr_tc_last_layer_ex(x_f16, wp_f16, bias, wrgb, brgb, img_prev, N, Nw, I, H, W, img_out, nullptr, 0, stream);
}

// ToRGB of a non-final block: x NHWC fp16 [N][H][W][C] -> img_out NCHW fp32 [N][3][H][W] (+ upsample2d(img_prev) + bias).
extern "C" int r3dp_sr_tc_torgb_ex(const void* x_f16, const float* wrgb, const float* brgb, const float* img_prev, int same_res, int N, int Nw, int C,
                                   int H, int W, float* img_out, r3dp_stream_t stream) {
    R3DP_REQUIRE(x_f16 && wrgb && brgb && img_out, "sr_tc_torgb: null pointer");
    R3DP_REQUIRE(N > 0 && (Nw == N || Nw == 1) && C % 8 == 0 && H % 2 == 0 && W % 2 == 0, "sr_tc_torgb: bad shape");
    dim3 grid((H * W + 255) / 256, N);
    torgb_f16_kernel<<<grid, 256, 3 * C * sizeof(float), as_stream(stream)>>>(reinterpret_cast<const __half*>(x_f16), wrgb, brgb, img_prev, H, W, C,
                                                                              Nw == 1, same_res, img_out);
    R3DP_LAUNCH_CHECK();
    count_launches(1);
    return 0;
}
extern "C" int r3dp_sr_tc_torgb(const void* x_f16, const float* wrgb, const float* brgb, const float* img_prev, int N, int Nw, int C, int H,
                                int W, float* img_out, r3dp_stream_t stream) {
    return r3dp_sr_tc_torgb_ex(x_f16, wrgb, brgb, img_prev, 0, N, Nw, C, H, W, img_out, stream);
}

// SynthesisLayer (up == 1) fused with the block's ToRGB + skip (networks_stylegan2.py:463-469): y [N,H,W,O] fp16 AND
// img_out [N,3,H,W] fp32 = upsample2d(img_prev [N,3,H/2,W/2]) + conv1x1(y, wrgb [Nw,3,O]) + brgb.  O = 128 or 256.
static int layer_torgb_impl(const void* x_f16, const void* wp_f16, const float* bias, const float* wrgb, const float* brgb,
                            const float* img_prev, int N, int Nw, int I, int O, int H, int W, void* y_f16, float* img_out, int split,
                            r3dp_stream_t stream) {
    R3DP_REQUIRE(x_f16 && wp_f16 && bias && wrgb && brgb && y_f16 && img_out, "sr_tc_layer_torgb: null pointer");
    R3DP_REQUIRE(N > 0 && (Nw == N || Nw == 1) && W % BM == 0 && O % BN == 0 && O <= 256 && H % 2 == 0,
                 "sr_tc_layer_torgb: bad shape (needs N > 0, Nw == N or Nw == 1, W %% 128 == 0, Cout 128 or 256, H %% 2 == 0; got N=%d, Nw=%d, Cout=%d, H=%d, W=%d)",
                 N, Nw, O, H, W);
    const int Ip = (I + 63) / 64 * 64;
    Conv2Args a = {};
    Taps t = {};
    t.n = 9;
    for (int i = 0; i < 9; ++i) { t.dy[i] = i / 3 - 1; t.dx[i] = i % 3 - 1; t.widx[i] = i; }
    a.n_phases = 1;
    fill_taps2(a.ph[0].taps, t);
    a.ph[0].rows = H; a.ph[0].oy_off = 0; a.ph[0].ox_off = 0;
    a.mode = kActRgb; a.out = reinterpret_cast<__half*>(y_f16); a.out_H = H; a.out_W = W; a.out_C = O; a.oy_mul = a.ox_mul = 1;
    a.bias = bias; a.wrgb = wrgb; a.brgb = brgb; a.img_prev = img_prev; a.img_out = img_out; a.img_H = H; a.img_W = W; a.split = split;
    return run_conv2(x_f16, N, H, W, Ip, wp_f16, Nw, O, a, H, as_stream(stream));
}
extern "C" int r3dp_sr_tc_layer_torgb(const void* x_f16, const void* wp_f16, const float* bias, const float* wrgb, const float* brgb,
                                      const float* img_prev, int N, int Nw, int I, int O, int H, int W, void* y_f16, float* img_out,
                                      r3dp_stream_t stream) {
    return layer_torgb_impl(x_f16, wp_f16, bias, wrgb, brgb, img_prev, N, Nw, I, O, H, W, y_f16, img_out, 0, stream);
}
extern "C" int r3dp_sr_tcx_layer_torgb(const void* x_f16, const void* wp_f16, const float* bias, const float* wrgb, const float* brgb,
                                       const float* img_prev, int N, int Nw, int I, int O, int H, int W, void* y_f16, float* img_out,
                                       r3dp_stream_t stream) {
    return layer_torgb_impl(x_f16, wp_f16, bias, wrgb, brgb, img_prev, N, Nw, I, O, H, W, y_f16, img_out, 1, stream);
}

// bilinear up-resize of a CHANNELS-LAST fp32 image [N,h,w,C] (e.g. the renderer's [N,M,32] output viewed as an image) to
// NHWC fp16 [N,size,size,Cpad]: one thread = one output pixel x 8 channels.
__global__ void resize_nhwc_to_f16_kernel(const float* __restrict__ x, int N, int C, int h, int w, int size, int Cp, int split, __half* __restrict__ y,
                                          float* __restrict__ rgb_out) {
    const int cv = Cp / 8;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)N * size * size * cv) return;
    const int c8 = (int)(idx % cv); const int ox = (int)((idx / cv) % size); const int oy = (int)((idx / ((long long)cv * size)) % size);
    const int n = (int)(idx / ((long long)cv * size * size));
    float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (c8 * 8 < C) {
        const float sy = fmaxf(((float)oy + 0.5f) * ((float)h / (float)size) - 0.5f, 0.f);
        const float sx = fmaxf(((float)ox + 0.5f) * ((float)w / (float)size) - 0.5f, 0.f);
        const int y0 = min((int)sy, h - 1), x0 = min((int)sx, w - 1), y1 = min(y0 + 1, h - 1), x1 = min(x0 + 1, w - 1);
        const float ty = sy - (float)y0, tx = sx - (float)x0;
        const float* b = x + (size_t)n * h * w * C + c8 * 8;
        const float4* p00 = reinterpret_cast<const float4*>(b + ((size_t)y0 * w + x0) * C);
        const float4* p10 = reinterpret_cast<const float4*>(b + ((size_t)y1 * w + x0) * C);
        const float4* p01 = reinterpret_cast<const float4*>(b + ((size_t)y0 * w + x1) * C);
        const float4* p11 = reinterpret_cast<const float4*>(b + ((size_t)y1 * w + x1) * C);
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const float4 a00 = __ldg(p00 + q), a10 = __ldg(p10 + q), a01 = __ldg(p01 + q), a11 = __ldg(p11 + q);
            const float e00[4] = {a00.x, a00.y, a00.z, a00.w}, e10[4] = {a10.x, a10.y, a10.z, a10.w};
            const float e01[4] = {a01.x, a01.y, a01.z, a01.w}, e11[4] = {a11.x, a11.y, a11.z, a11.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float r0 = e00[j] * (1.f - ty) + e10[j] * ty, r1 = e01[j] * (1.f - ty) + e11[j] * ty;
                v[q * 4 + j] = r0 * (1.f - tx) + r1 * tx;
            }
        }
    }
    if (rgb_out != nullptr && c8 == 0) {                       // channels 0..2 = the raw RGB image the SR takes beside the features (secc_img2plane.py:126), fp32 NCHW
#pragma unroll
        for (int c = 0; c < 3; ++c) rgb_out[(((size_t)n * 3 + c) * size + oy) * size + ox] = v[c];
    }
    uint4 pk; __half2* ph = reinterpret_cast<__half2*>(&pk);
#pragma unroll
    for (int j = 0; j < 4; ++j) ph[j] = __floats2half2_rn(v[2 * j], v[2 * j + 1]);
    if (!split) { *reinterpret_cast<uint4*>(y + idx * 8) = pk; return; }
    uint4 pl; __half2* pq = reinterpret_cast<__half2*>(&pl);
#pragma unroll
    for (int j = 0; j < 4; ++j) { const float2 hf = __half22float2(ph[j]); pq[j] = __floats2half2_rn(v[2 * j] - hf.x, v[2 * j + 1] - hf.y); }
    const size_t pix = (size_t)(idx / cv) * (size_t)(2 * Cp);
    *reinterpret_cast<uint4*>(y + pix + c8 * 8) = pk;
    *reinterpret_cast<uint4*>(y + pix + Cp + c8 * 8) = pl;
}

static int input_nhwc_impl(const float* x_nhwc, int N, int C, int h, int w, int size, void* y_f16, float* rgb_out, int split, r3dp_stream_t stream) {
    R3DP_REQUIRE(x_nhwc && y_f16, "sr_tc_input_nhwc: null pointer");
    R3DP_REQUIRE(N > 0 && C > 0 && C % 8 == 0 && h > 0 && w > 0 && size >= h && size >= w, "sr_tc_input_nhwc: bad shape (C %% 8 == 0, up-scaling only)");
    const int Cp = (C + 63) / 64 * 64;
    const long long total = (long long)N * size * size * (Cp / 8);
    resize_nhwc_to_f16_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(x_nhwc, N, C, h, w, size, Cp, split, reinterpret_cast<__half*>(y_f16), rgb_out);
    R3DP_LAUNCH_CHECK();
    count_launches(1);
    return 0;
}
extern "C" int r3dp_sr_tc_input_nhwc(const float* x_nhwc, int N, int C, int h, int w, int size, void* y_f16, r3dp_stream_t stream) { return input_nhwc_impl(x_nhwc, N, C, h, w, size, y_f16, nullptr, 0, stream); }
extern "C" int r3dp_sr_tcx_input_nhwc(const float* x_nhwc, int N, int C, int h, int w, int size, void* y_f16, r3dp_stream_t stream) { return input_nhwc_impl(x_nhwc, N, C, h, w, size, y_f16, nullptr, 1, stream); }
// the same, plus rgb_out [N,3,size,size] fp32 = the bilinear resize of channels 0..2 (the raw RGB image of the render head, secc_img2plane.py:126)
extern "C" int r3dp_sr_tc_input_nhwc_rgb(const float* x_nhwc, int N, int C, int h, int w, int size, void* y_f16, float* rgb_out, int split, r3dp_stream_t stream) {
    R3DP_REQUIRE(rgb_out != nullptr && C >= 3, "sr_tc_input_nhwc_rgb: needs rgb_out and at least 3 channels");
    return input_nhwc_impl(x_nhwc, N, C, h, w, size, y_f16, rgb_out, split != 0, stream);
}

// ---- composed up-convolution for small Cin -------------------------------------------------------------------------------
// FIR(conv_transpose(x, w)) == four 3x3 correlations on the low-resolution input, one per output parity (p,q), with weights
//   G[p][q][dy][dx] = sum_{ky,kx} A[p][dy][ky] * A[q][dx][kx] * w[ky][kx],   A[p][dy][ky] = sum_u g[u] * [p + u - 1 - ky == 2 dy],
// g = [1,3,3,1]/4 (FIR * gain 4), dy,dx in {-1,0,1}  (derivation in DESIGN.md).  This costs 4x the MACs of the two-step form but
// needs no (2H+1)x(2W+1) intermediate, no FIR pass and no edge column: a win when Cin is small (block0.conv0: 32 -> 256).
// wf fp32 [Nw][O][I][3][3] -> packed fp16 [Nw][36][O][Ip], tap index = (p*2+q)*9 + (dy+1)*3 + (dx+1).
__global__ void compose_up_weights_kernel(const float* __restrict__ wf, int Nw, int O, int I, int Ip, int split, __half* __restrict__ out) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)Nw * 36 * O * Ip;
    if (idx >= total) return;
    const int i = (int)(idx % Ip); const int o = (int)((idx / Ip) % O); const int t = (int)((idx / ((long long)Ip * O)) % 36);
    const int nw = (int)(idx / ((long long)Ip * O * 36));
    float acc = 0.f;
    if (i < I) {
        const int ph = t / 9, tap = t % 9, p = ph >> 1, q = ph & 1, dy = tap / 3 - 1, dx = tap % 3 - 1;
        const float g[4] = {0.25f, 0.75f, 0.75f, 0.25f};
        const float* w = wf + (((size_t)nw * O + o) * I + i) * 9;
        for (int ky = 0; ky < 3; ++ky) {
            const int u = 2 * dy + 1 + ky - p;                      // p + u - 1 - ky == 2 dy
            if (u < 0 || u > 3) continue;
            for (int kx = 0; kx < 3; ++kx) {
                const int v = 2 * dx + 1 + kx - q;
                if (v < 0 || v > 3) continue;
                acc = fmaf(g[u] * g[v], w[ky * 3 + kx], acc);
            }
        }
    }
    if (!split) { out[idx] = __float2half_rn(acc); return; }
    __half hi, lo;
    split_half(acc * kSplitWeightScale, hi, lo);
    const size_t row = (idx / Ip) * (size_t)(2 * Ip);
    out[row + i] = hi; out[row + Ip + i] = lo;
}

static int pack_up_composed_impl(const float* wf, int Nw, int O, int I, void* packed_f16, int split, r3dp_stream_t stream) {
    R3DP_REQUIRE(wf && packed_f16, "sr_tc_pack_weights_up_composed: null pointer");
    R3DP_REQUIRE(Nw > 0 && O > 0 && I > 0, "sr_tc_pack_weights_up_composed: bad shape");
    const int Ip = (I + 63) / 64 * 64;
    const long long total = (long long)Nw * 36 * O * Ip;
    compose_up_weights_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(wf, Nw, O, I, Ip, split, reinterpret_cast<__half*>(packed_f16));
    R3DP_LAUNCH_CHECK();
    count_launches(1);
    return 0;
}
extern "C" int r3dp_sr_tc_pack_weights_up_composed(const float* wf, int Nw, int O, int I, void* packed_f16, r3dp_stream_t stream) { return pack_up_composed_impl(wf, Nw, O, I, packed_f16, 0, stream); }
extern "C" int r3dp_sr_tcx_pack_weights_up_composed(const float* wf, int Nw, int O, int I, void* packed_f16, r3dp_stream_t stream) { return pack_up_composed_impl(wf, Nw, O, I, packed_f16, 1, stream); }

// SynthesisLayer with up == 2 through the composed weights: x [N][H][W][Ip] fp16 -> y [N][2H][2W][O] fp16 (bias + lrelu fused).
static int layer_up_composed_impl(const void* x_f16, const void* wpc_f16, const float* bias, int N, int Nw, int I, int O, int H,
                                  int W, void* y_f16, int split, r3dp_stream_t stream) {
    R3DP_REQUIRE(x_f16 && wpc_f16 && bias && y_f16, "sr_tc_layer_up_composed: null pointer");
    R3DP_REQUIRE(N > 0 && (Nw == N || Nw == 1) && W % BM == 0 && O % BN == 0 && O <= 256,
                 "sr_tc_layer_up_composed: bad shape (needs N > 0, Nw == N or Nw == 1, W %% 128 == 0, Cout 128 or 256; got N=%d, Nw=%d, Cout=%d, W=%d)", N, Nw, O, W);
    const int Ip = (I + 63) / 64 * 64;
    Conv2Args a = {};
    a.n_phases = 4;
    for (int ph = 0; ph < 4; ++ph) {
        Taps t = {};
        t.n = 9;
        for (int i = 0; i < 9; ++i) { t.dy[i] = i / 3 - 1; t.dx[i] = i % 3 - 1; t.widx[i] = ph * 9 + i; }
        fill_taps2(a.ph[ph].taps, t);
        a.ph[ph].rows = H; a.ph[ph].oy_off = ph >> 1; a.ph[ph].ox_off = ph & 1;
    }
    a.mode = kStoreAct; a.out = reinterpret_cast<__half*>(y_f16); a.out_H = 2 * H; a.out_W = 2 * W; a.out_C = O; a.oy_mul = a.ox_mul = 2;
    a.bias = bias; a.split = split;
    return run_conv2(x_f16, N, H, W, Ip, wpc_f16, Nw, O, a, H, as_stream(stream), 36);
}
extern "C" int r3dp_sr_tc_layer_up_composed(const void* x_f16, const void* wpc_f16, const float* bias, int N, int Nw, int I, int O, int H,
                                            int W, void* y_f16, r3dp_stream_t stream) {
    return layer_up_composed_impl(x_f16, wpc_f16, bias, N, Nw, I, O, H, W, y_f16, 0, stream);
}
extern "C" int r3dp_sr_tcx_layer_up_composed(const void* x_f16, const void* wpc_f16, const float* bias, int N, int Nw, int I, int O, int H,
                                             int W, void* y_f16, r3dp_stream_t stream) {
    return layer_up_composed_impl(x_f16, wpc_f16, bias, N, Nw, I, O, H, W, y_f16, 1, stream);
}

// ---- building blocks of the torso head (modules/real3d/super_resolution/sr_with_ref.py:16-162) --------------------------------
// Plain nn.Conv2d (k = 1 or 3, stride 1, "same" padding) [+ activation] on the tensor-core path: x [N][H][W][Ip] fp16, weights packed by
// r3dp_sr_tc_pack_weights from the [1][O][I][k][k] fp32 tensor (k = 1: the value sits in tap 4), y [N][H][W][O] fp16.
// act: 0 = linear, 1 = lrelu(0.2)*sqrt2 (bias_act), 2 = nn.LeakyReLU() (slope 0.01).
static int conv_res_impl(const void* x_f16, const void* wp_f16, const float* bias, int N, int Nw, int I, int O, int H, int W, int ksize,
                         int act, const void* residual_f16, void* y_f16, int split, r3dp_stream_t stream) {
    R3DP_REQUIRE(x_f16 && wp_f16 && bias && y_f16, "sr_tc_conv: null pointer");
    R3DP_REQUIRE(N > 0 && (Nw == N || Nw == 1) && W % BM == 0 && O % BN == 0 && O <= 256,
                 "sr_tc_conv: bad shape (needs N > 0, Nw == N or Nw == 1, W %% 128 == 0, Cout 128 or 256; got N=%d, Nw=%d, Cout=%d, W=%d)", N, Nw, O, W);
    R3DP_REQUIRE(ksize == 1 || ksize == 3, "sr_tc_conv: ksize must be 1 or 3 (got %d)", ksize);
    R3DP_REQUIRE(act >= 0 && act <= 3, "sr_tc_conv: act must be 0..3 (got %d)", act);
    const int Ip = (I + 63) / 64 * 64;
    Conv2Args a = {};
    Taps t = {};
    if (ksize == 3) { t.n = 9; for (int i = 0; i < 9; ++i) { t.dy[i] = i / 3 - 1; t.dx[i] = i % 3 - 1; t.widx[i] = i; } }
    else { t.n = 1; t.dy[0] = 0; t.dx[0] = 0; t.widx[0] = 4; }
    a.n_phases = 1;
    fill_taps2(a.ph[0].taps, t);
    a.ph[0].rows = H;
    a.mode = kStoreAct; a.out = reinterpret_cast<__half*>(y_f16); a.out_H = H; a.out_W = W; a.out_C = O; a.oy_mul = a.ox_mul = 1; a.bias = bias;
    a.act_slope = act == 0 ? 1.0f : (act == 1 ? 0.2f : (act == 2 ? 0.01f : 0.0f));      // max(v, v*slope): slope 0 = ReLU
    a.act_gain = act == 1 ? 1.4142135623730951f : 1.0f;
    a.residual = reinterpret_cast<const __half*>(residual_f16);
    a.split = split;
    return run_conv2(x_f16, N, H, W, Ip, wp_f16, Nw, O, a, H, as_stream(stream));
}
extern "C" int r3dp_sr_tc_conv_res(const void* x_f16, const void* wp_f16, const float* bias, int N, int Nw, int I, int O, int H, int W, int ksize,
                                   int act, const void* residual_f16, void* y_f16, r3dp_stream_t stream) {
    return conv_res_impl(x_f16, wp_f16, bias, N, Nw, I, O, H, W, ksize, act, residual_f16, y_f16, 0, stream);
}
// the same plain convolution with split fp16 operands ([hi | lo] tensors, see the r3dp_sr_tcx_* family): fp32-grade results
extern "C" int r3dp_sr_tcx_conv(const void* x_f16, const void* wp_f16, const float* bias, int N, int Nw, int I, int O, int H, int W, int ksize,
                                int act, void* y_f16, r3dp_stream_t stream) {
    return conv_res_impl(x_f16, wp_f16, bias, N, Nw, I, O, H, W, ksize, act, nullptr, y_f16, 1, stream);
}
extern "C" int r3dp_sr_tc_conv(const void* x_f16, const void* wp_f16, const float* bias, int N, int Nw, int I, int O, int H, int W, int ksize,
                               int act, void* y_f16, r3dp_stream_t stream) {
    return r3dp_sr_tc_conv_res(x_f16, wp_f16, bias, N, Nw, I, O, H, W, ksize, act, nullptr, y_f16, stream);
}

// SynthesisBlockNoUp tail (superresolution.py:159-258): conv3x3 (modulated, up == 1) + bias/lrelu -> y, and img_out = img_prev (SAME resolution)
// + ToRGB(y) + brgb.
extern "C" int r3dp_sr_tc_layer_torgb_noup(const void* x_f16, const void* wp_f16, const float* bias, const float* wrgb, const float* brgb,
                                           const float* img_prev, int N, int Nw, int I, int O, int H, int W, void* y_f16, float* img_out,
                                           r3dp_stream_t stream) {
    R3DP_REQUIRE(x_f16 && wp_f16 && bias && wrgb && brgb && y_f16 && img_out, "sr_tc_layer_torgb_noup: null pointer");
    R3DP_REQUIRE(N > 0 && (Nw == N || Nw == 1) && W % BM == 0 && O % BN == 0 && O <= 256,
                 "sr_tc_layer_torgb_noup: bad shape (needs N > 0, Nw == N or Nw == 1, W %% 128 == 0, Cout 128 or 256; got N=%d, Nw=%d, Cout=%d, W=%d)", N, Nw, O, W);
    const int Ip = (I + 63) / 64 * 64;
    Conv2Args a = {};
    Taps t = {};
    t.n = 9;
    for (int i = 0; i < 9; ++i) { t.dy[i] = i / 3 - 1; t.dx[i] = i % 3 - 1; t.widx[i] = i; }
    a.n_phases = 1;
    fill_taps2(a.ph[0].taps, t);
    a.ph[0].rows = H;
    a.mode = kActRgb; a.out = reinterpret_cast<__half*>(y_f16); a.out_H = H; a.out_W = W; a.out_C = O; a.oy_mul = a.ox_mul = 1;
    a.bias = bias; a.wrgb = wrgb; a.brgb = brgb; a.img_prev = img_prev; a.img_out = img_out; a.img_H = H; a.img_W = W; a.skip_same_res = 1;
    return run_conv2(x_f16, N, H, W, Ip, wp_f16, Nw, O, a, H, as_stream(stream));
}

// out[n,y,x,:] = [ xa[n,y,x,0:Ca] * alpha[n,y,x] , xb[n,y,x,0:Cb] * (1 - alpha[n,y,x]) ]   (sr_with_ref.py:111,122: alpha-cat fusion), fp16 NHWC
__global__ void alpha_cat_kernel(const __half* __restrict__ xa, int Ca, int sa, const __half* __restrict__ xb, int Cb, int sb,
                                 long long hw_b, const float* __restrict__ alpha, long long npix, __half* __restrict__ out) {
    const int cv = (Ca + Cb) / 8;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= npix * cv) return;
    const long long pix = idx / cv; const int c8 = (int)(idx - pix * cv);
    const float al = alpha[pix];
    const bool first = c8 * 8 < Ca;
    const long long pb = hw_b > 0 ? pix % hw_b : pix;                    // xb holds one frame shared by the batch
    const uint4 raw = __ldg(reinterpret_cast<const uint4*>(first ? xa + pix * sa + c8 * 8 : xb + pb * sb + (c8 * 8 - Ca)));
    const float m = first ? al : 1.0f - al;
    const __half2* h = reinterpret_cast<const __half2*>(&raw);
    uint4 pk; __half2* ph = reinterpret_cast<__half2*>(&pk);
#pragma unroll
    for (int j = 0; j < 4; ++j) { const float2 f = __half22float2(h[j]); ph[j] = __floats2half2_rn(f.x * m, f.y * m); }
    *reinterpret_cast<uint4*>(out + idx * 8) = pk;
}
extern "C" int r3dp_sr_alpha_cat_ex(const void* xa_f16, int Ca, int stride_a, const void* xb_f16, int Cb, int stride_b, int xb_shared,
                                    const float* alpha, int N, int H, int W, void* out_f16, r3dp_stream_t stream) {
    R3DP_REQUIRE(xa_f16 && xb_f16 && alpha && out_f16, "sr_alpha_cat: null pointer");
    R3DP_REQUIRE(N > 0 && H > 0 && W > 0 && Ca % 8 == 0 && Cb % 8 == 0 && stride_a >= Ca && stride_b >= Cb && stride_a % 8 == 0 && stride_b % 8 == 0,
                 "sr_alpha_cat: bad shape");
    const long long npix = (long long)N * H * W, total = npix * ((Ca + Cb) / 8);
    alpha_cat_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(reinterpret_cast<const __half*>(xa_f16), Ca, stride_a,
        reinterpret_cast<const __half*>(xb_f16), Cb, stride_b, xb_shared ? (long long)H * W : 0ll, alpha, npix, reinterpret_cast<__half*>(out_f16));
    R3DP_LAUNCH_CHECK();
    count_launches(1);
    return 0;
}
extern "C" int r3dp_sr_alpha_cat(const void* xa_f16, int Ca, int stride_a, const void* xb_f16, int Cb, int stride_b, const float* alpha, int N,
                                 int H, int W, void* out_f16, r3dp_stream_t stream) {
    return r3dp_sr_alpha_cat_ex(xa_f16, Ca, stride_a, xb_f16, Cb, stride_b, 0, alpha, N, H, W, out_f16, stream);
}

// out = a * alpha + b * (1 - alpha), fp32 NCHW [N,C,H,W] with alpha [N,1,H,W]  (sr_with_ref.py:110,132)
__global__ void blend_kernel(const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ alpha, int C, long long hw,
                             long long total, float* __restrict__ out) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const long long n = idx / (C * hw), p = idx % hw;
    const float al = alpha[n * hw + p];
    out[idx] = a[idx] * al + b[idx] * (1.0f - al);
}
extern "C" int r3dp_sr_blend(const float* a, const float* b, const float* alpha, int N, int C, int H, int W, float* out, r3dp_stream_t stream) {
    R3DP_REQUIRE(a && b && alpha && out && N > 0 && C > 0 && H > 0 && W > 0, "sr_blend: bad arguments");
    const long long hw = (long long)H * W, total = (long long)N * C * hw;
    blend_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(a, b, alpha, C, hw, total, out);
    R3DP_LAUNCH_CHECK();
    count_launches(1);
    return 0;
}

// person_occlusion = clamp(torso_occlusion + (w > threshold ? 1 : w), 0, 1)   (sr_with_ref.py:126-131)
__global__ void person_occlusion_kernel(const float* __restrict__ w, const float* __restrict__ torso, float thr, long long total, float* __restrict__ out) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const float h = w[idx] > thr ? 1.0f : w[idx];
    out[idx] = fminf(fmaxf(torso[idx] + h, 0.f), 1.f);
}
extern "C" int r3dp_sr_person_occlusion(const float* head_alpha, const float* torso_occlusion, float threshold, int N, int H, int W, float* out,
                                        r3dp_stream_t stream) {
    R3DP_REQUIRE(head_alpha && torso_occlusion && out && N > 0 && H > 0 && W > 0, "sr_person_occlusion: bad arguments");
    const long long total = (long long)N * H * W;
    person_occlusion_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(head_alpha, torso_occlusion, threshold, total, out);
    R3DP_LAUNCH_CHECK();
    count_launches(1);
    return 0;
}

// F.interpolate(scale 1/2, bilinear, align_corners=False, antialias=True) (sr_with_ref.py:79-82): separable triangle filter of support 2,
// taps [1,3,3,1]/8 in the interior, clipped and renormalised at the borders ([3,3,1]/7, [1,3,3]/7).  x [N*C][2h][2w] -> y [N*C][h][w], fp32.
__global__ void aa_down2_kernel(const float* __restrict__ x, int NC, int h, int w, float* __restrict__ y) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)NC * h * w) return;
    const int ox = (int)(idx % w), oy = (int)((idx / w) % h); const long long nc = idx / ((long long)w * h);
    const int H2 = 2 * h, W2 = 2 * w;
    const float* p = x + nc * H2 * W2;
    const float k4[4] = {0.25f, 0.75f, 0.75f, 0.25f};
    float wy[4], wx[4], sy = 0.f, sx = 0.f;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const int yy = 2 * oy - 1 + t, xx = 2 * ox - 1 + t;
        wy[t] = (yy >= 0 && yy < H2) ? k4[t] : 0.f; wx[t] = (xx >= 0 && xx < W2) ? k4[t] : 0.f;
        sy += wy[t]; sx += wx[t];
    }
    float acc = 0.f;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        if (wy[u] == 0.f) continue;
        const int yy = 2 * oy - 1 + u;
        float row = 0.f;
#pragma unroll
        for (int v = 0; v < 4; ++v) { if (wx[v] != 0.f) row = fmaf(wx[v] / sx, p[(size_t)yy * W2 + 2 * ox - 1 + v], row); }
        acc = fmaf(wy[u] / sy, row, acc);
    }
    y[idx] = acc;
}
extern "C" int r3dp_sr_resize_aa_down2(const float* x, int N, int C, int h_out, int w_out, float* y, r3dp_stream_t stream) {
    R3DP_REQUIRE(x && y && N > 0 && C > 0 && h_out > 0 && w_out > 0, "sr_resize_aa_down2: bad arguments");
    const long long total = (long long)N * C * h_out * w_out;
    aa_down2_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(x, N * C, h_out, w_out, y);
    R3DP_LAUNCH_CHECK();
    count_launches(1);
    return 0;
}

// out[n,y,x,0:C] = xa * alpha + xb * (1 - alpha)  (htbsr_head_weight_fuse_mode v1, sr_with_ref.py:98: plain alpha blend of the head and torso features), fp16 NHWC
__global__ void alpha_mix_kernel(const __half* __restrict__ xa, int sa, const __half* __restrict__ xb, int sb, const float* __restrict__ alpha, int C,
                                 long long npix, __half* __restrict__ out) {
    const int cv = C / 8;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= npix * cv) return;
    const long long pix = idx / cv; const int c8 = (int)(idx - pix * cv);
    const float al = alpha[pix];
    const uint4 ra = __ldg(reinterpret_cast<const uint4*>(xa + pix * sa + c8 * 8)), rb = __ldg(reinterpret_cast<const uint4*>(xb + pix * sb + c8 * 8));
    const __half2* ha = reinterpret_cast<const __half2*>(&ra); const __half2* hb = reinterpret_cast<const __half2*>(&rb);
    uint4 pk; __half2* ph = reinterpret_cast<__half2*>(&pk);
#pragma unroll
    for (int j = 0; j < 4; ++j) { const float2 a = __half22float2(ha[j]), b = __half22float2(hb[j]); ph[j] = __floats2half2_rn(a.x * al + b.x * (1.0f - al), a.y * al + b.y * (1.0f - al)); }
    *reinterpret_cast<uint4*>(out + idx * 8) = pk;
}
extern "C" int r3dp_sr_alpha_mix(const void* xa_f16, int stride_a, const void* xb_f16, int stride_b, const float* alpha, int C, int N, int H, int W,
                                 void* out_f16, r3dp_stream_t stream) {
    R3DP_REQUIRE(xa_f16 && xb_f16 && alpha && out_f16 && N > 0 && H > 0 && W > 0 && C > 0 && C % 8 == 0 && stride_a >= C && stride_b >= C &&
                 stride_a % 8 == 0 && stride_b % 8 == 0, "sr_alpha_mix: bad arguments");
    const long long npix = (long long)N * H * W, total = npix * (C / 8);
    alpha_mix_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(reinterpret_cast<const __half*>(xa_f16), stride_a,
        reinterpret_cast<const __half*>(xb_f16), stride_b, alpha, C, npix, reinterpret_cast<__half*>(out_f16));
    R3DP_LAUNCH_CHECK();
    count_launches(1);
    return 0;
}

// out[n,0,y,x] = min(sigmoid(logit), cap[n,0,y,x]) with logit = channel 0 of an NHWC fp16 tensor (+ its lo half lo_off channels further when lo_off > 0):
// the tail of head_torso_alpha_predictor and the `alpha[alpha > weights] = weights` cap of fuse mode v3 (sr_with_ref.py:130-132)
__global__ void alpha_gate_kernel(const __half* __restrict__ y, int stride, int lo_off, const float* __restrict__ cap, long long npix, float* __restrict__ out) {
    const long long pix = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (pix >= npix) return;
    float v = __half2float(y[pix * stride]);
    if (lo_off > 0) v += __half2float(y[pix * stride + lo_off]);
    const float sg = 1.0f / (1.0f + expf(-v));
    out[pix] = fminf(sg, cap[pix]);
}
extern "C" int r3dp_sr_alpha_gate(const void* logits_f16, int stride, int lo_off, const float* cap, int N, int H, int W, float* out, r3dp_stream_t stream) {
    R3DP_REQUIRE(logits_f16 && cap && out && N > 0 && H > 0 && W > 0, "sr_alpha_gate: bad arguments");
    R3DP_REQUIRE(stride > 0 && lo_off >= 0 && lo_off < stride, "sr_alpha_gate: needs 0 <= lo_off < stride (got lo_off=%d, stride=%d)", lo_off, stride);
    const long long npix = (long long)N * H * W;
    alpha_gate_kernel<<<(unsigned)((npix + 255) / 256), 256, 0, as_stream(stream)>>>(reinterpret_cast<const __half*>(logits_f16), stride, lo_off, cap, npix, out);
    R3DP_LAUNCH_CHECK();
    count_launches(1);
    return 0;
}

// Timing of the tensor-core conv launches: r3dp_sr_tc_prof(1) starts recording a CUDA-event pair around every conv_tc3 launch,
// r3dp_sr_tc_prof(0) stops; r3dp_sr_tc_prof_read synchronises the recorded events and returns their summed duration and count.
extern "C" int r3dp_sr_tc_prof(int enable) { g_prof.on = enable != 0; if (enable) g_prof.used = 0; return 0; }
extern "C" int r3dp_sr_tc_prof_read(float* total_ms, int* launches) {
    float sum = 0.f;
    for (size_t i = 0; i + 1 < g_prof.used; i += 2) {
        R3DP_CUDA(cudaEventSynchronize(g_prof.ev[i + 1]));
        float ms = 0.f;
        R3DP_CUDA(cudaEventElapsedTime(&ms, g_prof.ev[i], g_prof.ev[i + 1]));
        sum += ms;
    }
    if (total_ms) *total_ms = sum;
    if (launches) *launches = (int)(g_prof.used / 2);
    return 0;
}

// debug builds (-DR3DP_TC_DEBUG_TIMING=1): device buffer of 32 x 24 uint64; the i-th conv_tc3 launch after this call adds clock sums to row i: [0,8) MMA warp, [8,16) epilogue warp 2 (columns 0-63), [16,24) epilogue warp 6 (columns 64-127)
extern "C" int r3dp_sr_tc_debug_buffer(void* buf) { g_debug_buf = reinterpret_cast<unsigned long long*>(buf); g_debug_launch = 0; return 0; }
