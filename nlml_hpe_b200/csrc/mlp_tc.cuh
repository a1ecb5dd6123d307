// Tensor-core linear layer for sm_100a: y = act((A W^T) * inv_scale + b) with FP32-grade accuracy from
// FP16 tensor-core passes.
//
// The reference computes every Linear in FP32 (torch.nn.Linear on CPU, NLML_HPE_Model_Builder.py:33-53,
// 76-92) and the parity budget is 1e-3 degrees, which no single-pass 16-bit or TF32 product meets
// (SURVEY.md section 7).  Each FP32 operand is therefore carried as two FP16 planes, v = hi + lo with
// hi = fp16(v), lo = fp16(v - hi), and one algorithmic MAC becomes three tcgen05 MMAs into the same FP32
// TMEM accumulator:  hi*hi + lo*hi + hi*lo  (the lo*lo term is below FP32 resolution).
//
// Kernel anatomy (one CTA per SM, persistent over output tiles, 320 threads):
//   warp 0      TMA producer: cp.async.bulk.tensor 2D loads of the four operand planes (A_hi, A_lo, W_hi,
//               W_lo), 128-byte swizzle, into a ring of shared-memory stages guarded by full/empty mbarriers
//   warp 1      MMA issuer: allocates TMEM, one elected lane issues tcgen05.mma.kind::f16 (M=128, N=BN,
//               K=16) x 3 passes x 4 k-steps per stage, tcgen05.commit releases the stage / publishes the tile
//   warps 2-9   promotion + epilogue: tcgen05.ld every k-block's partial 128 x BN FP32 tile (double-buffered in
//               TMEM so the next k-block's MMAs overlap) and add it into FP32 registers with round-to-nearest;
//               after the last k-block scale + bias + activation, then either re-split into FP16 hi/lo planes
//               for the next tensor-core layer or store FP32 for the CUDA-core tail
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace nlml {
namespace tc {

constexpr int BM = 128;   // samples per tile (TMEM lanes)
constexpr int BK = 64;    // fp16 elements per k-block = one 128-byte swizzle row
constexpr int UMMA_K = 16;
constexpr int kEpilogueWarps = 8;
// Three warp groups: group 0 = TMA warp, MMA warp (+ two idle warps), groups 1 and 2 = the eight promotion / epilogue
// warps.  With ten warps on a uniform budget one SM sub-partition holds three of them and every thread is capped at 168
// registers (the epilogue keeps 128 FP32 partial sums per thread and spilled); setmaxnreg hands group 0's registers over.
constexpr int kFirstEpilogueWarp = 4;
constexpr int kThreads = 32 * (kFirstEpilogueWarp + kEpilogueWarps);
constexpr int kProducerRegs = 40, kEpilogueRegs = 232;   // (40 + 232 + 232) * 32 <= 16384 registers per sub-partition

// fused neck epilogue (BN = 64 only): W5 [9][64], B5 [12], head rows (w0,w1,w2,b) [3][128] float4, latent exchange [2][9][128]
constexpr int kNeckLatent = 9, kNeckHeadW = 128;
constexpr int kStoreStageBytes = 32 * 128;   // per epilogue warp: its 32 rows x 128 B of one plane (store_planes_staged)
constexpr int kNeckSmemFloats = kNeckLatent * 64 + 12 + 3 * kNeckHeadW * 4 + 2 * kNeckLatent * BM;

template <int BN>
struct Cfg {
    static constexpr int STAGES = BN == 256 ? 2 : 3;
    static constexpr int A_BYTES = BM * BK * 2;           // one plane of the A tile
    static constexpr int W_BYTES = BN * BK * 2;           // one plane of the W tile
    static constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * W_BYTES;
    static constexpr int TMEM_COLS = 2 * BN;              // two accumulator buffers
    static constexpr size_t SMEM_BYTES = 1024 /*align slack*/ + (size_t)STAGES * STAGE_BYTES + 256 /*barriers*/ +
                                         (BN == 64 ? 2 * kEpilogueWarps * (BN / 2) * 4 : 0) /*bias, dot weights*/ + 2 * BM * 4 /*dot exchange*/ +
                                         (BN == 64 ? kNeckSmemFloats * 4 : 0) /*fused neck epilogue*/ +
                                         kEpilogueWarps * kStoreStageBytes /*store staging (TMA)*/;
};

constexpr int kMaxProblems = 3;   // the three heads ride one launch

// k-blocks summed in the accumulator that starts at k-block kb (see LinearTcArgs::group / lead_kb)
__device__ __forceinline__ int group_len(int kb, int group, int lead_kb) { return (kb < lead_kb && group < 2) ? 2 : group; }

struct LinearTcArgs {
    long long N;        // rows (samples)
    int out, Kp;        // output features (multiple of BN), padded reduction length (multiple of BK)
    int y_tma;          // the FP16 output planes leave through TMA (maps.y_hi / y_lo valid; 128- and 256-wide tiles)
    int act;            // 0 none, 1 relu, 2 tanh
    int problems;       // independent problems of identical shape (1 for the encoder, 3 for the heads)
    int group;          // k-blocks accumulated in TMEM before a partial tile is promoted to FP32 registers
    int lead_kb;        // the first lead_kb k-blocks of every tile are summed in PAIRS whatever `group` says: while the epilogue
                        // warps are still converting and storing the previous tile (~5 k cycles) the MMA warp can run four
                        // k-blocks (6.1 k cycles) ahead on the two accumulators instead of two
    float inv_scale[kMaxProblems];    // 1 / (power-of-two scale folded into the W planes)
    const float* bias[kMaxProblems];  // [out]
    __half* Yhi[kMaxProblems];        // [N][ldy] or null
    __half* Ylo[kMaxProblems];
    float* Yf32[kMaxProblems];        // [N][ldy] or null
    long long ldy;
    // fused final layer (out == BN only): Ydot[row*ldd + z] = dot_b[z] + sum_j act(y[row][j]) * dot_w[z][j]
    const float* dot_w[kMaxProblems];   // [out] or null
    const float* dot_b[kMaxProblems];   // [1]
    float* Ydot;
    int ldd;
    // fused neck (out == BN == 64, act = tanh): latent = B5 + W5 . y (64 -> 9), LAT[row][9] (optional), then for each
    // head h the first hidden layer relu(Bh + Wh . latent[3h..3h+2]) (3 -> 128) written as FP16 hi/lo planes
    int neck;
    const float *neck_w5, *neck_b5;       // [9][64], [9]
    const float* neck_wh[3];              // [128][3]
    const float* neck_bh[3];              // [128]
    float* neck_lat;                      // [N][9] or null
    __half* neck_hi[3];                   // [N][128]
    __half* neck_lo[3];
#ifdef NLML_MLP_TIMING
    float* timing;   // development build only (scripts/time_mlp_tc.py): [CTA][epilogue warp][4] cycles per tile
#endif
};

// operand maps of up to three problems: A_hi, A_lo, W_hi, W_lo each
struct TcMaps {
    CUtensorMap a_hi[kMaxProblems], a_lo[kMaxProblems], w_hi[kMaxProblems], w_lo[kMaxProblems];
    CUtensorMap y_hi[kMaxProblems], y_lo[kMaxProblems];   // output planes, 32-row x 64-column boxes (LinearTcArgs::y_tma)
};

// ---- PTX wrappers -----------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
    } while (!done);
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, int c_inner, int c_outer, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(c_inner), "r"(c_outer), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void tma_load_2d_mcast(void* smem_dst, const CUtensorMap* map, int c_inner, int c_outer, uint64_t* bar,
                                                  uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%2, %3}], [%4], %5;"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(c_inner), "r"(c_outer), "r"(smem_u32(bar)), "h"(cta_mask)
        : "memory");
}
__device__ __forceinline__ void umma_commit_mcast(uint64_t* bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(cta_mask) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// The MMA warp runs its loop CONVERGED with warp-uniform values and lets the elected lane issue (elect.sync inside the asm
// block): descriptor arithmetic then stays in the uniform datapath.  A plain `if (lane == 0)` issue wraps every
// tcgen05.mma in a register->uniform-register broadcast loop (~100 cycles per MMA), which made the short-K / narrow layers
// issue-bound (their MMAs execute in 32-64 cycles).
__device__ __forceinline__ void umma_f16_elect(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, e;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit_elect(uint64_t* bar) {
    asm volatile(
        "{\n\t.reg .pred e;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
        ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void umma_commit_mcast_elect(uint64_t* bar, uint16_t cta_mask) {
    asm volatile(
        "{\n\t.reg .pred e;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n\t}"
        ::"r"(smem_u32(bar)), "h"(cta_mask) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
// 256-bit global store (sm_100): one full 32-byte sector per lane
__device__ __forceinline__ void st_global_v8(void* ptr, const uint32_t (&v)[8]) {
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(ptr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]),
                 "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}
__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major operand tile, 128-byte swizzle, rows 128 B apart, 8-row groups 1024 B apart (cute::UMMA::SmemDescriptor)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);  // start address, bits [0,14)
    d |= (uint64_t)1 << 16;                        // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;              // stride byte offset: 8 rows x 128 B
    d |= (uint64_t)1 << 46;                        // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;                        // SWIZZLE_128B
    return d;
}
// kind::f16 instruction descriptor: D=F32, A=B=F16, both K-major (cute::UMMA::InstrDescriptor)
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N) {
    return (1u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// The activation is a template parameter of everything that runs per element: with a run-time `act` every one of a
// thread's 128 outputs carried two uniform branches (and the inlined tanh body), ~13 k cycles per tile in which the
// epilogue warps promoted nothing and the tensor pipe of the long layers idled (29 % of encoder.0's time).
// ReLU that PROPAGATES NaN, as torch.relu does (fmaxf returns the other operand).  It matters for range errors: an
// activation beyond FP16's range becomes inf in its hi plane, the next layer's products turn it into NaN, and an
// fmaxf-ReLU would quietly map that NaN to 0 -- finite-but-wrong angles.  max.NaN costs the same single instruction.
__device__ __forceinline__ float relu_nan(float v) {
    float r;
    asm("max.NaN.f32 %0, %1, 0f00000000;" : "=f"(r) : "f"(v));
    return r;
}
template <int ACT>
__device__ __forceinline__ float act_fixed(float v) {
    if (ACT == 1) return relu_nan(v);
    if (ACT == 2) return tanhf(v);
    return v;
}
// runs BODY with `ACT` a compile-time constant equal to the run-time `act`
#define NLML_ACT_DISPATCH(act, ...)                              \
    if ((act) == 1) { constexpr int ACT = 1; __VA_ARGS__ }       \
    else if ((act) == 2) { constexpr int ACT = 2; __VA_ARGS__ }  \
    else { constexpr int ACT = 0; __VA_ARGS__ }

// Two FP32 values -> packed FP16 (hi, lo) words, value 0 in the low half.  Packed conversions (one F2FP per pair, the
// way back through HADD2.F32) instead of six scalar F2F per pair: the scalar form runs at a quarter of the ALU rate
// and made the epilogues of the short-K layers conversion-bound (ncu: F2F 10 % of the samples of the heads' layers).
// Same roundings (cvt.rn), bit-identical planes.
__device__ __forceinline__ void split_pair(float v0, float v1, uint32_t& hi, uint32_t& lo) {
    const __half2 h = __floats2half2_rn(v0, v1);
    const float2 hf = __half22float2(h);
    const __half2 l = __floats2half2_rn(v0 - hf.x, v1 - hf.y);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}

// One thread's row of a finished tile: y = act(sum * inv_scale + bias), written as FP32 and/or as FP16 hi/lo planes.
// `yf`, `dh`, `dl` point at this row's first column of the warp's column slice (null = not wanted).
// four consecutive bias values: from the warp's shared-memory slice (64-wide tiles) or straight from global memory
// through L1 (every lane reads the same address: one broadcast transaction; the 512 bytes stay L1-resident because
// nothing else in these kernels allocates in L1 -- TMA, tcgen05 and the write-through stores all bypass it)
template <bool SMEM>
__device__ __forceinline__ float4 bias4(const float* p) {
    if (SMEM) return *reinterpret_cast<const float4*>(p);
    return __ldg(reinterpret_cast<const float4*>(p));
}

template <int ACT, int HALF, bool BIAS_SMEM>
__device__ __forceinline__ void store_row(const float (&sum)[HALF], float inv_scale, const float* bias_s, float* yf, __half* dh,
                                          __half* dl) {
#pragma unroll
    for (int c0 = 0; c0 < HALF; c0 += 32) {
        float y[32];
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
            const float4 b = bias4<BIAS_SMEM>(bias_s + c0 + j);
            y[j] = act_fixed<ACT>(fmaf(sum[c0 + j], inv_scale, b.x));
            y[j + 1] = act_fixed<ACT>(fmaf(sum[c0 + j + 1], inv_scale, b.y));
            y[j + 2] = act_fixed<ACT>(fmaf(sum[c0 + j + 2], inv_scale, b.z));
            y[j + 3] = act_fixed<ACT>(fmaf(sum[c0 + j + 3], inv_scale, b.w));
        }
        if (yf) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                uint32_t w[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) w[e] = __float_as_uint(y[8 * j + e]);
                st_global_v8(yf + c0 + 8 * j, w);
            }
        }
        if (dh) {
            uint32_t hi[16], lo[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) split_pair(y[2 * j], y[2 * j + 1], hi[j], lo[j]);
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                uint32_t wh[8], wl[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) { wh[e] = hi[8 * j + e]; wl[e] = lo[8 * j + e]; }
                st_global_v8(dh + c0 + 16 * j, wh);
                st_global_v8(dl + c0 + 16 * j, wl);
            }
        }
    }
}


// The same outputs as store_row's FP16 planes, leaving through TMA.  A thread owns one ROW of the tile (that is how
// tcgen05.ld hands the accumulator over), so direct stores put every lane of a warp-wide store in a different line:
// 32 packets of 32 B per instruction, ~6 k cycles per 128 x 256 tile during which the warp promotes nothing, and a
// transpose through shared memory read back by the warp pays the shared-memory bandwidth twice on the warp's own
// time (measured 4.4 k cycles).  Here each warp writes its 32 rows x 64 columns of one plane into a 4 KB buffer in
// the 128-byte-swizzle layout (chunk c of row r at slot c ^ (r & 7): conflict-free) and one lane hands the box to
// TMA, which drains it asynchronously while the warp converts the next 64 columns; rows past N are clipped by the
// tensor map.  `bias` points at the warp's first column in GLOBAL memory; (col0, row0) is the box origin.
// Issued by the whole converged warp with the elected lane predicated inside the asm block: an `if (lane == 0)` around
// these makes nvcc wrap the uniform-datapath instruction in a divergence loop (1.1 k cycles per tile for four stores).
// elect.sync picks the same leader for the same member mask, so the bulk groups are committed and awaited by one thread.
__device__ __forceinline__ void tma_store_2d_elect(const CUtensorMap* map, const void* smem_src, int c_inner, int c_outer) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "elect.sync _|p, 0xffffffff;\n"
        "@p cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];\n"
        "@p cp.async.bulk.commit_group;\n"
        "}"
        ::"l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(smem_src)), "r"(c_inner), "r"(c_outer) : "memory");
}
template <int PENDING>
__device__ __forceinline__ void tma_store_wait_read_elect() {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "elect.sync _|p, 0xffffffff;\n"
        "@p cp.async.bulk.wait_group.read %0;\n"
        "}" ::"n"(PENDING) : "memory");
}
__device__ __forceinline__ void tma_store_wait_all_elect() {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "elect.sync _|p, 0xffffffff;\n"
        "@p cp.async.bulk.wait_group 0;\n"
        "}" ::: "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// one 32-row x 64-column box of a plane: this thread's 32 words (64 halves of its row) -> swizzled buffer -> TMA
__device__ __forceinline__ void stage_box_tma(uint4* buf, const uint32_t (&w)[32], const CUtensorMap* map, int col, int row0,
                                              int lane) {
    tma_store_wait_read_elect<0>();   // the previous box has left the buffer
    __syncwarp();
#pragma unroll
    for (int c = 0; c < 8; ++c) buf[lane * 8 + (c ^ (lane & 7))] = make_uint4(w[4 * c], w[4 * c + 1], w[4 * c + 2], w[4 * c + 3]);
    fence_async_smem();
    __syncwarp();
    tma_store_2d_elect(map, buf, col, row0);
}

template <int ACT, int HALF>
__device__ __forceinline__ void store_planes_tma(const float (&sum)[HALF], float inv_scale, const float* bias, uint4* buf,
                                                 const CUtensorMap* map_hi, const CUtensorMap* map_lo, int col0, int row0,
                                                 int lane) {
    static_assert(HALF % 64 == 0, "64 columns of a plane per box");
#pragma unroll
    for (int c0 = 0; c0 < HALF; c0 += 64) {
        uint32_t hi[32], lo[32];
#pragma unroll
        for (int j = 0; j < 64; j += 4) {
            const float4 b = bias4<false>(bias + c0 + j);
            const float y0 = act_fixed<ACT>(fmaf(sum[c0 + j], inv_scale, b.x)), y1 = act_fixed<ACT>(fmaf(sum[c0 + j + 1], inv_scale, b.y));
            const float y2 = act_fixed<ACT>(fmaf(sum[c0 + j + 2], inv_scale, b.z)), y3 = act_fixed<ACT>(fmaf(sum[c0 + j + 3], inv_scale, b.w));
            split_pair(y0, y1, hi[j / 2], lo[j / 2]);
            split_pair(y2, y3, hi[j / 2 + 1], lo[j / 2 + 1]);
        }
        stage_box_tma(buf, hi, map_hi, col0 + c0, row0, lane);
        stage_box_tma(buf, lo, map_lo, col0 + c0, row0, lane);
    }
}

// CL = CTAs per cluster (1 or 2).  With CL = 2 the two CTAs of a cluster work on M-tiles (2p, 2p+1) of the same
// N-tile: each loads its own A planes and HALF of the W tile, multicast into both CTAs' shared memory, which cuts
// the L2->SMEM operand traffic per MMA by a third (the wide layers are L2-bandwidth bound at 128x256 tiles).
template <int BN, int CL>
__global__ void __launch_bounds__(kThreads, 1)
linear_tc_kernel(const __grid_constant__ TcMaps maps, const __grid_constant__ LinearTcArgs a) {
    using C = Cfg<BN>;
    static_assert(CL == 1 || CL == 2, "cluster size");
    const uint32_t crank = CL > 1 ? cluster_ctarank() : 0;
    constexpr uint16_t kMask = (uint16_t)((1u << CL) - 1);
    constexpr int HALF = BN / 2;   // columns owned by one epilogue warp
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment by pointer arithmetic on the __shared__ array (a round trip through uintptr_t makes the compiler
    // lose the address space: the epilogue's bias reads became generic LD.E instead of LDS)
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* stage_base = smem;
    constexpr size_t kStoreStage = (size_t)kEpilogueWarps * kStoreStageBytes;                    // 1024-byte aligned (swizzle atoms)
    uint4* stage_all = reinterpret_cast<uint4*>(smem + (size_t)C::STAGES * C::STAGE_BYTES);     // [warp][32][8]
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)C::STAGES * C::STAGE_BYTES + kStoreStage);
    uint64_t* full = bars;                    // [STAGES]  operand stage landed
    uint64_t* empty = bars + C::STAGES;       // [STAGES]  operand stage consumed by the MMAs
    uint64_t* tfull = bars + 2 * C::STAGES;   // [2]  partial accumulator of one k-block complete
    uint64_t* tempty = tfull + 2;             // [2]  partial accumulator drained into registers
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
    float* bias_all = reinterpret_cast<float*>(smem + (size_t)C::STAGES * C::STAGE_BYTES + kStoreStage + 256);   // [warp][HALF], private per epilogue warp
    constexpr bool kBiasSmem = BN == 64;   // the wider tiles read the bias through L1 and use the space for store staging
    float* dotw_all = bias_all + (kBiasSmem ? kEpilogueWarps * HALF : 0);                          // [warp][HALF]  (BN == 64 only)
    float* dot_xch = dotw_all + (kBiasSmem ? kEpilogueWarps * HALF : 0);                           // [2][BM] partial dots of the upper column half
    float* neck_w5s = dot_xch + 2 * BM;                                   // [9][64]          (BN == 64 only, see Cfg)
    float* neck_b5s = neck_w5s + kNeckLatent * 64;                        // [12]
    float4* neck_whs = reinterpret_cast<float4*>(neck_b5s + 12);          // [3][128] (w0, w1, w2, bias)
    float* neck_xch = reinterpret_cast<float*>(neck_whs + 3 * kNeckHeadW);   // [2 halves][9][BM]

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;   // provably warp-uniform
    const int num_kb = a.Kp / BK;
    const int tiles_n = a.out / BN;
    const long long tiles_m = ((a.N + BM - 1) / BM + CL - 1) / CL;   // M-tile groups: CL consecutive M-tiles per cluster
    const long long tiles_per_problem = tiles_m * tiles_n;
    const long long num_tiles = tiles_per_problem * a.problems;    // work items per cluster
    const long long first = blockIdx.x / CL, step = gridDim.x / CL;

    if (warp == 0 && lane == 0) {
        for (int z = 0; z < a.problems; ++z) {
            prefetch_tmap(&maps.a_hi[z]); prefetch_tmap(&maps.a_lo[z]); prefetch_tmap(&maps.w_hi[z]); prefetch_tmap(&maps.w_lo[z]);
        }
        for (int s = 0; s < C::STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], CL); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], kEpilogueWarps); }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, C::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    if (CL > 1) cluster_sync_all();   // the peer's barriers must exist before anything is multicast into them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if constexpr (BN == 64) {
        if (a.neck && warp >= kFirstEpilogueWarp) {   // the epilogue warps stage the narrow layers' constants once per CTA
            const int e = threadIdx.x - 32 * kFirstEpilogueWarp, ne = 32 * kEpilogueWarps;
            for (int i = e; i < kNeckLatent * 64; i += ne) neck_w5s[i] = __ldg(a.neck_w5 + i);
            for (int i = e; i < kNeckLatent; i += ne) neck_b5s[i] = __ldg(a.neck_b5 + i);
            for (int i = e; i < 3 * kNeckHeadW; i += ne) {
                const int h = i / kNeckHeadW, j = i % kNeckHeadW;
                const float* w = a.neck_wh[h] + 3 * j;
                neck_whs[i] = make_float4(__ldg(w), __ldg(w + 1), __ldg(w + 2), __ldg(a.neck_bh[h] + j));
            }
            asm volatile("bar.sync 5, %0;" ::"r"(32 * kEpilogueWarps) : "memory");
        }
    }

    if (warp == 0) {
        // ===== TMA producer =====
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kProducerRegs));   // register hand-over, see kThreads
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (long long t = first; t < num_tiles; t += step) {
                const int z = (int)(t / tiles_per_problem);
                const long long tt = t % tiles_per_problem;
                const int m0 = (int)((tt / tiles_n) * CL + crank) * BM, n0 = (int)(tt % tiles_n) * BN;
                for (int kb = 0; kb < num_kb; ++kb) {
                    mbar_wait(&empty[stage], phase ^ 1);   // CL > 1: every CTA of the cluster has consumed this stage
                    uint8_t* st = stage_base + (size_t)stage * C::STAGE_BYTES;
                    mbar_expect_tx(&full[stage], C::STAGE_BYTES);
                    tma_load_2d(st, &maps.a_hi[z], kb * BK, m0, &full[stage]);
                    tma_load_2d(st + C::A_BYTES, &maps.a_lo[z], kb * BK, m0, &full[stage]);
                    if (CL == 1) {
                        tma_load_2d(st + 2 * C::A_BYTES, &maps.w_hi[z], kb * BK, n0, &full[stage]);
                        tma_load_2d(st + 2 * C::A_BYTES + C::W_BYTES, &maps.w_lo[z], kb * BK, n0, &full[stage]);
                    } else {
                        // this CTA's slice of the W tile (BN/CL rows), delivered to every CTA of the cluster
                        const int rows = BN / CL, off = (int)crank * rows * (BK * 2);
                        tma_load_2d_mcast(st + 2 * C::A_BYTES + off, &maps.w_hi[z], kb * BK, n0 + (int)crank * rows, &full[stage], kMask);
                        tma_load_2d_mcast(st + 2 * C::A_BYTES + C::W_BYTES + off, &maps.w_lo[z], kb * BK, n0 + (int)crank * rows, &full[stage], kMask);
                    }
                    if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kProducerRegs));   // register hand-over, see kThreads
        // The tensor core's FP32 accumulate truncates instead of rounding, which biases long accumulation
        // chains (measured: 3.6e-3 deg at the output when all K/16*3 steps of a layer went into one TMEM
        // accumulator).  So one TMEM accumulator only ever sums ONE k-block (4 k-steps x 3 passes = 12 MMAs);
        // the epilogue warps promote each partial tile into FP32 registers with round-to-nearest adds.
        {   // the whole warp, converged; the elected lane issues (see umma_f16_elect)
            constexpr uint32_t idesc = make_idesc_f16(BM, BN);
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            for (long long t = first; t < num_tiles; t += step) {
                int g_left = 0;
                for (int kb = 0; kb < num_kb; ++kb) {
                    const bool g_first = g_left == 0;
                    if (g_first) g_left = group_len(kb, a.group, a.lead_kb);
                    const bool g_last = --g_left == 0 || kb == num_kb - 1;
                    if (g_last) g_left = 0;
                    if (g_first) mbar_wait(&tempty[acc], acc_phase ^ 1);
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
                    const uint32_t st = smem_u32(stage_base) + (uint32_t)stage * (uint32_t)C::STAGE_BYTES;
                    const uint64_t a_hi = make_smem_desc(st), a_lo = make_smem_desc(st + C::A_BYTES);
                    const uint64_t w_hi = make_smem_desc(st + 2 * C::A_BYTES), w_lo = make_smem_desc(st + 2 * C::A_BYTES + C::W_BYTES);
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k) {
                        const uint64_t adv = (uint64_t)((k * UMMA_K * 2) >> 4);   // 32 B per k-step inside the swizzle row
                        umma_f16_elect(d_tmem, a_lo + adv, w_hi + adv, idesc, !(g_first && k == 0));   // small terms first
                        umma_f16_elect(d_tmem, a_hi + adv, w_lo + adv, idesc, 1);
                        umma_f16_elect(d_tmem, a_hi + adv, w_hi + adv, idesc, 1);
                    }
                    // operand stage free once these MMAs have read it (told to every CTA that writes into it)
                    if (CL == 1) umma_commit_elect(&empty[stage]);
                    else umma_commit_mcast_elect(&empty[stage], kMask);
                    if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
                    if (g_last) {
                        umma_commit_elect(&tfull[acc]);     // partial tile ready for promotion
                        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                    }
                }
            }
        }
    } else if (warp < kFirstEpilogueWarp) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kProducerRegs));   // idle warps of group 0
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kEpilogueRegs));
        // ===== epilogue warps: TMEM lane quadrant = warp id % 4, column half = (warp - 4) / 4 =====
        const int quad = warp & 3, half = (warp - kFirstEpilogueWarp) >> 2;
        int acc = 0; uint32_t acc_phase = 0;
        int tile_parity = 0;
        for (long long t = first; t < num_tiles; t += step) {
            const int z = (int)(t / tiles_per_problem);
            const long long tt = t % tiles_per_problem;
            const long long row = ((tt / tiles_n) * CL + crank) * BM + quad * 32 + lane;
            const int n0 = (int)(tt % tiles_n) * BN + half * HALF;
            const float inv_scale = a.inv_scale[z];
            const float* __restrict__ bias = a.bias[z];
            float* __restrict__ Yf32 = a.Yf32[z];
            __half* __restrict__ Yhi = a.Yhi[z];
            __half* __restrict__ Ylo = a.Ylo[z];
            float* bias_s = bias_all + (warp - kFirstEpilogueWarp) * HALF;   // this warp's slice of the bias, read back as broadcasts
            float* dotw_s = dotw_all + (warp - kFirstEpilogueWarp) * HALF;
            const float* __restrict__ dot_w = a.dot_w[z];
            // this tile's bias (and dot weights) are fetched now and parked in shared memory after the promotion loop:
            // the L2 latency hides behind the accumulator waits instead of stalling the start of every tile
            float bias_r[(HALF + 31) / 32], dotw_r[(HALF + 31) / 32];
            if constexpr (kBiasSmem) {
#pragma unroll
                for (int i = 0; i < (HALF + 31) / 32; ++i) {
                    const int j = lane + 32 * i;
                    bias_r[i] = j < HALF ? __ldg(bias + n0 + j) : 0.f;
                    dotw_r[i] = (dot_w && j < HALF) ? __ldg(dot_w + n0 + j) : 0.f;
                }
            } else if (lane < HALF / 32) {
                prefetch_l1(bias + n0 + lane * 32);   // the store phase reads the bias through L1
            }
            float sum[HALF];
#pragma unroll
            for (int j = 0; j < HALF; ++j) sum[j] = 0.f;
            for (int kb = 0; kb < num_kb; kb += group_len(kb, a.group, a.lead_kb)) {
                mbar_wait(&tfull[acc], acc_phase);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BN + half * HALF);
                // the next 32-column load is in flight while the previous one is added (two register buffers)
                uint32_t v[2][32];
                tmem_ld32(taddr, v[0]);
#pragma unroll
                for (int c0 = 0; c0 < HALF; c0 += 32) {
                    tmem_ld_wait();
                    if (c0 + 32 < HALF) tmem_ld32(taddr + c0 + 32, v[((c0 >> 5) + 1) & 1]);
#pragma unroll
                    for (int j = 0; j < 32; ++j) sum[c0 + j] += __uint_as_float(v[(c0 >> 5) & 1][j]);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty[acc]);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
            if constexpr (kBiasSmem) {
                __syncwarp();   // the previous tile's reads of the slices are done (same warp, program order + this fence)
#pragma unroll
                for (int i = 0; i < (HALF + 31) / 32; ++i) {
                    const int j = lane + 32 * i;
                    if (j < HALF) { bias_s[j] = bias_r[i]; dotw_s[j] = dotw_r[i]; }
                }
                __syncwarp();
            }
            if constexpr (BN == 64) {
                if (a.neck) {
                    // y = tanh(.) of this warp's 32 of the 64 columns -> partial latent -> exchange -> heads' first layers
                    float lat[kNeckLatent];
#pragma unroll
                    for (int m = 0; m < kNeckLatent; ++m) lat[m] = 0.f;
                    NLML_ACT_DISPATCH(a.act,
                        _Pragma("unroll")
                        for (int j = 0; j < HALF; ++j) {
                            const float y = act_fixed<ACT>(fmaf(sum[j], inv_scale, bias_s[j]));
                            _Pragma("unroll")
                            for (int m = 0; m < kNeckLatent; ++m) lat[m] = fmaf(y, neck_w5s[m * 64 + n0 + j], lat[m]);
                        })
                    const int r = quad * 32 + lane;
#pragma unroll
                    for (int m = 0; m < kNeckLatent; ++m) neck_xch[(half * kNeckLatent + m) * BM + r] = lat[m];
                    asm volatile("bar.sync %0, 64;" ::"r"(1 + quad) : "memory");
#pragma unroll
                    for (int m = 0; m < kNeckLatent; ++m)
                        lat[m] = (neck_xch[m * BM + r] + neck_xch[(kNeckLatent + m) * BM + r]) + neck_b5s[m];
                    asm volatile("bar.sync %0, 64;" ::"r"(1 + quad) : "memory");   // exchange buffer free for the next tile
                    if (row < a.N && half == 0 && a.neck_lat) {
#pragma unroll
                        for (int m = 0; m < kNeckLatent; ++m) a.neck_lat[row * kNeckLatent + m] = lat[m];
                    }
                    // 3 x 128 first-hidden-layer outputs per row; each column half takes 192 of them = three 64-column boxes
                    // (each inside one head), staged and handed to TMA like the wide tiles' planes (rows past N are clipped)
                    uint4* buf = stage_all + (warp - kFirstEpilogueWarp) * (kStoreStageBytes / 16);
#pragma unroll 1
                    for (int bi = 0; bi < 3; ++bi) {
                        const int o0 = half * 192 + 64 * bi, h = o0 / kNeckHeadW, j0 = o0 % kNeckHeadW;
                        const float l0 = h == 0 ? lat[0] : (h == 1 ? lat[3] : lat[6]);
                        const float l1 = h == 0 ? lat[1] : (h == 1 ? lat[4] : lat[7]);
                        const float l2 = h == 0 ? lat[2] : (h == 1 ? lat[5] : lat[8]);
                        uint32_t hi[32], lo[32];
#pragma unroll
                        for (int e = 0; e < 32; ++e) {
                            const float4 w0 = neck_whs[h * kNeckHeadW + j0 + 2 * e], w1 = neck_whs[h * kNeckHeadW + j0 + 2 * e + 1];
                            const float v0 = relu_nan(fmaf(l2, w0.z, fmaf(l1, w0.y, fmaf(l0, w0.x, w0.w))));
                            const float v1 = relu_nan(fmaf(l2, w1.z, fmaf(l1, w1.y, fmaf(l0, w1.x, w1.w))));
                            split_pair(v0, v1, hi[e], lo[e]);
                        }
                        stage_box_tma(buf, hi, &maps.y_hi[h], j0, (int)(row - lane), lane);
                        stage_box_tma(buf, lo, &maps.y_lo[h], j0, (int)(row - lane), lane);
                    }
                }
            }
            if (dot_w) {
                // fused final layer: this thread's share of the row's dot product, then the two column halves
                // of a lane quadrant meet through shared memory (named barrier of the two warps)
                float part = 0.f;
                NLML_ACT_DISPATCH(a.act,
                    _Pragma("unroll")
                    for (int j = 0; j < HALF; ++j)
                        part = fmaf(act_fixed<ACT>(fmaf(sum[j], inv_scale, bias_s[j])), dotw_s[j], part);)
                float* slot = dot_xch + (tile_parity * BM) + quad * 32 + lane;
                if (half == 1) *slot = part;
                asm volatile("bar.sync %0, 64;" ::"r"(1 + quad) : "memory");
                if (half == 0 && row < a.N) a.Ydot[row * a.ldd + z] = (part + *slot) + __ldg(a.dot_b[z]);
                tile_parity ^= 1;
            }
            if constexpr (BN >= 128) {
                if (a.y_tma) {   // planes only (every layer of the chain but the last)
                    uint4* buf = stage_all + (warp - kFirstEpilogueWarp) * (kStoreStageBytes / 16);
                    NLML_ACT_DISPATCH(a.act, store_planes_tma<ACT, HALF>(sum, inv_scale, bias + n0, buf, &maps.y_hi[z], &maps.y_lo[z],
                                                                         n0, (int)(row - lane), lane);)
                    continue;
                }
            }
            if (row < a.N && (Yf32 || Yhi)) {
                float* yf = Yf32 ? Yf32 + row * a.ldy + n0 : nullptr;
                __half* dh = Yhi ? Yhi + row * a.ldy + n0 : nullptr;
                __half* dl = Yhi ? Ylo + row * a.ldy + n0 : nullptr;
                NLML_ACT_DISPATCH(a.act, store_row<ACT, HALF, kBiasSmem>(sum, inv_scale, kBiasSmem ? bias_s : bias + n0, yf, dh, dl);)
            }
        }
        if (a.y_tma) tma_store_wait_all_elect();   // the last boxes are out before the CTA retires
    }
    tc_fence_before();
    __syncthreads();
    if (CL > 1) cluster_sync_all();   // no CTA may exit while its peer can still multicast into it
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, C::TMEM_COLS);
    }
}

// ---------------------------------------------------------------------------------------------------------
// 2-CTA variant for the 256-wide layers: a cluster of two CTAs (one SM pair) computes a 256 x 256 output tile
// with tcgen05.mma.cta_group::2.  Each CTA stages its own 128 rows of A and only HALF of the W tile, so a
// pipeline stage is 64 KB instead of 96 KB: three stages fit (the 2-stage ring of the 1-CTA kernel could not
// hide the TMA latency: tensor pipe 46 % busy) and each SM ingests a third less operand data per MMA.
// The leader CTA (cluster rank 0) issues every MMA; accumulators land in each CTA's own TMEM (its 128 rows),
// and each CTA's eight epilogue warps promote / finish their half exactly as in the 1-CTA kernel.
// ---------------------------------------------------------------------------------------------------------
#ifdef NLML_MLP_TIMING
// development build only: cycles the epilogue warps of linear_tc2_kernel spend per tile in (0) bias staging, (1) waiting for
// a partial accumulator, (2) promotion (TMEM loads + adds), (3) activation / plane split / stores
#define NLML_MT_DECL float mt_acc[4] = {0.f, 0.f, 0.f, 0.f}; uint32_t mt_prev = (uint32_t)clock(); int mt_tiles = 0;
#define NLML_MT_STAMP(i) { const uint32_t mt_now = (uint32_t)clock(); mt_acc[i] += (float)(mt_now - mt_prev); mt_prev = mt_now; }
#define NLML_MT_RESET() { mt_prev = (uint32_t)clock(); }
#else
#define NLML_MT_DECL
#define NLML_MT_STAMP(i)
#define NLML_MT_RESET()
#endif

constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;   // shared::cluster address of the same offset in the pair's even CTA

struct Cfg2 {
    static constexpr int BN = 256;
    static constexpr int STAGES = 3;
    static constexpr int A_BYTES = BM * BK * 2;            // one plane of this CTA's A tile (128 rows)
    static constexpr int W_BYTES = (BN / 2) * BK * 2;      // one plane of this CTA's half of the W tile (128 rows)
    static constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * W_BYTES;   // 64 KB
    static constexpr int TMEM_COLS = 2 * BN;
    static constexpr size_t SMEM_BYTES = 1024 + (size_t)STAGES * STAGE_BYTES + 256 +
                                         kEpilogueWarps * kStoreStageBytes /*line-forming store staging*/;
};

__device__ __forceinline__ void tma_load_2d_2sm(void* smem_dst, const CUtensorMap* map, int c_inner, int c_outer, uint64_t* leader_bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(c_inner), "r"(c_outer),
          "r"(smem_u32(leader_bar) & kPeerBitMask)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_f16_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_f16_2sm_elect(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, e;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "@e tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit_2sm_elect(uint64_t* bar, uint16_t cta_mask) {
    asm volatile(
        "{\n\t.reg .pred e;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "@e tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n\t}"
        ::"r"(smem_u32(bar)), "h"(cta_mask) : "memory");
}
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(cta_mask) : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerBitMask) : "memory");
}

__global__ void __launch_bounds__(kThreads, 1)
linear_tc2_kernel(const __grid_constant__ TcMaps maps, const __grid_constant__ LinearTcArgs a) {
    using C = Cfg2;
    constexpr int BN = C::BN, HALF = BN / 2;
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment by pointer arithmetic on the __shared__ array (a round trip through uintptr_t makes the compiler
    // lose the address space: the epilogue's bias reads became generic LD.E instead of LDS)
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* stage_base = smem;
    uint4* stage_all = reinterpret_cast<uint4*>(smem + (size_t)C::STAGES * C::STAGE_BYTES);   // [warp][32][8] store staging, 1024-byte aligned
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)C::STAGES * C::STAGE_BYTES + kEpilogueWarps * kStoreStageBytes);
    uint64_t* full = bars;                    // [STAGES]  (leader's copy is the live one) both CTAs' operand stage landed
    uint64_t* empty = bars + C::STAGES;       // [STAGES]  (own) stage consumed by the pair's MMAs
    uint64_t* tfull = bars + 2 * C::STAGES;   // [2]  (own) partial accumulator of one k-block complete
    uint64_t* tempty = tfull + 2;             // [2]  (leader's copy) drained by all 16 epilogue warps of the pair
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;   // provably warp-uniform
    const uint32_t crank = cluster_ctarank();
    const bool leader = crank == 0;
    const int num_kb = a.Kp / BK;
    const int tiles_n = a.out / BN;
    const long long tiles_m = ((a.N + BM - 1) / BM + 1) / 2;          // pairs of 128-row tiles
    const long long tiles_per_problem = tiles_m * tiles_n;
    const long long num_tiles = tiles_per_problem * a.problems;
    const long long first = blockIdx.x / 2, step = gridDim.x / 2;

    if (warp == 0 && lane == 0) {
        for (int z = 0; z < a.problems; ++z) {
            prefetch_tmap(&maps.a_hi[z]); prefetch_tmap(&maps.a_lo[z]); prefetch_tmap(&maps.w_hi[z]); prefetch_tmap(&maps.w_lo[z]);
        }
        for (int s = 0; s < C::STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 2 * kEpilogueWarps); }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc_2sm(tmem_slot, C::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kProducerRegs));   // register hand-over, see kThreads
        // ===== TMA producer (both CTAs): own A rows, own half of the W tile; bytes are counted on the leader's barrier =====
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (long long t = first; t < num_tiles; t += step) {
                const int z = (int)(t / tiles_per_problem);
                const long long tt = t % tiles_per_problem;
                const int m0 = (int)((tt / tiles_n) * 2 + crank) * BM;
                const int n0 = (int)(tt % tiles_n) * BN + (int)crank * HALF;
                for (int kb = 0; kb < num_kb; ++kb) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    uint8_t* st = stage_base + (size_t)stage * C::STAGE_BYTES;
                    if (leader) mbar_expect_tx(&full[stage], 2 * C::STAGE_BYTES);
                    tma_load_2d_2sm(st, &maps.a_hi[z], kb * BK, m0, &full[stage]);
                    tma_load_2d_2sm(st + C::A_BYTES, &maps.a_lo[z], kb * BK, m0, &full[stage]);
                    tma_load_2d_2sm(st + 2 * C::A_BYTES, &maps.w_hi[z], kb * BK, n0, &full[stage]);
                    tma_load_2d_2sm(st + 2 * C::A_BYTES + C::W_BYTES, &maps.w_lo[z], kb * BK, n0, &full[stage]);
                    if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kProducerRegs));   // register hand-over, see kThreads
        // ===== MMA issuer (leader CTA only; one instruction drives both SMs' tensor cores) =====
        if (leader) {   // the whole warp of the leader CTA, converged; the elected lane issues
            constexpr uint32_t idesc = make_idesc_f16(2 * BM, BN);
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            for (long long t = first; t < num_tiles; t += step) {
                int g_left = 0;
                for (int kb = 0; kb < num_kb; ++kb) {
                    const bool g_first = g_left == 0;
                    if (g_first) g_left = group_len(kb, a.group, a.lead_kb);
                    const bool g_last = --g_left == 0 || kb == num_kb - 1;
                    if (g_last) g_left = 0;
                    if (g_first) mbar_wait(&tempty[acc], acc_phase ^ 1);
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
                    const uint32_t st = smem_u32(stage_base) + (uint32_t)stage * (uint32_t)C::STAGE_BYTES;
                    const uint64_t a_hi = make_smem_desc(st), a_lo = make_smem_desc(st + C::A_BYTES);
                    const uint64_t w_hi = make_smem_desc(st + 2 * C::A_BYTES), w_lo = make_smem_desc(st + 2 * C::A_BYTES + C::W_BYTES);
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k) {
                        const uint64_t adv = (uint64_t)((k * UMMA_K * 2) >> 4);
                        umma_f16_2sm_elect(d_tmem, a_lo + adv, w_hi + adv, idesc, !(g_first && k == 0));
                        umma_f16_2sm_elect(d_tmem, a_hi + adv, w_lo + adv, idesc, 1);
                        umma_f16_2sm_elect(d_tmem, a_hi + adv, w_hi + adv, idesc, 1);
                    }
                    umma_commit_2sm_elect(&empty[stage], 3);   // both CTAs' producers may refill the stage
                    if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
                    if (g_last) {
                        umma_commit_2sm_elect(&tfull[acc], 3);     // both CTAs' epilogue warps may promote their half
                        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                    }
                }
            }
        }
    } else if (warp < kFirstEpilogueWarp) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kProducerRegs));   // idle warps of group 0
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kEpilogueRegs));
        // ===== epilogue warps of this CTA: rows of its own 128-row half =====
        const int quad = warp & 3, half = (warp - kFirstEpilogueWarp) >> 2;
        int acc = 0; uint32_t acc_phase = 0;
        NLML_MT_DECL
        for (long long t = first; t < num_tiles; t += step) {
            NLML_MT_RESET();
            const int z = (int)(t / tiles_per_problem);
            const long long tt = t % tiles_per_problem;
            const long long row = ((tt / tiles_n) * 2 + crank) * BM + quad * 32 + lane;
            const int n0 = (int)(tt % tiles_n) * BN + half * HALF;
            const float inv_scale = a.inv_scale[z];
            const float* __restrict__ bias = a.bias[z];
            float* __restrict__ Yf32 = a.Yf32[z];
            __half* __restrict__ Yhi = a.Yhi[z];
            __half* __restrict__ Ylo = a.Ylo[z];
            if (lane < HALF / 32) prefetch_l1(bias + n0 + lane * 32);   // the store phase reads the bias through L1
            NLML_MT_STAMP(0);
            float sum[HALF];
#pragma unroll
            for (int j = 0; j < HALF; ++j) sum[j] = 0.f;
            for (int kb = 0; kb < num_kb; kb += group_len(kb, a.group, a.lead_kb)) {
                mbar_wait(&tfull[acc], acc_phase);
                tc_fence_after();
                NLML_MT_STAMP(1);
                const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BN + half * HALF);
                // the next 32-column load is in flight while the previous one is added (two register buffers)
                uint32_t v[2][32];
                tmem_ld32(taddr, v[0]);
#pragma unroll
                for (int c0 = 0; c0 < HALF; c0 += 32) {
                    tmem_ld_wait();
                    if (c0 + 32 < HALF) tmem_ld32(taddr + c0 + 32, v[((c0 >> 5) + 1) & 1]);
#pragma unroll
                    for (int j = 0; j < 32; ++j) sum[c0 + j] += __uint_as_float(v[(c0 >> 5) & 1][j]);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_leader(&tempty[acc]);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                NLML_MT_STAMP(2);
            }
            if (a.y_tma) {   // planes only (every layer of the chain but the last)
                uint4* buf = stage_all + (warp - kFirstEpilogueWarp) * (kStoreStageBytes / 16);
                NLML_ACT_DISPATCH(a.act, store_planes_tma<ACT, HALF>(sum, inv_scale, bias + n0, buf, &maps.y_hi[z], &maps.y_lo[z], n0,
                                                                     (int)(row - lane), lane);)
            } else if (row < a.N) {
                float* yf = Yf32 ? Yf32 + row * a.ldy + n0 : nullptr;
                __half* dh = Yhi ? Yhi + row * a.ldy + n0 : nullptr;
                __half* dl = Yhi ? Ylo + row * a.ldy + n0 : nullptr;
                NLML_ACT_DISPATCH(a.act, store_row<ACT, HALF, false>(sum, inv_scale, bias + n0, yf, dh, dl);)
            }
            NLML_MT_STAMP(3);
#ifdef NLML_MLP_TIMING
            ++mt_tiles;
#endif
        }
        if (a.y_tma) tma_store_wait_all_elect();   // the last boxes are out before the CTA retires
#ifdef NLML_MLP_TIMING
        if (lane == 0 && a.timing && mt_tiles > 0)
            for (int i = 0; i < 4; ++i)
                a.timing[((size_t)blockIdx.x * kEpilogueWarps + (warp - kFirstEpilogueWarp)) * 4 + i] = mt_acc[i] / (float)mt_tiles;
#endif
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc_2sm(tmem_base, C::TMEM_COLS);
    }
}

// FP32 -> (hi, lo) FP16 planes, rows padded with zeros to Kp columns.
// IPD: the rows are RAW MediaPipe landmarks (x,y,z of landmark i at columns 3i..3i+2) and the translation /
// scale normalisation of helpers/FeatureExtractor.py:30-66 (+ :89-90, :105) is applied on the way in: subtract the
// nose tip (landmark 1), divide by the inter-pupillary distance ||lm33 - lm263|| (1e-6 when zero), in FLOAT64 as
// the reference's Python floats, then round to float32 (`.float()`) -- so the encoder sees bit-identical inputs
// (ipd_row / ipd_map in common.cuh, shared with the Tucker kernels' raw-landmark loads).
template <bool IPD>
__global__ void __launch_bounds__(256) split_planes_kernel(const float* __restrict__ X, long long N, long long ldx, int K,
                                                          int Kp, int vec_ok, __half* __restrict__ Xhi,
                                                          __half* __restrict__ Xlo) {
    const int groups = Kp / 4;
    const long long total = N * groups;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long row = idx / groups;
        const int k = (int)(idx % groups) * 4;
        const float* src = X + row * ldx;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (vec_ok && k + 3 < K) {
            v = __ldcs(reinterpret_cast<const float4*>(src + k));
        } else {
            if (k + 0 < K) v.x = __ldg(src + k + 0);
            if (k + 1 < K) v.y = __ldg(src + k + 1);
            if (k + 2 < K) v.z = __ldg(src + k + 2);
            if (k + 3 < K) v.w = __ldg(src + k + 3);
        }
        float f[4] = {v.x, v.y, v.z, v.w};
        if constexpr (IPD) {
            // the nine values every thread of the row needs come from L1 after the first touch
            const IpdRow nr = ipd_row(src);
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (k + j < K) f[j] = ipd_map(f[j], nr, (k + j) % 3);
        }
        uint32_t h[2], l[2];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            split_pair(f[2 * j], f[2 * j + 1], h[j], l[j]);
        }
        *reinterpret_cast<uint2*>(Xhi + row * Kp + k) = make_uint2(h[0], h[1]);
        *reinterpret_cast<uint2*>(Xlo + row * Kp + k) = make_uint2(l[0], l[1]);
    }
}

// Callers' post-processing of the three angles (radians, float32) in FLOAT64, as their Python statements:
//   deg = round(np.degrees(t.item()), decimals)       NLML_HPE_Test.py:273 (3), generatePose_on_video.py:210 (2)
//       = rint(rad * (180/pi) * 10^decimals) / 10^decimals     (numpy's round: scale, rint, divide)
// and, when alpha > 0, the exponential smoothing over consecutive frames (= consecutive rows) of
// generatePose_on_video.py:215-224:  s_0 = y_0,  s_t = alpha*y_t + (1-alpha)*s_{t-1}.
// The recurrence is evaluated in frame order by one thread per angle so the result is bit-identical to the Python
// loop (a parallel scan would re-associate the sums); it is three multiplies and an add per frame.
__global__ void __launch_bounds__(128) pose_post_kernel(const float* __restrict__ YPR, long long N, double scale, double alpha,
                                                       double one_minus_alpha, double* __restrict__ DEG) {
    constexpr double kRadToDeg = 180.0 / 3.14159265358979323846;
    if (alpha > 0.0) {
        const int j = blockIdx.x * blockDim.x + threadIdx.x;
        if (j >= 3) return;
        double s = 0.0;
        for (long long t0 = 0; t0 < N; t0 += 8) {
            double y[8];   // eight independent loads + roundings in flight, then the dependent chain
#pragma unroll
            for (int i = 0; i < 8; ++i)
                y[i] = (t0 + i < N) ? __ddiv_rn(rint(__dmul_rn(__dmul_rn((double)__ldg(YPR + (t0 + i) * 3 + j), kRadToDeg), scale)), scale) : 0.0;
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (t0 + i < N) {
                    s = (t0 + i == 0) ? y[i] : __dadd_rn(__dmul_rn(alpha, y[i]), __dmul_rn(one_minus_alpha, s));
                    DEG[(t0 + i) * 3 + j] = s;
                }
        }
        return;
    }
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < 3 * N; i += (long long)gridDim.x * blockDim.x)
        DEG[i] = __ddiv_rn(rint(__dmul_rn(__dmul_rn((double)YPR[i], kRadToDeg), scale)), scale);
}

// ---------------------------------------------------------------------------------------------------------
// Narrow layers (not dense contractions worth a tensor-core tile): thread-per-sample CUDA-core kernels with
// the weights broadcast from shared memory, several layers fused per launch.
// ---------------------------------------------------------------------------------------------------------

constexpr int kRowsPerBlock = 64;   // samples per block of the fused narrow-layer kernels
constexpr int kLanesPerRow = 1;     // lanes sharing one sample (1 measured faster than 4: the weight broadcast then
                                    // costs one shared-memory wavefront set per warp instead of one per quarter-warp)
constexpr int kNarrowThreads = kRowsPerBlock * kLanesPerRow;

// Stage kRowsPerBlock rows of IN floats into shared memory with coalesced 128-bit loads.  Row pitch IN+4
// floats keeps the later 128-bit reads of 8 different rows per warp conflict-free.
template <int IN>
__device__ __forceinline__ void stage_rows(const float* __restrict__ X, long long row0, long long N, float* xs) {
    constexpr int V = IN / 4, PITCH = IN + 4;
    for (int idx = threadIdx.x; idx < kRowsPerBlock * V; idx += kNarrowThreads) {
        const int r = idx / V, c4 = idx % V;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (row0 + r < N) v = __ldg(reinterpret_cast<const float4*>(X + (row0 + r) * IN) + c4);
        *reinterpret_cast<float4*>(xs + r * PITCH + 4 * c4) = v;
    }
}

// acc[j] += sum_k Wt[k][j0 + j] * x[k], j < OUTQ: one lane's quarter of a row's outputs.  Wt is the transposed
// weight in shared memory (row pitch WP floats) so the j index is contiguous; x is the staged row.
template <int IN, int OUTQ, int WP>
__device__ __forceinline__ void row_gemv(const float* __restrict__ xrow, const float* __restrict__ Wt_q, float (&acc)[OUTQ]) {
    static_assert(IN % 4 == 0 && OUTQ % 4 == 0, "vector widths");
#pragma unroll 4
    for (int k4 = 0; k4 < IN / 4; ++k4) {
        const float4 xv = *(reinterpret_cast<const float4*>(xrow) + k4);
        const float xs[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            const float4* wrow = reinterpret_cast<const float4*>(Wt_q + (4 * k4 + kk) * WP);
#pragma unroll
            for (int j4 = 0; j4 < OUTQ / 4; ++j4) {
                const float4 w = wrow[j4];
                acc[4 * j4 + 0] = fmaf(xs[kk], w.x, acc[4 * j4 + 0]);
                acc[4 * j4 + 1] = fmaf(xs[kk], w.y, acc[4 * j4 + 1]);
                acc[4 * j4 + 2] = fmaf(xs[kk], w.z, acc[4 * j4 + 2]);
                acc[4 * j4 + 3] = fmaf(xs[kk], w.w, acc[4 * j4 + 3]);
            }
        }
    }
}

__device__ __forceinline__ float quad_sum(float v) {
#pragma unroll
    for (int o = kLanesPerRow / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

struct NeckArgs {
    const float* X;      // [N][D_IN]   output of the last wide encoder layer (ReLU applied)
    long long N;
    const float *W4t, *B4;  // [D_IN][D_MID] (pre-transposed), [D_MID]     encoder.8  (Tanh)
    const float *W5, *B5;   // [D_LAT][D_MID], [D_LAT]    encoder.10 (none)
    const float* Wh[3];     // [HW][HIN]                  model.0 of yaw / pitch / roll (ReLU)
    const float* Bh[3];
    float* LAT;             // [N][D_LAT] or null
    __half* Hhi[3];         // [N][HW] planes of the head's first hidden layer, or null
    __half* Hlo[3];
    float* Hf32[3];         // [N][HW] FP32 instead (CUDA-core head path), or null
};

// encoder.8 (128->64, tanh) + encoder.10 (64->9) + latent split + model.0 of the three heads (3->128, ReLU)
template <int D_IN, int D_MID, int D_LAT, int HIN, int HW>
__global__ void __launch_bounds__(kNarrowThreads) neck_kernel(const __grid_constant__ NeckArgs a) {
    static_assert(D_LAT == 3 * HIN, "latent splits into three head inputs");
    constexpr int MQ = D_MID / kLanesPerRow, HQ = HW / kLanesPerRow;
    static_assert(MQ % 4 == 0 && HQ % 8 == 0, "quarter widths");
    extern __shared__ __align__(16) float nsm[];
    float* W4t = nsm;                       // [D_IN][D_MID]
    float* xs = W4t + D_IN * D_MID;         // [kRowsPerBlock][D_IN + 4]
    float* W5s = xs + kRowsPerBlock * (D_IN + 4);   // [D_LAT][D_MID]
    float* Whs = W5s + D_LAT * D_MID;       // [3][HW][HIN]
    float* Bs = Whs + 3 * HW * HIN;         // B4[D_MID], B5[D_LAT], Bh[3][HW]
    const long long row0 = (long long)blockIdx.x * kRowsPerBlock;
    stage_rows<D_IN>(a.X, row0, a.N, xs);
    for (int i = threadIdx.x; i < D_IN * D_MID / 4; i += kNarrowThreads)
        reinterpret_cast<float4*>(W4t)[i] = __ldg(reinterpret_cast<const float4*>(a.W4t) + i);
    for (int i = threadIdx.x; i < D_LAT * D_MID; i += kNarrowThreads) W5s[i] = __ldg(a.W5 + i);
    for (int i = threadIdx.x; i < 3 * HW * HIN; i += kNarrowThreads) Whs[i] = __ldg(a.Wh[i / (HW * HIN)] + i % (HW * HIN));
    for (int i = threadIdx.x; i < D_MID; i += kNarrowThreads) Bs[i] = __ldg(a.B4 + i);
    for (int i = threadIdx.x; i < D_LAT; i += kNarrowThreads) Bs[D_MID + i] = __ldg(a.B5 + i);
    for (int i = threadIdx.x; i < 3 * HW; i += kNarrowThreads) Bs[D_MID + D_LAT + i] = __ldg(a.Bh[i / HW] + i % HW);
    __syncthreads();
    const int s = threadIdx.x / kLanesPerRow, q = threadIdx.x % kLanesPerRow;
    const long long row = row0 + s;
    const bool valid = row < a.N;   // invalid rows compute on zeros and store nothing (the quad shuffles need all lanes)

    float h[MQ];
#pragma unroll
    for (int j = 0; j < MQ; ++j) h[j] = Bs[q * MQ + j];
    row_gemv<D_IN, MQ, D_MID>(xs + s * (D_IN + 4), W4t + q * MQ, h);
#pragma unroll
    for (int j = 0; j < MQ; ++j) h[j] = tanhf(h[j]);
    float lat[D_LAT];
#pragma unroll
    for (int l = 0; l < D_LAT; ++l) {
        float acc = 0.f;
#pragma unroll
        for (int j = 0; j < MQ; ++j) acc = fmaf(W5s[l * D_MID + q * MQ + j], h[j], acc);
        lat[l] = quad_sum(acc) + Bs[D_MID + l];
    }
    if (a.LAT && valid && q == 0) {
#pragma unroll
        for (int l = 0; l < D_LAT; ++l) a.LAT[row * D_LAT + l] = lat[l];
    }
    if (!valid) return;
#pragma unroll
    for (int z = 0; z < 3; ++z) {
        if (!a.Hhi[z] && !a.Hf32[z]) continue;
#pragma unroll 1
        for (int j0 = q * HQ; j0 < (q + 1) * HQ; j0 += 8) {
            float y[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float acc = Bs[D_MID + D_LAT + z * HW + j0 + j];
#pragma unroll
                for (int i = 0; i < HIN; ++i) acc = fmaf(Whs[(z * HW + j0 + j) * HIN + i], lat[z * HIN + i], acc);
                y[j] = relu_nan(acc);
            }
            if (a.Hf32[z]) {
                float4* d = reinterpret_cast<float4*>(a.Hf32[z] + row * HW + j0);
                d[0] = make_float4(y[0], y[1], y[2], y[3]);
                d[1] = make_float4(y[4], y[5], y[6], y[7]);
            }
            if (a.Hhi[z]) {
                uint32_t hi[4], lo[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    split_pair(y[2 * j], y[2 * j + 1], hi[j], lo[j]);
                }
                *reinterpret_cast<uint4*>(a.Hhi[z] + row * HW + j0) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                *reinterpret_cast<uint4*>(a.Hlo[z] + row * HW + j0) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
            }
        }
    }
}

struct HeadTailArgs {
    const float* X[3];      // [N][D_IN]  output of model.4 (ReLU applied) per head
    long long N;
    const float *W3t[3], *B3[3];  // [D_IN][D_MID] (pre-transposed), [D_MID]   model.6 (ReLU)
    const float *W4[3], *B4[3];   // [1][D_MID], [1]          model.8 (none)
    float* YPR;                   // [N][3]
};

// model.6 (128->64, ReLU) + model.8 (64->1) of one head per blockIdx.y
template <int D_IN, int D_MID>
__global__ void __launch_bounds__(kNarrowThreads) head_tail_kernel(const __grid_constant__ HeadTailArgs a) {
    constexpr int MQ = D_MID / kLanesPerRow;
    extern __shared__ __align__(16) float hsm[];
    float* W3t = hsm;                   // [D_IN][D_MID]
    float* xs = W3t + D_IN * D_MID;     // [kRowsPerBlock][D_IN + 4]
    float* rest = xs + kRowsPerBlock * (D_IN + 4);   // B3[D_MID], W4[D_MID], B4[1]
    const int z = blockIdx.y;
    const long long row0 = (long long)blockIdx.x * kRowsPerBlock;
    stage_rows<D_IN>(a.X[z], row0, a.N, xs);
    for (int i = threadIdx.x; i < D_IN * D_MID / 4; i += kNarrowThreads)
        reinterpret_cast<float4*>(W3t)[i] = __ldg(reinterpret_cast<const float4*>(a.W3t[z]) + i);
    for (int i = threadIdx.x; i < D_MID; i += kNarrowThreads) {
        rest[i] = __ldg(a.B3[z] + i);
        rest[D_MID + i] = __ldg(a.W4[z] + i);
    }
    if (threadIdx.x == 0) rest[2 * D_MID] = __ldg(a.B4[z]);
    __syncthreads();
    const int s = threadIdx.x / kLanesPerRow, q = threadIdx.x % kLanesPerRow;
    const long long row = row0 + s;
    float h[MQ];
#pragma unroll
    for (int j = 0; j < MQ; ++j) h[j] = rest[q * MQ + j];
    row_gemv<D_IN, MQ, D_MID>(xs + s * (D_IN + 4), W3t + q * MQ, h);
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < MQ; ++j) acc = fmaf(rest[D_MID + q * MQ + j], relu_nan(h[j]), acc);
    acc = quad_sum(acc) + rest[2 * D_MID];
    if (row < a.N && q == 0) a.YPR[row * 3 + z] = acc;
}

// ---- host side: tensor maps --------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// 2D map over a row-major fp16 plane [rows][pitch_elems] (first `cols` columns addressable), box = [BK cols][box_rows rows]
inline int make_plane_map(CUtensorMap* map, const __half* base, long long rows, int cols, long long pitch_elems, int box_rows) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return set_error(NLML_E_UNSUPPORTED, "cuTensorMapEncodeTiled entry point not available from the driver");
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)pitch_elems * 2};
    cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error(NLML_E_INVALID, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return 0;
}

}  // namespace tc
}  // namespace nlml
