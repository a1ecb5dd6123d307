// Run-time-rank tensor-core Tucker fit for sm_100a: enlarged cores (BASELINE.json configs[4]) and any rank set the
// (5,3,3,3) kernels are not compiled for.  Same recurrence (TD_Tester.optimize_with_sgd, /root/reference/TD_Tester.py:127-159)
// and the same folded Gram tensor S[A,B,C,D] as tucker_math.h; the reference takes the ranks from the arrays
// (/root/reference/TD_Inference.py:56-57, TD_main.py:66-76), so nothing here is fixed at compile time except an upper
// class for the roll rank (register arrays) and for the identity pairs (register accumulators).
//
// Once S no longer fits one shared-memory tile it is STREAMED: the (b,c,d) axis is cut into blocks of NB columns and the
// tile images (already split hi/lo and laid out as UMMA operands by build_tiles_kernel) arrive by 1-D TMA bulk copies
// (cp.async.bulk -> SASS UBLKCP) into a ring of shared-memory slots guarded by full/empty mbarriers; the ring degenerates
// to "resident" when every block fits.  Per iteration and block j, for the CTA's 128 samples (= 128 TMEM lanes):
//   GEMM-T   D_T[s, col]  = sum_A  UU[s,A] * S[A, col]          128 x NB x KA     A operand (UU hi|lo) in TENSOR MEMORY
//   GEMM-G   D_G[s, A]    = sum_col YPR[s,col] * S[A, col]      128 x NA16 x NB   A operand written to shared memory
// with col = (b,c) pair x padded roll pair, YPR = YY_b PP_c RR_d.  Operands are FP16 hi/lo planes (kind::f16, three of
// the four cross products: FP32-grade, 22 operand bits) with power-of-two scales: S by 2^s_exp from the plan (max |S|),
// UU and YPR by per-sample, per-iteration exponents; the scales come off where the accumulators are read.  16-deep MMAs: half the instructions and half the tile bytes of a 3xTF32 split.
// Accumulation chains inside tensor memory stay short (the tensor core's FP32 accumulate truncates, which biases long
// chains); every block's partial D_G is promoted into FP32 registers with round-to-nearest adds.
//
// 512 threads = four warp groups (setmaxnreg moves the registers to where they are needed):
//   group 0  warp 0 lane 0: TMA producer.  warp 1: TMEM allocation, lane 0 issues every MMA.
//   group 1  "T readers"  one thread per sample: publishes UU, reads D_T back (tcgen05.ld) and folds it into the three
//            angle gradients on the fly; afterwards clips and steps p (p lives in shared memory, one column per sample).
//   group 2  "G formers"  one thread per sample: writes the YPR operand rows, promotes D_G, finishes d/du.
//   group 3  "linear"     one thread per sample: the linear term -q.z from q = W2 x (computed once by
//            tucker_project_kernel, kept in the CTA's [R][128] slab of global memory, L2-resident), under the GEMMs.
// Two named barriers per iteration (features published / gradient parts published).
#pragma once
#include "common.cuh"
#include "tucker_math.h"

namespace nlml {
namespace tgen {

constexpr int kSamples = 128;
constexpr int kThreads = 512;
constexpr int kMaxRank = 16;
constexpr int kMaxSlots = 16;

// Chosen on the host per plan (choose_config in tucker_fit.cu)
struct GenCfg {
    int ri, ry, rp, rr, R;
    int rrmax;               // roll-rank class the kernel is instantiated for (5 or 8)
    int nA, KA, NA16;        // identity pairs; padded to 16 (K of GEMM-T, N of GEMM-G)
    int nC, nBC;             // pitch pairs, (yaw pair, pitch pair) combinations
    int nDp;                 // roll pairs of the rrmax triangle padded to 8 = columns per (b,c) pair
    int BCP, NB, nblocks;    // (b,c) pairs per block, columns per block (multiple of 16), blocks per iteration
    int tbufs, gbufs, ybufs; // TMEM buffers of D_T and D_G, buffers of the YPR operand
    int ypr_tmem;            // the YPR operand lives in tensor memory (packed halves: NB/2 hi | NB/2 lo columns) instead of shared memory
    int col_y;               // its first TMEM column
    int tslots, gslots;      // ring slots of T tiles / G tiles
    int resident;            // every tile has its own slot and is loaded once
    int tt_bytes, gt_bytes;  // bytes of one T tile / G tile (hi plane + lo plane)
    int col_g, col_a, col_t; // TMEM columns: D_G buffers, UU operand (hi | lo), D_T buffers
    int off_tring, off_gring, off_ypr, off_tab, off_bar, smem_bytes;
    int NP;                  // 3 + ri
    int s_exp;               // the tile images hold S * 2^s_exp
    // rows of the per-sample table (floats, [row][128]):
    int t_p, t_gx, t_gl, t_cy, t_dcy, t_cp, t_dcp, t_rows;
};

struct GenArgs {
    const float* q;          // [ctas][R][128]: q = W2 x of sample 128*cta + lane
    const uint8_t* tiles;    // per block: T tile (hi, lo) then G tile (hi, lo)
    float* P;
    long long ldp, N;
    int T;
    float lr, clip;
    GenCfg c;
    float rows_y[4 * kMaxRank], rows_p[4 * kMaxRank], rows_r[4 * kMaxRank];
};

// ---- small PTX helpers (the tf32 MMA / descriptor helpers are ttc:: in tucker_tc.cuh) -----------------------------
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(ttc::smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(ttc::smem_u32(bar)) : "memory");
}
// 1-D TMA bulk copy global -> shared, completion counted on an mbarrier
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(ttc::smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(ttc::smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float* v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
                   "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
                   "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])) : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const float* v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};"
                 ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
                   "r"(__float_as_uint(v[3])) : "memory");
}
// two FP32 values -> one word of the hi plane and one of the lo plane (element 0 in the low half: the packed-halves
// layout of a tensor-memory A operand and of a 16-byte shared-memory operand chunk)
__device__ __forceinline__ void split_pair16(float v0, float v1, float& hi, float& lo) {
    const __half2 h = __floats2half2_rn(v0, v1);
    const float2 hf = __half22float2(h);
    const __half2 l = __floats2half2_rn(v0 - hf.x, v1 - hf.y);
    hi = __uint_as_float(*reinterpret_cast<const uint32_t*>(&h));
    lo = __uint_as_float(*reinterpret_cast<const uint32_t*>(&l));
}
__device__ __forceinline__ void tc_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void named_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }

#ifdef NLML_GEN_TIMING
// development build only: per-phase cycle counts of one lane per role of CTA 0 (scripts/time_gen.py)
__device__ float g_gen_timing[64];
#define GT_DECL float gt_acc[10] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}; uint32_t gt_prev = (uint32_t)clock();
#define GT(i) { const uint32_t gt_now = (uint32_t)clock(); gt_acc[i] += (float)(gt_now - gt_prev); gt_prev = gt_now; }
#define GT_OUT(role) if (blockIdx.x == 0 && lane == 0 && (warp & 3) == 1) { for (int i = 0; i < 10; ++i) g_gen_timing[(role) * 16 + i] = gt_acc[i] / (float)a.T; }
#else
#define GT_DECL
#define GT(i)
#define GT_OUT(role)
#endif

// roll features (static class RRMAX): c_l, dc_l for l < rr (0 beyond), and the monomials RR_d = c_i c_j with their
// derivative along the roll angle, d = pair_index(i, j, RRMAX), padded with zeros to NDP
template <int RRMAX, int NDP>
__device__ __forceinline__ void roll_features(float w, const float* rows_r, int rr, float (&cr)[RRMAX], float (&dcr)[RRMAX],
                                              float (&RRv)[NDP], float (&dRR)[NDP]) {
#pragma unroll
    for (int l = 0; l < RRMAX; ++l) {
        float s = 0.f, co = 0.f;
        cr[l] = 0.f;
        dcr[l] = 0.f;
        if (l < rr) {
            const float a = rows_r[4 * l], b = rows_r[4 * l + 1], ph = rows_r[4 * l + 2], d = rows_r[4 * l + 3];
            sincos_small(fmaf(b, w, ph), &s, &co);
            cr[l] = fmaf(a, co, d);
            dcr[l] = -(a * b) * s;
        }
    }
#pragma unroll
    for (int d = 0; d < NDP; ++d) RRv[d] = dRR[d] = 0.f;
#pragma unroll
    for (int i = 0; i < RRMAX; ++i)
#pragma unroll
        for (int j = i; j < RRMAX; ++j) {
            RRv[pair_index(i, j, RRMAX)] = cr[i] * cr[j];
            dRR[pair_index(i, j, RRMAX)] = fmaf(dcr[i], cr[j], cr[i] * dcr[j]);
        }
}

// position in a ring of n buffers guarded by mbarriers: index and phase parity, advanced without divisions
struct Ring {
    int idx, n;
    uint32_t phase;
    __device__ __forceinline__ Ring(int n_) : idx(0), n(n_), phase(0) {}
    __device__ __forceinline__ void next() {
        if (++idx == n) {
            idx = 0;
            phase ^= 1u;
        }
    }
};

// walk over the (b,c) pairs in storage order: b = (bi <= bj) over the yaw rank, c = (ci <= cj) over the pitch rank, c fastest
struct PairWalk {
    int bi, bj, ci, cj;
    __device__ __forceinline__ void reset() { bi = bj = ci = cj = 0; }
    // advance to the next pair; true when c wrapped (a new b starts)
    __device__ __forceinline__ bool next(int ry, int rp) {
        if (++cj == rp) {
            ++ci;
            cj = ci;
        }
        if (ci == rp) {
            ci = cj = 0;
            if (++bj == ry) {
                ++bi;
                bj = bi;
            }
            return true;
        }
        return false;
    }
};

// NA16MAX: compile-time bound of the identity-pair accumulators held in registers by the G formers (48: ri <= 8, 144: ri <= 16)
template <int RRMAX, int NA16MAX>
__global__ void __launch_bounds__(kThreads, 1) tucker_fit_gen_kernel(const __grid_constant__ GenArgs a) {
    constexpr int NDP = (tri(RRMAX) + 7) / 8 * 8;
    constexpr int kRegsProducer = 24, kRegsT = NA16MAX > 48 ? 168 : 184, kRegsG = NA16MAX > 48 ? 232 : 184,
                  kRegsL = NA16MAX > 48 ? 88 : 120;
    static_assert(kRegsProducer + kRegsT + kRegsG + kRegsL <= 512, "register file: 4 warp groups x 128 threads");
    extern __shared__ __align__(1024) uint8_t gsm[];
    const GenCfg& c = a.c;
    float* tab = reinterpret_cast<float*>(gsm + c.off_tab);
    uint64_t* bars = reinterpret_cast<uint64_t*>(gsm + c.off_bar);
    uint64_t* fullT = bars;                    // [kMaxSlots]
    uint64_t* emptyT = fullT + kMaxSlots;
    uint64_t* fullG = emptyT + kMaxSlots;
    uint64_t* emptyG = fullG + kMaxSlots;
    uint64_t* tfull = emptyG + kMaxSlots;      // [2] D_T buffer complete
    uint64_t* tempty = tfull + 2;              // [2] D_T buffer read back
    uint64_t* gfull = tempty + 2;              // [2] D_G partial complete
    uint64_t* gempty = gfull + 2;              // [2] D_G partial promoted
    uint64_t* afull = gempty + 2;              // [2] YPR operand block written
    uint64_t* aempty = afull + 2;              // [2] YPR operand block consumed by its GEMM
    uint64_t* uu_ready = aempty + 2;           // UU operand of this iteration is in tensor memory
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(uu_ready + 1);

    // the warp index through a shuffle: the compiler then knows it is warp-uniform and keeps the MMA warp's descriptor
    // arithmetic in the uniform datapath (without it every tcgen05.mma is preceded by a register->uniform broadcast loop)
    const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31, group = warp >> 2;
    const int row = tid & 127;
    const long long s0 = (long long)blockIdx.x * kSamples;
    const int nblocks = c.nblocks, NB = c.NB, KA = c.KA, NA16 = c.NA16;

    if (tid == 0) {
        for (int i = 0; i < kMaxSlots; ++i) {
            ttc::mbar_init(&fullT[i], 1); ttc::mbar_init(&emptyT[i], 1);
            ttc::mbar_init(&fullG[i], 1); ttc::mbar_init(&emptyG[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            ttc::mbar_init(&tfull[i], 1); ttc::mbar_init(&tempty[i], 4);
            ttc::mbar_init(&gfull[i], 1); ttc::mbar_init(&gempty[i], 4);
            ttc::mbar_init(&afull[i], 4); ttc::mbar_init(&aempty[i], 1);
        }
        ttc::mbar_init(uu_ready, 4);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc_cols(tmem_slot, 512);
    // p = 0 (TD_Tester.py:130) and the gradient exchange rows
    for (int i = tid; i < c.t_rows * kSamples; i += kThreads) tab[i] = 0.f;
    // the YPR operand's pad columns (NB is rounded up to the MMA's N granularity) are never written again: zero them once
    if (!c.ypr_tmem)
        for (int i = tid; i < c.ybufs * NB * kSamples; i += kThreads) reinterpret_cast<float*>(gsm + c.off_ypr)[i] = 0.f;   // 2 planes x 2 bytes
    ttc::fence_async_smem();
    tc_before();
    __syncthreads();
    tc_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t lane_addr = tmem + ((uint32_t)((warp & 3) * 32) << 16);

    if (group == 0) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegsProducer));
        if (warp == 0 && lane == 0) {
            // ===== TMA producer: tile images of block j = [T tile | G tile], contiguous in global memory =====
            const uint32_t tt = (uint32_t)c.tt_bytes, gt = (uint32_t)c.gt_bytes;
            const size_t stride = (size_t)tt + gt;
            if (c.resident) {
                for (int j = 0; j < nblocks; ++j) {
                    mbar_expect_tx(&fullT[j], tt);
                    bulk_load(gsm + c.off_tring + (size_t)j * tt, a.tiles + j * stride, tt, &fullT[j]);
                    mbar_expect_tx(&fullG[j], gt);
                    bulk_load(gsm + c.off_gring + (size_t)j * gt, a.tiles + j * stride + tt, gt, &fullG[j]);
                }
            } else {
                Ring ts(c.tslots), gs(c.gslots);
                for (int it = 0; it < a.T; ++it)
                    for (int j = 0; j < nblocks; ++j, ts.next(), gs.next()) {
                        ttc::mbar_wait(&emptyT[ts.idx], ts.phase ^ 1u);
                        mbar_expect_tx(&fullT[ts.idx], tt);
                        bulk_load(gsm + c.off_tring + (size_t)ts.idx * tt, a.tiles + j * stride, tt, &fullT[ts.idx]);
                        ttc::mbar_wait(&emptyG[gs.idx], gs.phase ^ 1u);
                        mbar_expect_tx(&fullG[gs.idx], gt);
                        bulk_load(gsm + c.off_gring + (size_t)gs.idx * gt, a.tiles + j * stride + tt, gt, &fullG[gs.idx]);
                    }
            }
        } else if (warp == 1) {
            // ===== MMA issuer: the whole warp runs the loop with warp-uniform values (descriptor arithmetic in the uniform
            // datapath); lane 0 issues the MMAs and commits =====
            const uint32_t ypr_plane = (uint32_t)NB * kSamples * 2;   // one FP16 plane of one YPR operand buffer
            Ring ts(c.resident ? nblocks : c.tslots), gs(c.resident ? nblocks : c.gslots), tb(c.tbufs), gb(c.gbufs), yb(c.ybufs);
            GT_DECL
            for (int it = 0; it < a.T; ++it) {
                ttc::mbar_wait(uu_ready, (uint32_t)(it & 1));
                GT(0)   // wait for the UU operand
                for (int j = 0; j < nblocks; ++j, ts.next(), gs.next(), tb.next(), gb.next(), yb.next()) {
                    // GEMM-T: D_T[tb] = UU (tensor memory) x T tile        (resident tiles: ts.idx == j, loaded once)
                    if (!c.resident || it == 0) ttc::mbar_wait(&fullT[ts.idx], c.resident ? 0u : ts.phase);
                    GT(1)   // wait T tile
                    ttc::mbar_wait(&tempty[tb.idx], tb.phase ^ 1u);
                    GT(2)   // wait D_T buffer
                    tc_after();
                    {
                        const uint32_t t_hi = ttc::smem_u32(gsm + c.off_tring) + (uint32_t)ts.idx * (uint32_t)c.tt_bytes;
                        ttc::gemm3h_ts(tmem + c.col_t + tb.idx * NB, tmem + c.col_a, t_hi, t_hi + c.tt_bytes / 2, KA, NB);
                    }
                    ttc::umma_commit_elect(&tfull[tb.idx]);
                    if (!c.resident) ttc::umma_commit_elect(&emptyT[ts.idx]);
                    GT(3)   // issue GEMM-T
                    // GEMM-G: D_G[gb] = YPR block (shared memory) x G tile
                    if (!c.resident || it == 0) ttc::mbar_wait(&fullG[gs.idx], c.resident ? 0u : gs.phase);
                    GT(4)   // wait G tile
                    ttc::mbar_wait(&afull[yb.idx], yb.phase);
                    GT(5)   // wait YPR operand
                    ttc::mbar_wait(&gempty[gb.idx], gb.phase ^ 1u);
                    GT(6)   // wait D_G buffer
                    tc_after();
                    {
                        const uint32_t g_hi = ttc::smem_u32(gsm + c.off_gring) + (uint32_t)gs.idx * (uint32_t)c.gt_bytes;
                        if (c.ypr_tmem) {
                            ttc::gemm3h_ts(tmem + c.col_g + gb.idx * NA16, tmem + c.col_y + yb.idx * NB, g_hi, g_hi + c.gt_bytes / 2, NB, NA16);
                        } else {
                            const uint32_t y_hi = ttc::smem_u32(gsm + c.off_ypr) + (uint32_t)yb.idx * 2u * ypr_plane;
                            ttc::gemm3h_ss(tmem + c.col_g + gb.idx * NA16, y_hi, y_hi + ypr_plane, g_hi, g_hi + c.gt_bytes / 2, NB, NA16);
                        }
                    }
                    ttc::umma_commit_elect(&gfull[gb.idx]);
                    ttc::umma_commit_elect(&aempty[yb.idx]);
                    if (!c.resident) ttc::umma_commit_elect(&emptyG[gs.idx]);
                    GT(7)   // issue GEMM-G
                }
            }
            GT_OUT(0)
        }
    } else if (group == 1) {
        // ===== T readers =====
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegsT));
        float* my = tab + row;   // this sample's column of the table: element r at my[r * 128]
        Ring tb(c.tbufs);
        GT_DECL
        for (int it = 0; it < a.T; ++it) {
            // features: roll in registers, yaw into the table; UU operand into tensor memory
            // (p of this iteration is final: barrier 3 below closes the previous iteration's step)
            float cr[RRMAX], dcr[RRMAX], RRv[NDP], dRR[NDP];
            roll_features<RRMAX, NDP>(my[(c.t_p + 2) * kSamples], a.rows_r, c.rr, cr, dcr, RRv, dRR);
            {
                const float w = my[(c.t_p + 0) * kSamples];
                for (int j = 0; j < c.ry; ++j) {
                    const float ra = a.rows_y[4 * j], rb = a.rows_y[4 * j + 1], rc = a.rows_y[4 * j + 2], rd = a.rows_y[4 * j + 3];
                    float s, co;
                    sincos_small(fmaf(rb, w, rc), &s, &co);
                    my[(c.t_cy + j) * kSamples] = fmaf(ra, co, rd);
                    my[(c.t_dcy + j) * kSamples] = -(ra * rb) * s;
                }
            }
            int uu_exp;   // this iteration's power-of-two scale of the UU operand: the largest |UU| = (max |u_i|)^2 lands in [2^12, 2^13)
            {
                float m = 0.f;
                for (int i = 0; i < c.ri; ++i) m = fmaxf(m, fabsf(my[(c.t_p + 3 + i) * kSamples]));
                m *= m;
                int eu = 12 - (((__float_as_int(m) >> 23) & 0xff) - 127);
                eu = m > 0.f ? max(min(eu, 100), -80) : 0;
                uu_exp = eu;
                const float su = __int_as_float((eu + 127) << 23);
                int i = 0, j = 0;
                for (int k0 = 0; k0 < KA; k0 += 16) {   // 16 elements = 8 packed columns per plane
                    float hi[8], lo[8];
#pragma unroll
                    for (int x = 0; x < 8; ++x) {
                        float v[2] = {0.f, 0.f};
#pragma unroll
                        for (int h = 0; h < 2; ++h)
                            if (k0 + 2 * x + h < c.nA) {
                                v[h] = my[(c.t_p + 3 + i) * kSamples] * my[(c.t_p + 3 + j) * kSamples] * su;
                                if (++j == c.ri) { ++i; j = i; }
                            }
                        split_pair16(v[0], v[1], hi[x], lo[x]);
                    }
                    tmem_st8(lane_addr + c.col_a + k0 / 2, hi);
                    tmem_st8(lane_addr + c.col_a + KA / 2 + k0 / 2, lo);
                }
                tmem_store_wait();
                tc_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(uu_ready);
            }
            GT(0)   // features + UU
            named_sync(1, 384);   // features published (yaw here, pitch by the G formers)
            GT(1)

            // D_T read-back: fold every (b,c) pair's NDP columns into the three angle gradients
            PairWalk pw;
            pw.reset();
            float YY = my[c.t_cy * kSamples] * my[c.t_cy * kSamples];
            float dYY = 2.0f * my[c.t_cy * kSamples] * my[c.t_dcy * kSamples];
            float gy = 0.f, gp = 0.f, gr = 0.f, gy_cur = 0.f;
            int pair = 0;
            for (int j = 0; j < nblocks; ++j, tb.next()) {
                ttc::mbar_wait(&tfull[tb.idx], tb.phase);
                GT(2)   // wait D_T
                tc_after();
                const uint32_t tbase = lane_addr + c.col_t + tb.idx * NB;
                // one pair = NDP columns; the next pair's tcgen05.ld is in flight while this one is folded
                auto fold = [&](const uint32_t (&t)[NDP]) {
                    const float cpi = my[(c.t_cp + pw.ci) * kSamples], cpj = my[(c.t_cp + pw.cj) * kSamples];
                    const float dpi = my[(c.t_dcp + pw.ci) * kSamples], dpj = my[(c.t_dcp + pw.cj) * kSamples];
                    const float PP = cpi * cpj, dPP = fmaf(dpi, cpj, cpi * dpj);
                    float tr0 = 0.f, tr1 = 0.f, td0 = 0.f, td1 = 0.f;   // two chains each: shorter dependent-FMA latency
#pragma unroll
                    for (int d = 0; d < NDP; d += 2) {
                        tr0 = fmaf(__uint_as_float(t[d]), RRv[d], tr0);
                        td0 = fmaf(__uint_as_float(t[d]), dRR[d], td0);
                        tr1 = fmaf(__uint_as_float(t[d + 1]), RRv[d + 1], tr1);
                        td1 = fmaf(__uint_as_float(t[d + 1]), dRR[d + 1], td1);
                    }
                    const float tr = tr0 + tr1, tdr = td0 + td1;
                    gr = fmaf(YY * PP, tdr, gr);
                    gp = fmaf(YY * dPP, tr, gp);
                    gy_cur = fmaf(PP, tr, gy_cur);
                    if (pw.next(c.ry, c.rp)) {
                        gy = fmaf(gy_cur, dYY, gy);
                        gy_cur = 0.f;
                        if (pw.bi < c.ry) {
                            const float yi = my[(c.t_cy + pw.bi) * kSamples], yj = my[(c.t_cy + pw.bj) * kSamples];
                            const float di = my[(c.t_dcy + pw.bi) * kSamples], dj = my[(c.t_dcy + pw.bj) * kSamples];
                            YY = yi * yj;
                            dYY = fmaf(di, yj, yi * dj);
                        }
                    }
                };
                auto load = [&](int pl, uint32_t (&t)[NDP]) {
#pragma unroll
                    for (int x = 0; x < NDP / 8; ++x) tmem_ld8(tbase + pl * NDP + 8 * x, t + 8 * x);
                };
                const int np = min(c.BCP, c.nBC - pair);   // pairs of this block (the last block may be short)
                uint32_t t0[NDP], t1[NDP];
                load(0, t0);
                for (int pl = 0; pl < np; pl += 2) {
                    tmem_load_wait();
                    if (pl + 1 < np) load(pl + 1, t1);
                    fold(t0);
                    if (pl + 1 < np) {
                        tmem_load_wait();
                        if (pl + 2 < np) load(pl + 2, t0);
                        fold(t1);
                    }
                }
                pair += np;
                tc_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty[tb.idx]);
                GT(3)   // fold
            }
            {
                const float kt = __int_as_float((127 - c.s_exp - uu_exp) << 23);   // 2^-(s_exp + uu_exp): the D_T accumulators' scale off
                my[(c.t_gx + 0) * kSamples] = gy * kt;
                my[(c.t_gx + 1) * kSamples] = gp * kt;
                my[(c.t_gx + 2) * kSamples] = gr * kt;
            }
            named_sync(2, 384);   // gradient parts published (d/du by the G formers, linear term by group 3)
            GT(4)

            // g = quadratic part - linear part; joint L2 clip (TD_Tester.py:150); p -= lr * g (:153-154)
            float ss = 0.f;
            for (int i = 0; i < c.NP; ++i) {
                const float g = my[(c.t_gx + i) * kSamples] - my[(c.t_gl + i) * kSamples];
                my[(c.t_gx + i) * kSamples] = g;
                ss = fmaf(g, g, ss);
            }
            float coef = a.clip / (sqrtf(ss) + 1e-6f);
            coef = coef < 1.0f ? coef : 1.0f;
            for (int i = 0; i < c.NP; ++i)
                my[(c.t_p + i) * kSamples] = __fsub_rn(my[(c.t_p + i) * kSamples], __fmul_rn(a.lr, __fmul_rn(my[(c.t_gx + i) * kSamples], coef)));
            GT(5)   // clip + step
            named_sync(3, 384);   // p stepped: the other groups may read it
        }
        GT_OUT(1)
        if (s0 + row < a.N) {
            float* out = a.P + (s0 + row) * a.ldp;
            for (int i = 0; i < c.NP; ++i) out[i] = my[(c.t_p + i) * kSamples];
        }
    } else if (group == 2) {
        // ===== G formers =====
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegsG));
        float* my = tab + row;
        const uint32_t ypr_plane = (uint32_t)NB * kSamples * 2;   // one FP16 plane
        Ring yb(c.ybufs), gb(c.gbufs);
        GT_DECL
        for (int it = 0; it < a.T; ++it) {
            float cr[RRMAX], dcr[RRMAX], RRv[NDP], dRR[NDP];
            roll_features<RRMAX, NDP>(my[(c.t_p + 2) * kSamples], a.rows_r, c.rr, cr, dcr, RRv, dRR);
            {
                const float w = my[(c.t_p + 1) * kSamples];
                for (int k = 0; k < c.rp; ++k) {
                    const float ra = a.rows_p[4 * k], rb = a.rows_p[4 * k + 1], rc = a.rows_p[4 * k + 2], rd = a.rows_p[4 * k + 3];
                    float s, co;
                    sincos_small(fmaf(rb, w, rc), &s, &co);
                    my[(c.t_cp + k) * kSamples] = fmaf(ra, co, rd);
                    my[(c.t_dcp + k) * kSamples] = -(ra * rb) * s;
                }
            }
            named_sync(1, 384);

            // per-sample, per-iteration power-of-two scale of the YPR operand: the largest |YY_b PP_c RR_d| =
            // (max|cy| max|cp| max|cr|)^2 lands in [2^12, 2^13).  (A fixed scale from the rows' bounds leaves the small
            // products of three monomials in FP16's subnormal range: 0.04 degrees off at T = 3000 on (16,8,8,8).)
            int y_exp;
            float kY;
            {
                float m = 0.f, mp = 0.f, mr = 0.f;
                for (int j = 0; j < c.ry; ++j) m = fmaxf(m, fabsf(my[(c.t_cy + j) * kSamples]));
                for (int k = 0; k < c.rp; ++k) mp = fmaxf(mp, fabsf(my[(c.t_cp + k) * kSamples]));
#pragma unroll
                for (int l = 0; l < RRMAX; ++l) mr = fmaxf(mr, fabsf(cr[l]));
                m = m * mp * mr;
                m *= m;
                int e = 12 - (((__float_as_int(m) >> 23) & 0xff) - 127);
                y_exp = m > 0.f ? max(min(e, 60), -60) : 0;
                kY = __int_as_float((y_exp + 127) << 23);
            }

            float GU[NA16MAX];
#pragma unroll
            for (int i = 0; i < NA16MAX; ++i) GU[i] = 0.f;
            PairWalk pw;
            pw.reset();
            float YY = my[c.t_cy * kSamples] * my[c.t_cy * kSamples];
            int pair = 0;
            // write block jf of the YPR operand (rows = samples, K = the block's columns, UMMA no-swizzle layout)
            auto form = [&]() {
                GT(0)
                ttc::mbar_wait(&aempty[yb.idx], yb.phase ^ 1u);
                GT(1)   // wait operand buffer
                uint8_t* yhi = gsm + c.off_ypr + (size_t)yb.idx * 2 * ypr_plane;
                uint8_t* ylo = yhi + ypr_plane;
                const int rbase = (row / 8) * ((NB / 8) * 128) + (row % 8) * 16;   // ttc::op16_offset(row, k, NB) = rbase + (k/8)*128 + (k%8)*2
                const uint32_t ybase = lane_addr + c.col_y + yb.idx * NB;           // tensor-memory form: NB/2 packed hi columns, then NB/2 lo
                if (c.ypr_tmem) {
                    // the pad columns [BCP * NDP, NB) of this buffer: zero (they multiply zero tile entries, but must be finite)
                    const float z[4] = {0.f, 0.f, 0.f, 0.f};
                    for (int w0 = c.BCP * NDP / 2; w0 < NB / 2; w0 += 4) {
                        tmem_st4(ybase + w0, z);
                        tmem_st4(ybase + NB / 2 + w0, z);
                    }
                }
                for (int pl = 0; pl < c.BCP; ++pl) {
                    float yp = 0.f;
                    if (pair < c.nBC) {
                        yp = YY * (my[(c.t_cp + pw.ci) * kSamples] * my[(c.t_cp + pw.cj) * kSamples]) * kY;
                        ++pair;
                        if (pw.next(c.ry, c.rp) && pw.bi < c.ry)
                            YY = my[(c.t_cy + pw.bi) * kSamples] * my[(c.t_cy + pw.bj) * kSamples];
                    }
                    if (c.ypr_tmem) {
#pragma unroll
                        for (int w0 = 0; w0 < NDP / 2; w0 += 8) {   // NDP/2 packed words per plane: 8 (roll rank <= 5) or 8 + 8 + 4
                            float h[8], l[8];
#pragma unroll
                            for (int e = 0; e < 8; ++e)
                                if (w0 + e < NDP / 2) split_pair16(yp * RRv[2 * (w0 + e)], yp * RRv[2 * (w0 + e) + 1], h[e], l[e]);
                            if (w0 + 8 <= NDP / 2) {
                                tmem_st8(ybase + pl * (NDP / 2) + w0, h);
                                tmem_st8(ybase + NB / 2 + pl * (NDP / 2) + w0, l);
                            } else {
                                tmem_st4(ybase + pl * (NDP / 2) + w0, h);
                                tmem_st4(ybase + NB / 2 + pl * (NDP / 2) + w0, l);
                            }
                        }
                    } else {
#pragma unroll
                        for (int d8 = 0; d8 < NDP / 8; ++d8) {      // one 16-byte chunk = 8 halves of this row per plane
                            float h[4], l[4];
#pragma unroll
                            for (int e = 0; e < 4; ++e) split_pair16(yp * RRv[8 * d8 + 2 * e], yp * RRv[8 * d8 + 2 * e + 1], h[e], l[e]);
                            const int off = rbase + ((pl * NDP) / 8 + d8) * 128;
                            *reinterpret_cast<float4*>(yhi + off) = make_float4(h[0], h[1], h[2], h[3]);
                            *reinterpret_cast<float4*>(ylo + off) = make_float4(l[0], l[1], l[2], l[3]);
                        }
                    }
                }
                GT(2)   // form
                if (c.ypr_tmem) {
                    tmem_store_wait();
                    tc_before();
                } else {
                    ttc::fence_async_smem();
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&afull[yb.idx]);
                yb.next();
                GT(3)   // fence + arrive
            };
            form();
            for (int j = 0; j < nblocks; ++j, gb.next()) {
                if (j + 1 < nblocks) form();
                // promote this block's partial D_G into the FP32 accumulators (round-to-nearest adds)
                GT(0)
                ttc::mbar_wait(&gfull[gb.idx], gb.phase);
                GT(4)   // wait D_G
                tc_after();
                const uint32_t gbase = lane_addr + c.col_g + gb.idx * NA16;
#pragma unroll
                for (int x0 = 0; x0 < NA16MAX / 8; x0 += 4) {
                    if (8 * x0 < NA16) {
                        uint32_t v[32];
#pragma unroll
                        for (int x = 0; x < 4; ++x)
                            if (x0 + x < NA16MAX / 8 && 8 * (x0 + x) < NA16) tmem_ld8(gbase + 8 * (x0 + x), v + 8 * x);
                        tmem_load_wait();
#pragma unroll
                        for (int x = 0; x < 4; ++x)
                            if (x0 + x < NA16MAX / 8 && 8 * (x0 + x) < NA16) {
#pragma unroll
                                for (int e = 0; e < 8; ++e) GU[8 * (x0 + x) + e] += __uint_as_float(v[8 * x + e]);
                            }
                    }
                }
                tc_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&gempty[gb.idx]);
                GT(5)   // promote
            }
            // d/du_m of sum_A GU_A UU_A: for the pair A = (i,j): i == j -> 2 GU u_i, else GU u_j to i and GU u_i to j
            for (int i = 0; i < c.ri; ++i) my[(c.t_gx + 3 + i) * kSamples] = 0.f;
            {
                const float kg = __int_as_float((127 - c.s_exp - y_exp) << 23);   // 2^-(s_exp + y_exp): the D_G accumulators' scale off
                int i = 0, j = 0;
#pragma unroll
                for (int A = 0; A < NA16MAX; ++A) {
                    if (A < c.nA) {
                        const float ui = my[(c.t_p + 3 + i) * kSamples] * kg, uj = my[(c.t_p + 3 + j) * kSamples] * kg;
                        if (i == j) {
                            my[(c.t_gx + 3 + i) * kSamples] += 2.0f * GU[A] * ui;
                        } else {
                            my[(c.t_gx + 3 + i) * kSamples] += GU[A] * uj;
                            my[(c.t_gx + 3 + j) * kSamples] += GU[A] * ui;
                        }
                        if (++j == c.ri) { ++i; j = i; }
                    }
                }
            }
            GT(6)   // d/du
            named_sync(2, 384);
            named_sync(3, 384);
            GT(7)
        }
        GT_OUT(2)
    } else {
        // ===== linear term: F1 = -sum q[ijkl] u_i cy_j cp_k cr_l and its derivatives =====
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegsL));
        float* my = tab + row;
        const float* __restrict__ q = a.q + (size_t)blockIdx.x * c.R * kSamples + row;
        GT_DECL
        for (int it = 0; it < a.T; ++it) {
            float cr[RRMAX], dcr[RRMAX];
#pragma unroll
            for (int l = 0; l < RRMAX; ++l) {
                float s = 0.f, co = 0.f;
                cr[l] = 0.f;
                dcr[l] = 0.f;
                if (l < c.rr) {
                    const float ra = a.rows_r[4 * l], rb = a.rows_r[4 * l + 1], rc = a.rows_r[4 * l + 2], rd = a.rows_r[4 * l + 3];
                    sincos_small(fmaf(rb, my[(c.t_p + 2) * kSamples], rc), &s, &co);
                    cr[l] = fmaf(ra, co, rd);
                    dcr[l] = -(ra * rb) * s;
                }
            }
            named_sync(1, 384);
            GT(0)
            float ly = 0.f, lp = 0.f, lr_ = 0.f;
            const float* qi = q;
            const int blk_lines = c.rp * c.rr * 4;   // one (i,j) block of the slab = rp*rr rows of 128 floats = 4 lines each
            for (int i = 0; i < c.ri; ++i) {
                float lin = 0.f, gyi = 0.f, gpi = 0.f, gri = 0.f;
                for (int j = 0; j < c.ry; ++j) {
                    // the NEXT (i,j) block into L1 while this one is contracted: the group's 128 threads touch its lines once, so
                    // the loads below hit L1 instead of paying the L2 round trip twice per block (they are the group's critical path)
                    if (i * c.ry + j + 1 < c.ri * c.ry) {
                        const float* nxt = (qi - row) + (size_t)(blk_lines / 4) * kSamples;
                        for (int t = row; t < blk_lines; t += kSamples)
                            asm volatile("prefetch.global.L1 [%0];" ::"l"(nxt + (size_t)(t >> 2) * kSamples + (t & 3) * 32));
                    }
                    float A0 = 0.f, A1 = 0.f, A2 = 0.f;
#pragma unroll 4
                    for (int k = 0; k < c.rp; ++k) {
                        float s = 0.f, sd = 0.f;
#pragma unroll
                        for (int l = 0; l < RRMAX; ++l)
                            if (l < c.rr) {
                                const float qv = __ldg(qi + (size_t)(k * c.rr + l) * kSamples);
                                s = fmaf(qv, cr[l], s);
                                sd = fmaf(qv, dcr[l], sd);
                            }
                        const float cpk = my[(c.t_cp + k) * kSamples], dpk = my[(c.t_dcp + k) * kSamples];
                        A0 = fmaf(cpk, s, A0);
                        A1 = fmaf(dpk, s, A1);
                        A2 = fmaf(cpk, sd, A2);
                    }
                    qi += (size_t)c.rp * c.rr * kSamples;
                    const float cyj = my[(c.t_cy + j) * kSamples], dyj = my[(c.t_dcy + j) * kSamples];
                    lin = fmaf(cyj, A0, lin);
                    gyi = fmaf(dyj, A0, gyi);
                    gpi = fmaf(cyj, A1, gpi);
                    gri = fmaf(cyj, A2, gri);
                }
                const float ui = my[(c.t_p + 3 + i) * kSamples];
                my[(c.t_gl + 3 + i) * kSamples] = lin;
                ly = fmaf(ui, gyi, ly);
                lp = fmaf(ui, gpi, lp);
                lr_ = fmaf(ui, gri, lr_);
            }
            my[(c.t_gl + 0) * kSamples] = ly;
            my[(c.t_gl + 1) * kSamples] = lp;
            my[(c.t_gl + 2) * kSamples] = lr_;
            GT(1)   // linear term
            named_sync(2, 384);
            named_sync(3, 384);
        }
        GT_OUT(3)
    }
    tc_before();
    __syncthreads();
    if (warp == 1) tmem_free_cols(tmem, 512);
}

// q = W2 x for a batch, written as the CTA-blocked slabs the generic kernel reads: Q[(s / 128) * R + r][s % 128].
// Plain FP32 tiled GEMM (128 samples x 64 rows of W2 per block, 16 features per step): one pass, ~1 % of a T = 3000 fit.
// ipd: the X rows are raw landmarks; the block derives its 128 rows' (ref, ipd) once and applies the IPD normalisation
// (common.cuh) to each staged X tile.
__global__ void __launch_bounds__(256) tucker_project_kernel(const float* __restrict__ X, long long N, long long ldx,
                                                            const float* __restrict__ W2, int R, int F, int vec_ok,
                                                            float* __restrict__ Q, int ipd) {
    constexpr int BM = 128, BR = 64, BK = 16;
    __shared__ __align__(16) float Xs[BK][BM + 4];
    __shared__ __align__(16) float Ws[BK][BR + 4];
    extern __shared__ IpdRow ipd_s[];   // [BM], launched with sizeof(IpdRow) * BM bytes of dynamic shared memory when ipd
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;   // tx: 16 sample groups (sample = tx + 16 i), ty: 16 row groups of 4
    const long long m0 = (long long)blockIdx.x * BM;
    const int r0 = blockIdx.y * BR;
    if (ipd) {
        if (tid < BM && m0 + tid < N) ipd_s[tid] = ipd_row(X + (m0 + tid) * ldx);
        __syncthreads();
    }
    float acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int f0 = 0; f0 < F; f0 += BK) {
        for (int idx = tid; idx < BM * (BK / 4); idx += 256) {
            const int s = idx >> 2, c4 = idx & 3;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (m0 + s < N) {
                const float* src = X + (m0 + s) * ldx;
                const int f = f0 + 4 * c4;
                if (vec_ok && f + 3 < F) v = __ldg(reinterpret_cast<const float4*>(src + f));
                else {
                    if (f + 0 < F) v.x = __ldg(src + f + 0);
                    if (f + 1 < F) v.y = __ldg(src + f + 1);
                    if (f + 2 < F) v.z = __ldg(src + f + 2);
                    if (f + 3 < F) v.w = __ldg(src + f + 3);
                }
            }
            Xs[4 * c4 + 0][s] = v.x; Xs[4 * c4 + 1][s] = v.y; Xs[4 * c4 + 2][s] = v.z; Xs[4 * c4 + 3][s] = v.w;
        }
        for (int idx = tid; idx < BR * (BK / 4); idx += 256) {
            const int r = idx >> 2, c4 = idx & 3;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r0 + r < R) {
                const float* src = W2 + (long long)(r0 + r) * F;
                const int f = f0 + 4 * c4;
                if ((F % 4 == 0) && f + 3 < F) v = __ldg(reinterpret_cast<const float4*>(src + f));
                else {
                    if (f + 0 < F) v.x = __ldg(src + f + 0);
                    if (f + 1 < F) v.y = __ldg(src + f + 1);
                    if (f + 2 < F) v.z = __ldg(src + f + 2);
                    if (f + 3 < F) v.w = __ldg(src + f + 3);
                }
            }
            Ws[4 * c4 + 0][r] = v.x; Ws[4 * c4 + 1][r] = v.y; Ws[4 * c4 + 2][r] = v.z; Ws[4 * c4 + 3][r] = v.w;
        }
        __syncthreads();
        if (ipd) {
            ipd_tile(&Xs[0][0], BM + 4, BK, BM, ipd_s, N - m0, f0, F, tid, 256);
            __syncthreads();
        }
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            float xv[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) xv[i] = Xs[k][tx + 16 * i];
            const float4 w = *reinterpret_cast<const float4*>(&Ws[k][4 * ty]);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                acc[i][0] = fmaf(xv[i], w.x, acc[i][0]);
                acc[i][1] = fmaf(xv[i], w.y, acc[i][1]);
                acc[i][2] = fmaf(xv[i], w.z, acc[i][2]);
                acc[i][3] = fmaf(xv[i], w.w, acc[i][3]);
            }
        }
        __syncthreads();
    }
    float* slab = Q + (size_t)blockIdx.x * R * BM;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int r = r0 + 4 * ty + j;
        if (r < R) {
#pragma unroll
            for (int i = 0; i < 8; ++i) slab[(size_t)r * BM + tx + 16 * i] = acc[i][j];   // rows beyond N hold 0 (x = 0)
        }
    }
}

// Tile images of the folded Gram tensor: for block j the T tile [NB cols][KA] and the G tile [NA16][NB cols], each as a
// FP16 hi plane followed by a lo plane (S times 2^s_exp) in the UMMA no-swizzle K-major layout (ttc::op16_offset).  Column col = pair * NDP + dd:
// pair = b * nC + c, dd = pair_index(i, j, rrmax) of the roll pair (entries with j >= rr are zero).
__global__ void build_tiles_kernel(const float* __restrict__ S, int NAP, GenCfg c, uint8_t* __restrict__ tiles) {
    const int nD = tri(c.rr);
    const float s_scale = __int_as_float((127 + c.s_exp) << 23);
    const long long per_block = (long long)c.NB * c.KA + (long long)c.NA16 * c.NB;
    const long long total = per_block * c.nblocks;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int blk = (int)(idx / per_block);
        long long e = idx % per_block;
        const bool is_t = e < (long long)c.NB * c.KA;
        int A, col;
        if (is_t) { col = (int)(e / c.KA); A = (int)(e % c.KA); }
        else { e -= (long long)c.NB * c.KA; A = (int)(e / c.NB); col = (int)(e % c.NB); }
        const int pair = blk * c.BCP + col / c.nDp, dd = col % c.nDp;
        float v = 0.f;
        if (A < c.nA && col < c.BCP * c.nDp && pair < c.nBC && dd < tri(c.rrmax)) {
            int i, j;
            unpair(dd, c.rrmax, &i, &j);
            if (j < c.rr) v = S[((long long)pair * nD + pair_index(i, j, c.rr)) * NAP + A];
        }
        __half hi, lo;
        ttc::split_half(v * s_scale, hi, lo);
        uint8_t* base = tiles + (size_t)blk * ((size_t)c.tt_bytes + c.gt_bytes);
        if (is_t) {
            const int off = ttc::op16_offset(col, A, c.KA);
            *reinterpret_cast<__half*>(base + off) = hi;
            *reinterpret_cast<__half*>(base + c.tt_bytes / 2 + off) = lo;
        } else {
            const int off = ttc::op16_offset(A, col, c.NB);
            *reinterpret_cast<__half*>(base + c.tt_bytes + off) = hi;
            *reinterpret_cast<__half*>(base + c.tt_bytes + c.gt_bytes / 2 + off) = lo;
        }
    }
}

// 64 x 64 tiles of M = W2 W2^T in float64 (plan creation for large cores: R up to 8192)
__global__ void __launch_bounds__(256) gram_tiled_kernel(const float* __restrict__ W2, int R, int F, double* __restrict__ M) {
    if (blockIdx.x < blockIdx.y) return;   // symmetric: upper block triangle, mirrored on write
    constexpr int BT = 64, BK = 16;
    __shared__ float As[BK][BT + 1], Bs[BK][BT + 1];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int r0 = blockIdx.y * BT, c0 = blockIdx.x * BT;
    double acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
    for (int f0 = 0; f0 < F; f0 += BK) {
        for (int idx = tid; idx < BT * BK; idx += 256) {
            const int r = idx / BK, k = idx % BK;
            As[k][r] = (r0 + r < R && f0 + k < F) ? __ldg(W2 + (long long)(r0 + r) * F + f0 + k) : 0.f;
            Bs[k][r] = (c0 + r < R && f0 + k < F) ? __ldg(W2 + (long long)(c0 + r) * F + f0 + k) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            double av[4], bv[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) { av[i] = (double)As[k][ty + 16 * i]; bv[i] = (double)Bs[k][tx + 16 * i]; }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fma(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int r = r0 + ty + 16 * i, cc = c0 + tx + 16 * j;
            if (r < R && cc < R) {
                M[(long long)r * R + cc] = acc[i][j];
                M[(long long)cc * R + r] = acc[i][j];
            }
        }
}

}  // namespace tgen
}  // namespace nlml
