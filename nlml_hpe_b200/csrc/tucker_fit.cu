// Batched Tucker fit for sm_100a: the fixed-iteration fit of TD_Tester.optimize_with_sgd
// (/root/reference/TD_Tester.py:127-159) and the converged fit TD_Tester.Test searches for (:191-199), for a whole
// batch of feature vectors.  Same arithmetic everywhere (tucker_math.h); kernels chosen by batch size and ranks:
//
//   tucker_fit_tc_kernel   the default from 1536 samples: 128 samples per CTA, two threads per sample; the two
//                          contractions with the folded Gram tensor run as FP16 hi/lo tcgen05 GEMMs (FP32-grade),
//                          tensor memory holds the accumulators, each sample's q = W2 x and one MMA operand;
//                          q comes from tucker_project_tc_kernel (3xTF32 tcgen05 GEMM) for batches of 4096+ rows.
//   tucker_fit_gen_kernel  the same formulation for run-time ranks (tucker_gen.cuh): enlarged cores.
//   tucker_fit_tps_kernel  thread-per-sample, FP32 only, ranks fixed at compile time (5,3,3,3 = the shipped /
//                          configured ranks, configs/config_TD_main.yaml:8-13).  A CTA owns THREADS consecutive
//                          samples: phase A streams their rows of X once from HBM and leaves q in shared memory;
//                          phase B runs all T iterations with p, the monomials and the gradient in registers, the
//                          folded Gram tensor S broadcast from shared memory.  Its SOLVE variant runs the damped-Newton
//                          converged fit instead of the T iterations.
//   tucker_fit_wps_kernel  warp-per-sample: small batches and the single-image case of TD_Inference.py, where the
//                          latency of the 3000-step chain matters more than throughput.
//   tucker_fit_cta_kernel  CTA-per-sample, ranks at run time, FP32: tiny batches of other rank sets, roll rank > 8.
// No kernel touches global memory between iterations.
#include <cuda.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "common.cuh"
#include "tucker_math.h"
#include "powell_math.h"

namespace nlml {

constexpr int kMaxModeRank = 16;
constexpr int kMaxPairs = kMaxModeRank * (kMaxModeRank + 1) / 2;  // 136
constexpr int kMaxBCD = 8192;                                    // CTA kernel keeps T[] and ypr[] in shared memory

struct TuckerArgs {
    const float* X;
    long long N, ldx;
    const float* W2;  // [R][F]
    const float* S;   // [nBCD][NAP]   thread-per-sample layout
    const float* St;  // [nA][nBCDp]   CTA-per-sample layout
    const uint8_t* tc_ops;   // tensor-core kernel: shared-memory image of the two B operands (S in both GEMM views, hi/lo)
    int s_exp;               // tensor-core kernel: its S operand image holds S * 2^s_exp
    int pr_exp;              // ... and the PP (x) RR operand is written times 2^pr_exp (from the bound (|a|+|d|)^4 of the pitch / roll rows)
    const float* Qpre;       // q = W2 x precomputed by tucker_project_tc_kernel, CTA-blocked [N/128][RPAD][128]; null: phase A runs here
    float* P;
    long long ldp;
    int F, T;
    float lr, clip;
    int ri, ry, rp, rr;
    int nBCDp;
    int vec_ok;  // X rows and W2 rows are 16-byte aligned and F % 4 == 0
    int ipd;     // X rows are raw landmarks: phase A reads them through the IPD normalisation (common.cuh)
#ifdef NLML_TC_DBG
    int dbg;     // development build only (-DNLML_TC_DBG): tensor-core kernel 1 = no MMAs / waits, 2 = no TMEM consumption
#endif
    LmOptions lm;   // converged solve only
    int* evals;     // converged solve only: optional [N] evaluations used per sample
    float rows_y[4 * kMaxModeRank], rows_p[4 * kMaxModeRank], rows_r[4 * kMaxModeRank];
};

// ---------------------------------------------------------------------------------------------
// one-time constant preparation
// ---------------------------------------------------------------------------------------------
__global__ void gram_kernel(const float* __restrict__ W2, int R, int F, double* __restrict__ M) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= R * R) return;
    const int r = idx / R, c = idx % R;
    if (c < r) return;  // symmetric: compute the upper triangle, mirror
    const double v = gram_entry(W2, F, r, c);
    M[(long long)r * R + c] = v;
    M[(long long)c * R + r] = v;
}

__global__ void fold_kernel(const double* __restrict__ M, int ri, int ry, int rp, int rr, int NAP, int nBCDp,
                            float* __restrict__ S, float* __restrict__ St) {
    const int nA = tri(ri), nB = tri(ry), nC = tri(rp), nD = tri(rr);
    const int nBCD = nB * nC * nD;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= nA * nBCD) return;
    const int a = idx / nBCD, bcd = idx % nBCD;
    const int b = bcd / (nC * nD), c = (bcd / nD) % nC, d = bcd % nD;
    const float v = fold_entry(M, ri, ry, rp, rr, a, b, c, d);
    S[(long long)bcd * NAP + a] = v;
    St[(long long)a * nBCDp + bcd] = v;
}

// ---------------------------------------------------------------------------------------------
// tensor memory as per-thread storage: a thread of warp w owns TMEM lane 32*(w%4) + laneid and reads / writes
// 32 consecutive columns of it per instruction (tcgen05.ld/st .32x32b.x32)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc_cols(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_free_cols(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_load32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
// same load without the wait: the caller overlaps it with arithmetic and calls tmem_load_wait() before touching r[]
__device__ __forceinline__ void tmem_load32_async(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_load_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_store32(uint32_t taddr, const float* v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
          "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
          "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
          "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15])),
          "r"(__float_as_uint(v[16])), "r"(__float_as_uint(v[17])), "r"(__float_as_uint(v[18])), "r"(__float_as_uint(v[19])),
          "r"(__float_as_uint(v[20])), "r"(__float_as_uint(v[21])), "r"(__float_as_uint(v[22])), "r"(__float_as_uint(v[23])),
          "r"(__float_as_uint(v[24])), "r"(__float_as_uint(v[25])), "r"(__float_as_uint(v[26])), "r"(__float_as_uint(v[27])),
          "r"(__float_as_uint(v[28])), "r"(__float_as_uint(v[29])), "r"(__float_as_uint(v[30])), "r"(__float_as_uint(v[31]))
        : "memory");
}
__device__ __forceinline__ void tmem_store4(uint32_t taddr, const float* v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};"
                 ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3]))
                 : "memory");
}
__device__ __forceinline__ void tmem_store_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// q accessor for the TMEM-resident variant (same interface as QStrided in tucker_math.h)
struct QTmem {
    uint32_t taddr;   // this thread's lane, first column of its q
    template <int R0, int CNT>
    __device__ __forceinline__ void load(int /*n*/, float (&v)[32]) const { tmem_load32(taddr + R0, v); }
};

}  // namespace nlml
#include "tucker_tc.cuh"
#include "tucker_gen.cuh"
namespace nlml {

// ---------------------------------------------------------------------------------------------
// thread-per-sample kernel
// ---------------------------------------------------------------------------------------------
// QTMEM: keep q in tensor memory instead of shared memory.  q is what limits the SM to 8 resident warps
// (69 KB per 128 samples); in TMEM (unused by this kernel otherwise) a 384-thread CTA fits and 12 warps hide the
// FMA / shared-memory latencies of the iteration better.
template <int RI, int RY, int RP, int RR, int THREADS, int NS, bool QTMEM = false>
struct TpsCfg {
    static constexpr int R = RI * RY * RP * RR;
    static constexpr int RPAD = (R + 3) / 4 * 4;
    static constexpr int NP = 3 + RI;
    static constexpr int nA = tri(RI);
    static constexpr int NAP = (nA + 3) / 4 * 4;
    static constexpr int nBCD = tri(RY) * tri(RP) * tri(RR);
    static constexpr int FC = 16;              // feature columns per staged tile
    static constexpr int XSTR = THREADS + 2;   // == 2 (mod 8): transposed tile stores are conflict-free
    static constexpr int S_FLOATS = nBCD * NAP;
    static constexpr int SAMPLES = THREADS * NS;   // samples per CTA; thread t owns samples t, t+THREADS, ...
    static constexpr int Q_FLOATS = QTMEM ? 0 : R * SAMPLES;   // [NS][R][THREADS] (shared-memory variant)
    static constexpr int QCOLS = (RPAD + 31) / 32 * 32;        // TMEM columns per thread (TMEM variant)
    static constexpr int TMEM_COLS = 512;
    static_assert(!QTMEM || (NS == 1 && (THREADS / 128) * QCOLS <= TMEM_COLS && THREADS % 128 == 0), "TMEM budget");
    static constexpr int SCR_FLOATS = tri(RY) * tri(RP) * SAMPLES;  // [NS][nB*nC][THREADS] scratch of tucker_gradient
    static constexpr int TILE_FLOATS = FC * XSTR + FC * RPAD;

    static_assert(!QTMEM || TILE_FLOATS <= SCR_FLOATS, "phase-A tiles alias the scratch buffer in the TMEM variant");
    // raw-landmark input: the (ref, ipd) of the pass's THREADS rows live in the scratch buffer during phase A (after the
    // tiles in the TMEM variant)
    static constexpr int IPD_OFF = QTMEM ? (TILE_FLOATS + 1) / 2 * 2 : 0;
    static_assert(IPD_OFF * 4 + THREADS * sizeof(IpdRow) <= SCR_FLOATS * 4, "IPD constants fit the scratch buffer");
    static constexpr size_t SMEM_BYTES = sizeof(float) * (S_FLOATS + Q_FLOATS + SCR_FLOATS) + 16;
};

__device__ __forceinline__ float4 load_row4(const float* __restrict__ row, int f, int F, bool vec_ok) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (vec_ok && f + 3 < F) {
        v = __ldg(reinterpret_cast<const float4*>(row + f));
    } else {
        if (f + 0 < F) v.x = __ldg(row + f + 0);
        if (f + 1 < F) v.y = __ldg(row + f + 1);
        if (f + 2 < F) v.z = __ldg(row + f + 2);
        if (f + 3 < F) v.w = __ldg(row + f + 3);
    }
    return v;
}

// SOLVE: phase B is the converged damped-Newton solve (tucker_lm_solve) instead of the T fixed iterations.
template <int RI, int RY, int RP, int RR, int THREADS, int NS, int MINB, bool QTMEM, bool SOLVE = false>
__global__ void __launch_bounds__(THREADS, MINB) tucker_fit_tps_kernel(const __grid_constant__ TuckerArgs a) {
    using C = TpsCfg<RI, RY, RP, RR, THREADS, NS, QTMEM>;
    extern __shared__ __align__(16) float smem[];
    float* S_s = smem;
    float* q_s = smem + C::S_FLOATS;
    float* scr_s = q_s + C::Q_FLOATS;
    float* xs = q_s;                     // [FC][XSTR]   (phase A only)
    float* ws = q_s + C::FC * C::XSTR;   // [FC][RPAD]   (phase A only)
    static_assert(C::TILE_FLOATS <= C::R * THREADS, "phase-A tiles must fit inside one sample slab of q");
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(scr_s + C::SCR_FLOATS);
    uint32_t q_taddr = 0;
    if constexpr (QTMEM) {
        if (threadIdx.x < 32) tmem_alloc_cols(tmem_slot, C::TMEM_COLS);
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int w = threadIdx.x >> 5;
        q_taddr = *tmem_slot + ((uint32_t)((w & 3) * 32) << 16) + (uint32_t)((w >> 2) * C::QCOLS);
    }

    const int tid = threadIdx.x;
    const long long s0 = (long long)blockIdx.x * C::SAMPLES;
    const bool vec_ok = a.vec_ok != 0;
    const int F = a.F;

    // S is broadcast from shared memory.  (Measured alternative: S in the kernel parameters, read through the
    // constant path with LDC c[0x0][R+off], ran at 473 k-602 k poses/s against 913 k.)
    for (int i = tid; i < C::S_FLOATS / 4; i += THREADS)
        reinterpret_cast<float4*>(S_s)[i] = __ldg(reinterpret_cast<const float4*>(a.S) + i);

    // ---- phase A: q[r] = sum_f W2[r][f] * x[f], one pass per sample owned by this thread ----
    // (the tiles alias the q buffer of the pass in flight only: pass n stages its tiles in q slab n)
    if constexpr (THREADS == 128 && NS == 1 && !QTMEM) {
        if (a.Qpre) {   // projected already by the tensor-core GEMM (tucker_project_tc_kernel): coalesced copy of this CTA's slab
            const float* slab = a.Qpre + (size_t)blockIdx.x * C::RPAD * 128;
            for (int r = 0; r < C::R; ++r) q_s[r * THREADS + tid] = __ldg(slab + r * 128 + tid);
        }
    }
    const int n_passes = (THREADS == 128 && NS == 1 && !QTMEM && a.Qpre) ? 0 : NS;
#pragma unroll 1
    for (int n = 0; n < n_passes; ++n) {
    float* qn_s = QTMEM ? scr_s : q_s + n * (C::R * THREADS);   // TMEM variant: tiles live in the scratch buffer
    xs = qn_s;
    ws = qn_s + C::FC * C::XSTR;
    IpdRow* ipd_s = reinterpret_cast<IpdRow*>(scr_s + C::IPD_OFF);
    if (a.ipd) {   // raw landmarks: each row's (ref, ipd) once per pass, applied to the staged tiles below
        const long long row = s0 + n * THREADS + tid;
        if (row < a.N) ipd_s[tid] = ipd_row(a.X + row * a.ldx);
        __syncthreads();
    }
    float acc[C::RPAD];
#pragma unroll
    for (int r = 0; r < C::RPAD; ++r) acc[r] = 0.f;

    for (int f0 = 0; f0 < F; f0 += C::FC) {
        for (int idx = tid; idx < THREADS * (C::FC / 4); idx += THREADS) {
            const int s = idx / (C::FC / 4), c4 = idx % (C::FC / 4);
            const long long row = s0 + n * THREADS + s;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (row < a.N) v = load_row4(a.X + row * a.ldx, f0 + 4 * c4, F, vec_ok);
            xs[(4 * c4 + 0) * C::XSTR + s] = v.x;
            xs[(4 * c4 + 1) * C::XSTR + s] = v.y;
            xs[(4 * c4 + 2) * C::XSTR + s] = v.z;
            xs[(4 * c4 + 3) * C::XSTR + s] = v.w;
        }
        for (int idx = tid; idx < C::RPAD * (C::FC / 4); idx += THREADS) {
            const int r = idx / (C::FC / 4), c4 = idx % (C::FC / 4);
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r < C::R) v = load_row4(a.W2 + (long long)r * F, f0 + 4 * c4, F, vec_ok);
            ws[(4 * c4 + 0) * C::RPAD + r] = v.x;
            ws[(4 * c4 + 1) * C::RPAD + r] = v.y;
            ws[(4 * c4 + 2) * C::RPAD + r] = v.z;
            ws[(4 * c4 + 3) * C::RPAD + r] = v.w;
        }
        __syncthreads();
        if (a.ipd) {
            ipd_tile(xs, C::XSTR, C::FC, THREADS, ipd_s, a.N - (s0 + n * THREADS), f0, F, tid, THREADS);
            __syncthreads();
        }
#pragma unroll 4
        for (int f = 0; f < C::FC; ++f) {
            const float xv = xs[f * C::XSTR + tid];
#pragma unroll
            for (int r4 = 0; r4 < C::RPAD / 4; ++r4) {
                const float4 w = *reinterpret_cast<const float4*>(&ws[f * C::RPAD + 4 * r4]);
                acc[4 * r4 + 0] = fmaf(xv, w.x, acc[4 * r4 + 0]);
                acc[4 * r4 + 1] = fmaf(xv, w.y, acc[4 * r4 + 1]);
                acc[4 * r4 + 2] = fmaf(xv, w.z, acc[4 * r4 + 2]);
                acc[4 * r4 + 3] = fmaf(xv, w.w, acc[4 * r4 + 3]);
            }
        }
        __syncthreads();
    }
    if constexpr (QTMEM) {
#pragma unroll
        for (int c = 0; c < C::QCOLS / 32; ++c) {
            float v[32];
#pragma unroll
            for (int x = 0; x < 32; ++x) v[x] = (32 * c + x < C::RPAD) ? acc[(32 * c + x < C::RPAD) ? 32 * c + x : 0] : 0.f;
            tmem_store32(q_taddr + 32 * c, v);
        }
        tmem_store_wait();
    } else {
#pragma unroll
        for (int r = 0; r < C::R; ++r) qn_s[r * THREADS + tid] = acc[r];
    }
    __syncthreads();  // S_s complete, tiles dead
    }
    if (n_passes == 0) __syncthreads();   // S_s and the copied q slab complete

    if constexpr (SOLVE) {
        // ---- phase B': converged fit, data-dependent number of Newton evaluations per sample ----
        static_assert(!SOLVE || (NS == 1 && !QTMEM), "the solve variant keeps one sample per thread with q in shared memory");
        static_assert(!SOLVE || 3 * (tri(RY) + tri(RP)) <= tri(RY) * tri(RP), "scratch column too small for the solve");
        float ps[C::NP], Lf;
        const int evals = tucker_lm_solve<RI, RY, RP, RR, C::NAP>(S_s, q_s + tid, THREADS, scr_s + tid, THREADS, a.rows_y,
                                                                  a.rows_p, a.rows_r, a.lm, ps, Lf);
        const long long row = s0 + tid;
        if (row < a.N) {
            float* out = a.P + row * a.ldp;
#pragma unroll
            for (int i = 0; i < C::NP; ++i) out[i] = ps[i];
            if (a.evals) a.evals[row] = evals;
        }
        return;
    }

    // ---- phase B: T iterations entirely on chip ----
    float p[NS][C::NP];
#pragma unroll
    for (int n = 0; n < NS; ++n)
#pragma unroll
        for (int i = 0; i < C::NP; ++i) p[n][i] = 0.f;  // zero init, TD_Tester.py:130
    const float lr = a.lr, clip = a.clip;
#pragma unroll 1
    for (int it = 0; it < a.T; ++it) {
        float g[NS][C::NP];
        if constexpr (QTMEM)
            tucker_gradient<RI, RY, RP, RR, C::NAP, NS>(p, S_s, QTmem{q_taddr}, scr_s + tid, THREADS,
                                                        tri(RY) * tri(RP) * THREADS, a.rows_y, a.rows_p, a.rows_r, g);
        else
            tucker_gradient<RI, RY, RP, RR, C::NAP, NS>(p, S_s, QStrided{q_s + tid, THREADS, C::R * THREADS}, scr_s + tid, THREADS,
                                                        tri(RY) * tri(RP) * THREADS, a.rows_y, a.rows_p, a.rows_r, g);
#pragma unroll
        for (int n = 0; n < NS; ++n) clip_and_step<C::NP>(p[n], g[n], lr, clip);
    }
#pragma unroll
    for (int n = 0; n < NS; ++n) {
        const long long row = s0 + n * THREADS + tid;
        if (row < a.N) {
            float* out = a.P + row * a.ldp;
#pragma unroll
            for (int i = 0; i < C::NP; ++i) out[i] = p[n][i];
        }
    }
    if constexpr (QTMEM) {
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (threadIdx.x < 32) tmem_free_cols(*tmem_slot, C::TMEM_COLS);
    }
}

// ---------------------------------------------------------------------------------------------
// CTA-per-sample kernel (run-time ranks)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

struct CtaLayout {
    // offsets in floats into dynamic shared memory
    int x, q, T, ypr, fac, dfac, prod, G, lin, p, pairs, St, total;
};

__host__ __device__ inline CtaLayout cta_layout(int F, int R, int nBCD, int nA, int nBCDp, bool st_in_smem) {
    CtaLayout L;
    int o = 0;
    auto take = [&](int n) { int r = o; o += (n + 3) / 4 * 4; return r; };
    L.x = take(F);
    L.q = take(R);
    L.T = take(nBCD);
    L.ypr = take(nBCD);
    L.fac = take(4 * kMaxModeRank);
    L.dfac = take(4 * kMaxModeRank);
    L.prod = take(4 * kMaxPairs);
    L.G = take(4 * kMaxPairs);
    L.lin = take(4 * kMaxModeRank);
    L.p = take(2 * (3 + kMaxModeRank));
    L.pairs = take(4 * kMaxPairs);  // packed (i | j<<8) per mode, stored as int
    L.St = take(st_in_smem ? nA * nBCDp : 0);
    L.total = o;
    return L;
}

template <int THREADS>
__global__ void __launch_bounds__(THREADS) tucker_fit_cta_kernel(const __grid_constant__ TuckerArgs a, int st_in_smem) {
    extern __shared__ __align__(16) float smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = THREADS / 32;
    const int dims[4] = {a.ri, a.ry, a.rp, a.rr};
    const int R = a.ri * a.ry * a.rp * a.rr;
    const int nP[4] = {tri(a.ri), tri(a.ry), tri(a.rp), tri(a.rr)};
    const int nA = nP[0], nB = nP[1], nC = nP[2], nD = nP[3];
    const int nBCD = nB * nC * nD, nBCDp = a.nBCDp;
    const int NP = 3 + a.ri;
    const int F = a.F;
    const CtaLayout L = cta_layout(F, R, nBCD, nA, nBCDp, st_in_smem != 0);
    float* xb = smem + L.x;
    float* q = smem + L.q;
    float* Tb = smem + L.T;
    float* ypr = smem + L.ypr;
    float* fac = smem + L.fac;    // [4][kMaxModeRank]: u, cy, cp, cr
    float* dfac = smem + L.dfac;  // [4][kMaxModeRank]: -, dcy, dcp, dcr
    float* prod = smem + L.prod;  // [4][kMaxPairs]: UU, YY, PP, RR
    float* G = smem + L.G;        // [4][kMaxPairs]: GU, GY, GP, GR
    float* lin = smem + L.lin;    // [4][kMaxModeRank]: d(q.z)/d(factor entry)
    float* p = smem + L.p;
    int* pairs = reinterpret_cast<int*>(smem + L.pairs);
    const float* St = a.St;

    const long long s = blockIdx.x;
    const float* xrow = a.X + s * a.ldx;
    if (a.ipd) {   // raw landmarks: every thread derives the row's (ref, ipd) from the same nine L1-resident values
        const IpdRow nr = ipd_row(xrow);
        for (int f = tid; f < F; f += THREADS) xb[f] = ipd_map(__ldg(xrow + f), nr, f % 3);
    } else {
        for (int f = tid; f < F; f += THREADS) xb[f] = __ldg(xrow + f);
    }
    for (int idx = tid; idx < 4 * kMaxPairs; idx += THREADS) {
        const int m = idx / kMaxPairs, k = idx % kMaxPairs;
        int i = 0, j = 0;
        if (k < nP[m]) unpair(k, dims[m], &i, &j);
        pairs[idx] = i | (j << 8);
    }
    if (st_in_smem) {
        float* St_s = smem + L.St;
        for (int i = tid; i < nA * nBCDp; i += THREADS) St_s[i] = __ldg(a.St + i);
        St = St_s;
    }
    if (tid < 2 * (3 + kMaxModeRank)) p[tid] = 0.f;  // zero init, TD_Tester.py:130
    __syncthreads();

    // phase A: q = W2 x, one warp per row
    for (int r = warp; r < R; r += NW) {
        const float* wrow = a.W2 + (long long)r * F;
        float acc = 0.f;
        if (a.vec_ok) {
            for (int f = 4 * lane; f < F; f += 128) {
                const float4 w = __ldg(reinterpret_cast<const float4*>(wrow + f));
                const float4 x = *reinterpret_cast<const float4*>(xb + f);
                acc = fmaf(w.x, x.x, acc);
                acc = fmaf(w.y, x.y, acc);
                acc = fmaf(w.z, x.z, acc);
                acc = fmaf(w.w, x.w, acc);
            }
        } else {
            for (int f = lane; f < F; f += 32) acc = fmaf(__ldg(wrow + f), xb[f], acc);
        }
        acc = warp_sum(acc);
        if (lane == 0) q[r] = acc;
    }
    __syncthreads();

    const int n_lin_tasks = a.ri + a.ry + a.rp + a.rr;
    const int n_tasks = nA + nB + nC + nD + n_lin_tasks;

    for (int it = 0; it < a.T; ++it) {
        // (0) factor vectors
        if (tid < a.ri) {
            fac[tid] = p[3 + tid];
        } else if (tid >= 32 && tid < 32 + a.ry + a.rp + a.rr) {
            int k = tid - 32, m = 1;
            const float* rows = a.rows_y;
            if (k >= a.ry) { k -= a.ry; m = 2; rows = a.rows_p; }
            if (m == 2 && k >= a.rp) { k -= a.rp; m = 3; rows = a.rows_r; }
            const float w = p[m - 1];
            const float ca = rows[4 * k], cb = rows[4 * k + 1], cc = rows[4 * k + 2], cd = rows[4 * k + 3];
            float sn, cs;
            sincosf(cb * w + cc, &sn, &cs);
            fac[m * kMaxModeRank + k] = ca * cs + cd;
            dfac[m * kMaxModeRank + k] = -(ca * cb) * sn;
        }
        __syncthreads();
        // (1) symmetric products
        for (int idx = tid; idx < 4 * kMaxPairs; idx += THREADS) {
            const int m = idx / kMaxPairs, k = idx % kMaxPairs;
            if (k < nP[m]) {
                const int pr = pairs[idx];
                prod[idx] = fac[m * kMaxModeRank + (pr & 255)] * fac[m * kMaxModeRank + (pr >> 8)];
            }
        }
        __syncthreads();
        // (2) T[bcd] = sum_a S[a,bcd] UU[a];  ypr[bcd] = YY_b PP_c RR_d
        for (int bcd = tid; bcd < nBCD; bcd += THREADS) {
            const int b = bcd / (nC * nD), c = (bcd / nD) % nC, d = bcd % nD;
            ypr[bcd] = prod[kMaxPairs + b] * prod[2 * kMaxPairs + c] * prod[3 * kMaxPairs + d];
            float t = 0.f;
            for (int aa = 0; aa < nA; ++aa) t = fmaf(St[(long long)aa * nBCDp + bcd], prod[aa], t);
            Tb[bcd] = t;
        }
        __syncthreads();
        // (3) warp tasks: the four G vectors and the linear-term derivatives
        for (int task = warp; task < n_tasks; task += NW) {
            float acc = 0.f;
            int k = task;
            if (k < nA) {
                const float* row = St + (long long)k * nBCDp;
                for (int bcd = lane; bcd < nBCD; bcd += 32) acc = fmaf(row[bcd], ypr[bcd], acc);
                acc = warp_sum(acc);
                if (lane == 0) G[k] = acc;
                continue;
            }
            k -= nA;
            if (k < nB) {
                for (int i = lane; i < nC * nD; i += 32) {
                    const int c = i / nD, d = i % nD;
                    acc = fmaf(Tb[(k * nC + c) * nD + d], prod[2 * kMaxPairs + c] * prod[3 * kMaxPairs + d], acc);
                }
                acc = warp_sum(acc);
                if (lane == 0) G[kMaxPairs + k] = acc;
                continue;
            }
            k -= nB;
            if (k < nC) {
                for (int i = lane; i < nB * nD; i += 32) {
                    const int b = i / nD, d = i % nD;
                    acc = fmaf(Tb[(b * nC + k) * nD + d], prod[kMaxPairs + b] * prod[3 * kMaxPairs + d], acc);
                }
                acc = warp_sum(acc);
                if (lane == 0) G[2 * kMaxPairs + k] = acc;
                continue;
            }
            k -= nC;
            if (k < nD) {
                for (int i = lane; i < nB * nC; i += 32) {
                    const int b = i / nC, c = i % nC;
                    acc = fmaf(Tb[(b * nC + c) * nD + k], prod[kMaxPairs + b] * prod[2 * kMaxPairs + c], acc);
                }
                acc = warp_sum(acc);
                if (lane == 0) G[3 * kMaxPairs + k] = acc;
                continue;
            }
            k -= nD;
            // linear term: mode m, entry e:  sum over the other three modes of q[r] * prod(other factors)
            int m = 0;
            while (k >= dims[m]) { k -= dims[m]; ++m; }
            const int o0 = m == 0 ? 1 : 0, o1 = m <= 1 ? 2 : 1, o2 = m <= 2 ? 3 : 2;
            const int n0 = dims[o0], n1 = dims[o1], n2 = dims[o2];
            for (int i = lane; i < n0 * n1 * n2; i += 32) {
                int idx4[4];
                idx4[m] = k;
                idx4[o0] = i / (n1 * n2);
                idx4[o1] = (i / n2) % n1;
                idx4[o2] = i % n2;
                const int r = ((idx4[0] * a.ry + idx4[1]) * a.rp + idx4[2]) * a.rr + idx4[3];
                const float w = fac[o0 * kMaxModeRank + idx4[o0]] * fac[o1 * kMaxModeRank + idx4[o1]] *
                                fac[o2 * kMaxModeRank + idx4[o2]];
                acc = fmaf(q[r], w, acc);
            }
            acc = warp_sum(acc);
            if (lane == 0) lin[m * kMaxModeRank + k] = acc;
        }
        __syncthreads();
        // (4) assemble, clip, step (one thread; O(sum of squared ranks))
        if (tid == 0) {
            float g[3 + kMaxModeRank];
            for (int m = 0; m < 4; ++m) {
                const int r = dims[m];
                float gang = 0.f;
                for (int e = 0; e < r; ++e) {
                    float acc = 2.0f * G[m * kMaxPairs + pair_index(e, e, r)] * fac[m * kMaxModeRank + e];
                    for (int i = 0; i < r; ++i) {
                        if (i == e) continue;
                        const int lo = i < e ? i : e, hi = i < e ? e : i;
                        acc = fmaf(G[m * kMaxPairs + pair_index(lo, hi, r)], fac[m * kMaxModeRank + i], acc);
                    }
                    const float d = acc - lin[m * kMaxModeRank + e];
                    if (m == 0) g[3 + e] = d;
                    else gang = fmaf(d, dfac[m * kMaxModeRank + e], gang);
                }
                if (m > 0) g[m - 1] = gang;
            }
            float ss = 0.f;
            for (int i = 0; i < NP; ++i) ss = fmaf(g[i], g[i], ss);
            float coef = a.clip / (sqrtf(ss) + 1e-6f);
            coef = coef < 1.0f ? coef : 1.0f;
            for (int i = 0; i < NP; ++i) p[i] = __fsub_rn(p[i], __fmul_rn(a.lr, __fmul_rn(g[i], coef)));
        }
        __syncthreads();
    }
    if (tid < NP) a.P[s * a.ldp + tid] = p[tid];
}

// ---------------------------------------------------------------------------------------------
// warp-per-sample kernel (compile-time ranks): the small-batch / single-image case.
// The 3000-step chain is a latency problem there, so one sample is spread over the 32 lanes of a warp:
// the folded Gram tensor lives in REGISTERS (each lane owns 7 of the 216 (b,c,d) rows), every lane keeps
// an identical copy of p, partial gradients are combined with one xor-butterfly of 8 values per step
// (bitwise identical in all lanes), and nothing but two tiny per-warp tables touches shared memory.
// ---------------------------------------------------------------------------------------------
template <int RI, int RY, int RP, int RR, int WARPS>
__global__ void __launch_bounds__(32 * WARPS) tucker_fit_wps_kernel(const __grid_constant__ TuckerArgs a) {
    constexpr int R = RI * RY * RP * RR, NP = 3 + RI;
    constexpr int nA = tri(RI), NAP = (nA + 3) / 4 * 4, nB = tri(RY), nC = tri(RP), nD = tri(RR);
    constexpr int nBCD = nB * nC * nD, ROWS = (nBCD + 31) / 32, JKL = RY * RP * RR;
    constexpr int NANG = RY + RP + RR, NPAIR = nB + nC + nD;
    static_assert(JKL <= 32 && NANG <= 32 && NPAIR <= 32, "one lane per angle-mode entry");
    extern __shared__ __align__(16) float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int F = a.F, Fp = (F + 3) / 4 * 4;
    static_assert(2 * NANG + 2 * NPAIR <= 64, "table space");
    float* xb = smem + warp * (Fp + 64);  // this warp's x row (16B aligned), then its two tables
    float* fac = xb + Fp;          // [2*NANG]: c_y,c_p,c_r then dc_y,dc_p,dc_r
    float* tab = fac + 2 * NANG;   // [2*NPAIR]: YY,PP,RR then dYY/dw_y, dPP/dw_p, dRR/dw_r
    const long long s = (long long)blockIdx.x * WARPS + warp;
    const bool live = s < a.N;     // warp-uniform

    // ---- static per-lane roles ----
    // (i) cosine row of lanes < NANG
    float ra = 0.f, rb = 0.f, rc = 0.f, rd = 0.f;
    int my_angle = 0;
    if (lane < NANG) {
        const float* rows = lane < RY ? a.rows_y + 4 * lane
                          : lane < RY + RP ? a.rows_p + 4 * (lane - RY) : a.rows_r + 4 * (lane - RY - RP);
        ra = rows[0]; rb = rows[1]; rc = rows[2]; rd = rows[3];
        my_angle = lane < RY ? 0 : (lane < RY + RP ? 1 : 2);
    }
    // (ii) symmetric pair of lanes < NPAIR (index into fac[])
    int pj0 = 0, pj1 = 0;
    if (lane < NPAIR) {
        int m = lane < nB ? 0 : (lane < nB + nC ? 1 : 2);
        int e = lane - (m == 0 ? 0 : (m == 1 ? nB : nB + nC));
        int r = m == 0 ? RY : (m == 1 ? RP : RR), base = m == 0 ? 0 : (m == 1 ? RY : RY + RP);
        int i, j;
        unpair(e, r, &i, &j);
        pj0 = base + i; pj1 = base + j;
    }
    // (iii) the lane's rows of the folded Gram tensor and their (b,c,d)
    float Srow[ROWS][nA];
    int rb_[ROWS], rc_[ROWS], rd_[ROWS];
#pragma unroll
    for (int m = 0; m < ROWS; ++m) {
        const int bcd = lane + 32 * m;
        const bool ok = bcd < nBCD;
        rb_[m] = ok ? bcd / (nC * nD) : 0;
        rc_[m] = ok ? nB + (bcd / nD) % nC : 0;
        rd_[m] = ok ? nB + nC + bcd % nD : 0;
#pragma unroll
        for (int aa = 0; aa < nA; ++aa) Srow[m][aa] = ok ? __ldg(a.S + (long long)bcd * NAP + aa) : 0.f;
    }
    // (iv) linear-term role of lanes < JKL: entry (j,k,l) and q[i][jkl]
    const int lj = lane < JKL ? lane / (RP * RR) : 0, lk = lane < JKL ? RY + (lane / RR) % RP : 0,
              ll = lane < JKL ? RY + RP + lane % RR : 0;
    float q[RI];
#pragma unroll
    for (int i = 0; i < RI; ++i) q[i] = 0.f;

    // ---- phase A: q = W2 x (warp-cooperative dot products, x staged in shared memory) ----
    if (live) {
        const float* xrow = a.X + s * a.ldx;
        if (a.ipd) {   // raw landmarks: each lane derives the row's (ref, ipd); the pad columns stay zero
            const IpdRow nr = ipd_row(xrow);
            for (int f = lane; f < Fp; f += 32) xb[f] = f < F ? ipd_map(__ldg(xrow + f), nr, f % 3) : 0.f;
        } else {
            for (int f = lane; f < Fp; f += 32) xb[f] = f < F ? __ldg(xrow + f) : 0.f;
        }
    }
    __syncwarp();
    if (live) {
        for (int jkl = 0; jkl < JKL; ++jkl) {
#pragma unroll
            for (int i = 0; i < RI; ++i) {
                const float* wrow = a.W2 + (long long)(i * JKL + jkl) * F;
                float acc = 0.f;
                if (a.vec_ok) {
                    for (int f = 4 * lane; f < F; f += 128) {
                        const float4 w = __ldg(reinterpret_cast<const float4*>(wrow + f));
                        const float4 x = *reinterpret_cast<const float4*>(xb + f);
                        acc = fmaf(w.x, x.x, acc); acc = fmaf(w.y, x.y, acc);
                        acc = fmaf(w.z, x.z, acc); acc = fmaf(w.w, x.w, acc);
                    }
                } else {
                    for (int f = lane; f < F; f += 32) acc = fmaf(__ldg(wrow + f), xb[f], acc);
                }
                acc = warp_sum(acc);
                if (lane == jkl) q[i] = acc;
            }
        }
    }

    // ---- phase B ----
    float p[NP];
#pragma unroll
    for (int i = 0; i < NP; ++i) p[i] = 0.f;  // zero init, TD_Tester.py:130
    const float lr = a.lr, clip = a.clip;
    const int T = live ? a.T : 0;
#pragma unroll 1
    for (int it = 0; it < T; ++it) {
        // cosine features: lane j < NANG evaluates row j once, shares through the per-warp table
        {
            const float w = my_angle == 0 ? p[0] : (my_angle == 1 ? p[1] : p[2]);
            float sn, cs;
            sincosf(rb * w + rc, &sn, &cs);
            if (lane < NANG) {
                fac[lane] = ra * cs + rd;
                fac[NANG + lane] = -(ra * rb) * sn;
            }
        }
        __syncwarp();
        if (lane < NPAIR) {
            const float x0 = fac[pj0], x1 = fac[pj1], d0 = fac[NANG + pj0], d1 = fac[NANG + pj1];
            tab[lane] = x0 * x1;
            tab[NPAIR + lane] = fmaf(d0, x1, x0 * d1);   // d(x0*x1)/dw
        }
        __syncwarp();
        float u[RI], UU[nA];
#pragma unroll
        for (int i = 0; i < RI; ++i) u[i] = p[3 + i];
        sym_products<RI>(u, UU);

        float GU[nA];
#pragma unroll
        for (int aa = 0; aa < nA; ++aa) GU[aa] = 0.f;
        float g[NP];
#pragma unroll
        for (int i = 0; i < NP; ++i) g[i] = 0.f;
#pragma unroll
        for (int m = 0; m < ROWS; ++m) {
            const float y = tab[rb_[m]], pp = tab[rc_[m]], r = tab[rd_[m]];
            const float dy = tab[NPAIR + rb_[m]], dp = tab[NPAIR + rc_[m]], dr = tab[NPAIR + rd_[m]];
            const float ypr = y * pp * r;
            float t0 = 0.f, t1 = 0.f, t2 = 0.f;
#pragma unroll
            for (int aa = 0; aa < nA; ++aa) {
                const float sv = Srow[m][aa];
                if (aa % 3 == 0) t0 = fmaf(sv, UU[aa], t0);
                else if (aa % 3 == 1) t1 = fmaf(sv, UU[aa], t1);
                else t2 = fmaf(sv, UU[aa], t2);
                GU[aa] = fmaf(sv, ypr, GU[aa]);
            }
            const float t = (t0 + t1) + t2;
            g[0] = fmaf(t, dy * pp * r, g[0]);
            g[1] = fmaf(t, y * dp * r, g[1]);
            g[2] = fmaf(t, y * pp * dr, g[2]);
        }
        {
            float du[RI];
            sym_backprop<RI>(GU, u, du);
#pragma unroll
            for (int i = 0; i < RI; ++i) g[3 + i] = du[i];
        }
        // linear term -q.z : lane jkl owns q[:, jkl]
        {
            const float cyj = fac[lj], cpk = fac[lk], crl = fac[ll];
            const float dyj = fac[NANG + lj], dpk = fac[NANG + lk], drl = fac[NANG + ll];
            const float tj = cyj * cpk * crl;
            float e = 0.f;
#pragma unroll
            for (int i = 0; i < RI; ++i) {
                e = fmaf(u[i], q[i], e);
                g[3 + i] = fmaf(-q[i], tj, g[3 + i]);
            }
            g[0] = fmaf(-e, dyj * cpk * crl, g[0]);
            g[1] = fmaf(-e, cyj * dpk * crl, g[1]);
            g[2] = fmaf(-e, cyj * cpk * drl, g[2]);
        }
        // xor butterfly: every lane ends with the same bits (fp add commutes, pairs swap operands)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
#pragma unroll
            for (int i = 0; i < NP; ++i) g[i] += __shfl_xor_sync(0xffffffffu, g[i], o);
        clip_and_step<NP>(p, g, lr, clip);
        __syncwarp();   // tables are rewritten next step
    }
    if (live && lane < NP) {
        float v = p[0];
#pragma unroll
        for (int i = 1; i < NP; ++i) v = lane == i ? p[i] : v;
        a.P[s * a.ldp + lane] = v;
    }
}

// ---------------------------------------------------------------------------------------------
// tensor-core iteration kernel (ranks 5,3,3,3): SURVEY.md section 8f row 2.
// One CTA = 128 samples = 128 TMEM lanes; a thread owns one sample.  The two contractions with the folded Gram
// tensor leave the FP32 pipe:
//   T[s, bcd]   = sum_A UU[s,A] * S[A,bcd]                          tcgen05 GEMM  128 x 224 x 16
//   V[s, A,b]   = sum_{c,D} (PP_c RR_D)[s] * S[A,b,c,D]             tcgen05 GEMM  128 x 96 x 40
//   GU[s,A]     = sum_b YY_b V[s,A,b]                               90 FMAs per sample, from TMEM
// (3xTF32: FP32-grade products; 6 resp. 15 accumulation steps per TMEM accumulator, so the tensor core's truncating
// accumulate stays below the split's own error).  Reading results back from TMEM is what this kernel is bound by
// (a first version that produced V[s,A,b,c] = 540 columns per sample spent 42 % of its time in tcgen05.ld).  Per iteration a thread computes its cosine features and monomials, writes its
// row of the two A operands (UU, RR) into shared memory in the UMMA no-swizzle layout, thread 0 issues the MMAs,
// the linear term runs while they execute, and the results come back with tcgen05.ld.
// FP32-pipe work per sample-iteration drops from ~7.7 k FMAs to ~1.9 k.
// ---------------------------------------------------------------------------------------------
struct TcFitCfg {
    static constexpr int RI = 5, RY = 3, RP = 3, RR = 3, R = 135, RPAD = 136, NP = 8;
    static constexpr int nA = 15, nB = 6, nC = 6, nD = 6, nBCD = 216;
    static constexpr int THREADS = 128;               // samples per CTA (= TMEM lanes); the CTA has 2 threads per sample
    // Operands are FP16 hi/lo planes (kind::f16, K = 16 per MMA): 12 MMAs per iteration instead of the 21 of a 3xTF32 split at
    // the same cycle cost per instruction -- the V-issuing warp, which blocks while the MMA queue drains, is the iteration's
    // critical path -- with the same 22 operand bits.  Ranges: S carries a per-plan power-of-two scale (s_exp), UU a
    // per-sample, per-iteration one (it grows from 0), PP (x) RR a fixed 2^kPrExp; the scales come off in the read-back.
    static constexpr int K1 = 16, N1 = 224;           // T GEMM: K = A (15 -> 16: one k-step), N = bcd (216 -> 224)
    static constexpr int KV = 48, NV = 96;            // V GEMM: K = (c,D) (36 -> 48: three k-steps), N = (A,b) (90 -> 96)
    static constexpr int B1_BYTES = ttc::op16_bytes(N1, K1);    // 7168 per plane
    static constexpr int BV_BYTES = ttc::op16_bytes(NV, KV);    // 9216 per plane
    static constexpr int AV_BYTES = ttc::op16_bytes(128, KV);   // 12288 per plane
    static constexpr int OFF_B1 = 0;                                   // hi, lo
    static constexpr int OFF_BV = OFF_B1 + 2 * B1_BYTES;               // hi, lo
    static constexpr int OFF_AV = OFF_BV + 2 * BV_BYTES;               // hi, lo   (the T GEMM's A operand lives in tensor memory)
    // q lives in TENSOR MEMORY (columns COL_Q .. COL_Q+135 of each sample's lane): the 17 KB per warp and iteration that
    // both roles read would otherwise be 38 % of the SM's shared-memory traffic (the UMMA operand reads and the operand
    // stores share the same 128 B/clk).  The region below only holds the phase-A staging tiles.
    static constexpr int FC = 16, XSTR = THREADS + 2;                  // phase-A tiles, as in the thread-per-sample kernel
    static constexpr int OFF_Q = OFF_AV + 2 * AV_BYTES;                // phase-A tiles [FC][XSTR] + [FC][RPAD]
    static constexpr int OFF_BAR = OFF_Q + (FC * XSTR + FC * RPAD) * 4;
    static constexpr int OFF_GX = OFF_BAR + 64;                        // exchange between the two roles [NGX][128] floats
    static constexpr int NGX = 9;                                      // 8 gradient parts + the identity thread's part of d/d(yaw)
    static constexpr size_t SMEM_BYTES = OFF_GX + NGX * THREADS * 4;
    static constexpr int TMEM_COLS = 512;
    static constexpr int COL_T = 0, COL_V = 224, COL_Q = 320, COL_A1 = 456;   // A1: the T GEMM's A operand (UU hi | lo, 2 x 8 columns of packed halves)
};

// shared-memory image of the tensor-core kernel's constant B operands, built once per plan:
//   B1[n = bcd][k = A]            = S[A,b,c,d]      (T GEMM, 224 x 16)
//   BV[n = A*6 + b][k = c*6 + d]  = S[A,b,c,d]      (V GEMM,  96 x 40)
// each as a hi plane followed by a lo plane (FP16, scaled by the plan's power of two), UMMA no-swizzle K-major layout
__global__ void build_tc_operands_kernel(const float* __restrict__ S, float s_scale, uint8_t* __restrict__ img) {
    using C = TcFitCfg;
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    for (int idx = tid; idx < C::N1 * C::K1; idx += nth) {
        const int n = idx / C::K1, k = idx % C::K1;
        const float v = (n < C::nBCD && k < C::nA) ? S[n * 16 + k] * s_scale : 0.f;
        __half hi, lo;
        ttc::split_half(v, hi, lo);
        *reinterpret_cast<__half*>(img + C::OFF_B1 + ttc::op16_offset(n, k, C::K1)) = hi;
        *reinterpret_cast<__half*>(img + C::OFF_B1 + C::B1_BYTES + ttc::op16_offset(n, k, C::K1)) = lo;
    }
    for (int idx = tid; idx < C::NV * C::KV; idx += nth) {
        const int n = idx / C::KV, k = idx % C::KV;
        float v = 0.f;
        if (n < C::nA * C::nB && k < C::nC * C::nD) {
            const int aa = n / C::nB, b = n % C::nB;
            v = S[(b * 36 + k) * 16 + aa] * s_scale;
        }
        __half hi, lo;
        ttc::split_half(v, hi, lo);
        *reinterpret_cast<__half*>(img + C::OFF_BV + ttc::op16_offset(n, k, C::KV)) = hi;
        *reinterpret_cast<__half*>(img + C::OFF_BV + C::BV_BYTES + ttc::op16_offset(n, k, C::KV)) = lo;
    }
}

// Packed FP32 (f32x2) forms of the tensor-core kernel's scalar products: each lane does the scalar code's IEEE operation,
// so the results are bit for bit those of the scalar loops they replace.
// y[i] = x[i] * k
template <int N>
__device__ __forceinline__ void scale_packed(const float* x, float k, float* y) {
#pragma unroll
    for (int i = 0; i + 1 < N; i += 2) {
        const float2 t = __fmul2_rn(make_float2(x[i], x[i + 1]), make_float2(k, k));
        y[i] = t.x;
        y[i + 1] = t.y;
    }
    if (N % 2) y[N - 1] = x[N - 1] * k;
}
// sym_products with one factor pre-scaled: vv[(i,j)] = vs[i] * v[j] for i <= j, paired along even j within a row
template <int R>
__device__ __forceinline__ void sym_products_packed(const float* vs, const float* v, float* vv) {
#pragma unroll
    for (int i = 0; i < R; ++i)
#pragma unroll
        for (int j = i; j < R; ++j) {
            if (j % 2 == 0 && j + 1 < R) {
                const float2 t = __fmul2_rn(make_float2(vs[i], vs[i]), make_float2(v[j], v[j + 1]));
                vv[pair_index(i, j, R)] = t.x;
                vv[pair_index(i, j + 1, R)] = t.y;
            } else if (j % 2 == 0 || j == i) {
                vv[pair_index(i, j, R)] = vs[i] * v[j];
            }
        }
}

// All of T contracted over b first: s[c,d] = sum_b T[b,c,d] * YYk[b] (216 FMAs; YYk carries the inverse operand scales).
// GR[d] = sum_c PP_c s[c,d] and GP[c] = sum_d RR_d s[c,d] follow from it (72 FMAs); GY comes from the V accumulator
// (GY[b] = sum_A UU_A V[A,b], on the identity thread).  The earlier form (tr[b,c] = sum_d T RR_d for GY and GP, plus
// GR on its own) took 504 FMAs on the angle thread.
// The FMAs run as 108 packed pairs s[c, d..d+1] (FFMA2, YYk[b] broadcast): column bcd = 36b + 6c + d, so an even column
// starts a pair of one (b, c), and it sits in an aligned register pair of the load.  Each lane is the scalar fmaf chain.
__device__ __forceinline__ void tc_reduce_t_b(uint32_t taddr, const float (&YYk)[6], float2 (&s)[18]) {
#pragma unroll
    for (int i = 0; i < 18; ++i) s[i] = make_float2(0.f, 0.f);
    constexpr int NL = 7;   // 224 columns, 216 used
    uint32_t buf[2][32];
    tmem_load32_async(taddr, buf[0]);
#pragma unroll
    for (int ci = 0; ci < NL; ++ci) {
        tmem_load_wait();
        if (ci + 1 < NL) tmem_load32_async(taddr + 32 * (ci + 1), buf[(ci + 1) & 1]);
#pragma unroll
        for (int x = 0; x < 32; x += 2) {
            const int bcd = 32 * ci + x;
            if (bcd < 216) {
                const float2 t = make_float2(__uint_as_float(buf[ci & 1][x]), __uint_as_float(buf[ci & 1][x + 1]));
                const float y = YYk[bcd / 36];
                s[(bcd % 36) / 2] = __ffma2_rn(t, make_float2(y, y), s[(bcd % 36) / 2]);
            }
        }
    }
}

// Two threads per sample (256 threads = 8 warps per CTA; warps w and w+4 own the same TMEM lanes):
//   role 0 ("angle thread", warps 0-3): writes the UU operand, consumes the first half of T, finishes d/d(angles)
//   role 1 ("identity thread", warps 4-7): writes the PP (x) RR operand, consumes the second half of T and V -> d/du
// Both keep a bitwise-identical copy of p; partial sums and gradient parts cross through shared memory.
// development build only (-DNLML_TC_DBG): the product kernel has no switch that skips work
#ifdef NLML_TC_DBG
#define NLML_DBG_MMA (a.dbg != 1)
#define NLML_DBG_READ (a.dbg != 2)
#else
#define NLML_DBG_MMA true
#define NLML_DBG_READ true
#endif
__global__ void __launch_bounds__(256, 1) tucker_fit_tc_kernel(const __grid_constant__ TuckerArgs a) {
    using C = TcFitCfg;
    extern __shared__ __align__(1024) uint8_t tsm[];
    uint8_t* b1_hi = tsm + C::OFF_B1;
    uint8_t* b1_lo = b1_hi + C::B1_BYTES;
    uint8_t* bv_hi = tsm + C::OFF_BV;
    uint8_t* bv_lo = bv_hi + C::BV_BYTES;
    uint8_t* av_hi = tsm + C::OFF_AV;
    uint8_t* av_lo = av_hi + C::AV_BYTES;
    float* q_s = reinterpret_cast<float*>(tsm + C::OFF_Q);
    uint64_t* bar = reinterpret_cast<uint64_t*>(tsm + C::OFF_BAR);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 2);
    float* gx = reinterpret_cast<float*>(tsm + C::OFF_GX);

    // the warp index through a shuffle: provably warp-uniform, so the two MMA-issuing warps keep their descriptor arithmetic
    // in the uniform datapath (a plain `tid == 0` issue wraps every tcgen05.mma in a register->uniform broadcast loop,
    // ~100 cycles per MMA on the iteration's critical path)
    const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int row = tid & 127, role = warp >> 2;
    const long long s0 = (long long)blockIdx.x * C::THREADS;
    const bool vec_ok = a.vec_ok != 0;
    const int F = a.F;

    if (tid == 0) {
        ttc::mbar_init(bar, 1);       // T GEMM done
        ttc::mbar_init(bar + 1, 1);   // V GEMM done
        ttc::mbar_init(bar + 3, 1);   // B operands landed (TMA)
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) tmem_alloc_cols(tmem_slot, C::TMEM_COLS);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");   // (phase A's barriers publish the allocation)

    // ---- constant B operands: the folded Gram tensor in both GEMM views (hi/lo TF32 planes in the UMMA layout), staged
    // once per CTA by ONE 1-D TMA bulk copy of the image build_tc_operands_kernel prepared at plan creation ----
    if (tid == 0) {
        tgen::mbar_expect_tx(bar + 3, (uint32_t)C::OFF_AV);
        tgen::bulk_load(tsm + C::OFF_B1, a.tc_ops, (uint32_t)C::OFF_AV, bar + 3);
    }
    // ---- phase A: q[r] = sum_f W2[r][f] * x[f]; the two threads of a sample take half of the rows r each ----
    {
        constexpr int RH = C::RPAD / 2;   // 68 rows per role
        float* xs = q_s;
        float* ws = q_s + C::FC * C::XSTR;
        float acc[RH];
#pragma unroll
        for (int r = 0; r < RH; ++r) acc[r] = 0.f;
        if (a.Qpre) {   // projected already by tucker_project_tc_kernel: coalesced reads of this CTA's [RPAD][128] slab
            const float* slab = a.Qpre + (size_t)blockIdx.x * C::RPAD * 128 + (size_t)role * RH * 128 + row;
#pragma unroll
            for (int r = 0; r < RH; ++r) acc[r] = __ldg(slab + r * 128);
        }
        // raw landmarks: the 128 rows' (ref, ipd) once, in the gradient exchange buffer (unused until phase B)
        IpdRow* ipd_s = reinterpret_cast<IpdRow*>(gx);
        static_assert(C::THREADS * sizeof(IpdRow) <= C::NGX * C::THREADS * 4, "IPD constants fit the exchange buffer");
        if (a.ipd && !a.Qpre) {
            if (role == 0 && s0 + row < a.N) ipd_s[row] = ipd_row(a.X + (s0 + row) * a.ldx);
            __syncthreads();
        }
        for (int f0 = 0; f0 < (a.Qpre ? 0 : F); f0 += C::FC) {
            for (int idx = tid; idx < C::THREADS * (C::FC / 4); idx += 256) {
                const int s = idx / (C::FC / 4), c4 = idx % (C::FC / 4);
                const long long grow = s0 + s;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (grow < a.N) v = load_row4(a.X + grow * a.ldx, f0 + 4 * c4, F, vec_ok);
                xs[(4 * c4 + 0) * C::XSTR + s] = v.x;
                xs[(4 * c4 + 1) * C::XSTR + s] = v.y;
                xs[(4 * c4 + 2) * C::XSTR + s] = v.z;
                xs[(4 * c4 + 3) * C::XSTR + s] = v.w;
            }
            for (int idx = tid; idx < C::RPAD * (C::FC / 4); idx += 256) {
                const int r = idx / (C::FC / 4), c4 = idx % (C::FC / 4);
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (r < C::R) v = load_row4(a.W2 + (long long)r * F, f0 + 4 * c4, F, vec_ok);
                ws[(4 * c4 + 0) * C::RPAD + r] = v.x;
                ws[(4 * c4 + 1) * C::RPAD + r] = v.y;
                ws[(4 * c4 + 2) * C::RPAD + r] = v.z;
                ws[(4 * c4 + 3) * C::RPAD + r] = v.w;
            }
            __syncthreads();
            if (a.ipd) {
                ipd_tile(xs, C::XSTR, C::FC, C::THREADS, ipd_s, a.N - s0, f0, F, tid, 256);
                __syncthreads();
            }
#pragma unroll 4
            for (int f = 0; f < C::FC; ++f) {
                const float xv = xs[f * C::XSTR + row];
#pragma unroll
                for (int r4 = 0; r4 < RH / 4; ++r4) {
                    const float4 w = *reinterpret_cast<const float4*>(&ws[f * C::RPAD + role * RH + 4 * r4]);
                    acc[4 * r4 + 0] = fmaf(xv, w.x, acc[4 * r4 + 0]);
                    acc[4 * r4 + 1] = fmaf(xv, w.y, acc[4 * r4 + 1]);
                    acc[4 * r4 + 2] = fmaf(xv, w.z, acc[4 * r4 + 2]);
                    acc[4 * r4 + 3] = fmaf(xv, w.w, acc[4 * r4 + 3]);
                }
            }
            __syncthreads();
        }
        // q -> tensor memory: this thread's 68 rows into columns COL_Q + 68*role .. of its sample's lane
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t qdst = *tmem_slot + ((uint32_t)((warp & 3) * 32) << 16) + C::COL_Q + role * RH;
        static_assert(RH == 68, "two 32-column stores and one 4-column store");
        tmem_store32(qdst, acc);
        tmem_store32(qdst + 32, acc + 32);
        tmem_store4(qdst + 64, acc + 64);
        tmem_store_wait();
    }
    ttc::mbar_wait(bar + 3, 0);   // the B operands are in shared memory (async proxy writes: visible to the MMAs)
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tmem_slot;
    const uint32_t lane_addr = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const QTmem qa{lane_addr + C::COL_Q};

    // ---- phase B ----
    float p[C::NP];
#pragma unroll
    for (int i = 0; i < C::NP; ++i) p[i] = 0.f;  // zero init, TD_Tester.py:130
    const float lr = a.lr, clip = a.clip;
    uint32_t phase = 0;
    int uu_exp = 0;   // role 0: exponent of this iteration's UU operand scale
#ifdef NLML_TC_TIMING
    // development build only (scripts/time_tucker_tc.py): per-phase cycle counts of one thread per role
    float tacc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    uint32_t tprev = 0;
#define NLML_TSTAMP(i) { const uint32_t tnow = (uint32_t)clock(); tacc[i] += (float)(tnow - tprev); tprev = tnow; }
#define NLML_TSTART() { tprev = (uint32_t)clock(); }
#else
#define NLML_TSTAMP(i)
#define NLML_TSTART()
#endif
#pragma unroll 1
    for (int it = 0; it < a.T; ++it) {
        NLML_TSTART();
        float cy[3], dcy[3], cp[3], dcp[3], cr[3], dcr[3], u[5];
#pragma unroll
        for (int i = 0; i < 5; ++i) u[i] = p[3 + i];
        // The T GEMM needs only u: the angle threads publish the UU operand first and thread 0 launches that GEMM
        // before anybody evaluates a cosine; it runs underneath the feature computation.  (Named barrier 1: the 128
        // angle threads only.)
        if (role == 0) {
            // the UU operand goes to TENSOR MEMORY (one 32-column store: hi | lo), not through shared memory: no operand
            // stores, no generic->async proxy fence, and the MMA reads A without touching the shared-memory ports
            float UU[16], hl[16];
            // per-sample power-of-two scale: the largest |UU| = (max |u_i|)^2 lands in [2^12, 2^13) (UU starts at 0 and grows over the fit)
            float m = 0.f;
#pragma unroll
            for (int k = 0; k < 5; ++k) m = fmaxf(m, fabsf(u[k]));
            m *= m;
            int eu = 12 - (((__float_as_int(m) >> 23) & 0xff) - 127);
            eu = m > 0.f ? max(min(eu, 100), -80) : 0;
            uu_exp = eu;
            {
                const float su = __int_as_float((eu + 127) << 23);
                float us[5];   // the scale rides on one factor of every product (exact: a power of two)
                scale_packed<5>(u, su, us);
                sym_products_packed<5>(us, u, UU);
                UU[15] = 0.f;
            }
#pragma unroll
            for (int k2 = 0; k2 < 8; ++k2) {   // packed pairs: element 2c in the low half of column c
                const float2 v = make_float2(UU[2 * k2], UU[2 * k2 + 1]);
                const __half2 h = __float22half2_rn(v);
                const float2 hf = __half22float2(h);
                const __half2 l = __float22half2_rn(__fadd2_rn(v, make_float2(-hf.x, -hf.y)));
                hl[k2] = __uint_as_float(*reinterpret_cast<const uint32_t*>(&h));
                hl[8 + k2] = __uint_as_float(*reinterpret_cast<const uint32_t*>(&l));
            }
            tgen::tmem_st8(lane_addr + C::COL_A1, hl);
            tgen::tmem_st8(lane_addr + C::COL_A1 + 8, hl + 8);
            tmem_store_wait();
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            asm volatile("bar.sync 1, 128;" ::: "memory");
            if (warp == 0 && NLML_DBG_MMA) {   // the whole warp, converged; the elected lane issues
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                ttc::gemm3h_ts(tmem + C::COL_T, tmem + C::COL_A1, ttc::smem_u32(b1_hi), ttc::smem_u32(b1_lo), C::K1, C::N1);
                ttc::umma_commit_elect(bar);
            }
        }
        NLML_TSTAMP(0);   // role 0: UU publish + T GEMM issue
        // pitch and roll features first: they are all the V GEMM's operand needs; yaw follows once it is launched
        if (role == 0) {   // only the angle thread differentiates along pitch and roll
            cos_features_sfu<3>(p[1], a.rows_p, cp, dcp);
            cos_features_sfu<3>(p[2], a.rows_r, cr, dcr);
        } else {
            cos_values_sfu<3>(p[1], a.rows_p, cp);
            cos_values_sfu<3>(p[2], a.rows_r, cr);
#pragma unroll
            for (int j = 0; j < 3; ++j) dcp[j] = dcr[j] = 0.f;
        }
        float YY[6], PP[6], RRv[8];
        sym_products<3>(cp, PP);
        sym_products<3>(cr, RRv);
        RRv[6] = RRv[7] = 0.f;
        // the identity threads publish the PP (x) RR operand; thread 160 launches the V GEMM (named barrier 2)
        if (role == 1) {
            float PPs[6];   // the operand's power-of-two scale rides on PP
            {
                const float kPrScale = __int_as_float((127 + a.pr_exp) << 23);
                scale_packed<6>(PP, kPrScale, PPs);
            }
#pragma unroll
            for (int k8 = 0; k8 < C::KV / 8; ++k8) {   // one 16-byte chunk = 8 halves of this row per plane
                uint32_t wh[4], wl[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int k0 = 8 * k8 + 2 * e;   // k = 6c + D: an even k starts a pair (D, D+1) of one c
                    const float2 v = k0 < 36 ? __fmul2_rn(make_float2(PPs[k0 / 6], PPs[k0 / 6]),
                                                          make_float2(RRv[k0 % 6], RRv[k0 % 6 + 1]))
                                             : make_float2(0.f, 0.f);
                    const __half2 h = __float22half2_rn(v);
                    const float2 hf = __half22float2(h);
                    const __half2 l = __float22half2_rn(__fadd2_rn(v, make_float2(-hf.x, -hf.y)));
                    wh[e] = *reinterpret_cast<const uint32_t*>(&h);
                    wl[e] = *reinterpret_cast<const uint32_t*>(&l);
                }
                *reinterpret_cast<uint4*>(av_hi + ttc::op16_offset(row, 8 * k8, C::KV)) = make_uint4(wh[0], wh[1], wh[2], wh[3]);
                *reinterpret_cast<uint4*>(av_lo + ttc::op16_offset(row, 8 * k8, C::KV)) = make_uint4(wl[0], wl[1], wl[2], wl[3]);
            }
            ttc::fence_async_smem();
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            asm volatile("bar.sync 2, 128;" ::: "memory");
            if (warp == 5 && NLML_DBG_MMA) {   // warp 5: not on the sub-partition of the T GEMM's issuer (warp 0)
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                ttc::gemm3h_ss(tmem + C::COL_V, ttc::smem_u32(av_hi), ttc::smem_u32(av_lo), ttc::smem_u32(bv_hi),
                               ttc::smem_u32(bv_lo), C::KV, C::NV);
                ttc::umma_commit_elect(bar + 1);
            }
        }
        NLML_TSTAMP(1);   // pitch/roll features (+ role 1: PP(x)RR publish + V GEMM issue)
        cos_features_sfu<3>(p[0], a.rows_y, cy, dcy);
        sym_products<3>(cy, YY);
        // the linear term does not depend on the MMAs: it runs while they execute.  Each role keeps only the outputs it
        // needs (the angle thread ey/ep/er, the identity thread lin_u); the other half is dead code in its branch.
        float lin_u[5], ey[3], ep[3], er[3];
        if (role == 0) {
            float unused[5];
            linear_term<5, 3, 3, 3>(qa, 0, cy, cp, cr, u, unused, ey, ep, er);
        } else {
            float u0[3], u1[3], u2[3];
            linear_term<5, 3, 3, 3>(qa, 0, cy, cp, cr, u, lin_u, u0, u1, u2);
        }

        NLML_TSTAMP(2);   // yaw features + linear term
        if (role == 1) {
            // V[A,b] = sum_{c,D} PP_c RR_D S[A,b,c,D]  ->  GU[A] = sum_b YY_b V[A,b]  ->  d/du
            //                                          and  GY[b] = sum_A UU_A V[A,b]  ->  the quadratic part of d/d(yaw)
            float GU[15], GYv[6], YYk[6], UUk[15];
            {
                const float kv = __int_as_float((127 - a.s_exp - a.pr_exp) << 23);   // 2^-(s_exp + pr_exp): the V accumulator's scale off
                scale_packed<6>(YY, kv, YYk);
                float uk[5];   // the scale rides on one factor of every product
                scale_packed<5>(u, kv, uk);
                sym_products_packed<5>(uk, u, UUk);
            }
            float2 GY2[3];   // GY[b..b+1] as packed pairs (UUk[A] broadcast); GU[A] stays one scalar chain per A
#pragma unroll
            for (int i = 0; i < 15; ++i) GU[i] = 0.f;
#pragma unroll
            for (int i = 0; i < 3; ++i) GY2[i] = make_float2(0.f, 0.f);
            if (NLML_DBG_MMA) ttc::mbar_wait(bar + 1, phase);   // V GEMM
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            NLML_TSTAMP(3);   // wait for the GEMM
            if (NLML_DBG_READ) {
                uint32_t vb[2][32];   // the next 32 columns are in flight while these are reduced
                tmem_load32_async(lane_addr + C::COL_V, vb[0]);
#pragma unroll
                for (int ci = 0; ci < C::NV / 32; ++ci) {
                    tmem_load_wait();
                    if (ci + 1 < C::NV / 32) tmem_load32_async(lane_addr + C::COL_V + 32 * (ci + 1), vb[(ci + 1) & 1]);
#pragma unroll
                    for (int x = 0; x < 32; x += 2) {   // column n = 6A + b: an even column starts a pair (b, b+1) of one A
                        const int n = 32 * ci + x;
                        if (n < 90) {
                            const float2 v = make_float2(__uint_as_float(vb[ci & 1][x]), __uint_as_float(vb[ci & 1][x + 1]));
                            GU[n / 6] = fmaf(v.x, YYk[n % 6], GU[n / 6]);
                            GU[n / 6] = fmaf(v.y, YYk[n % 6 + 1], GU[n / 6]);
                            GY2[(n % 6) / 2] = __ffma2_rn(v, make_float2(UUk[n / 6], UUk[n / 6]), GY2[(n % 6) / 2]);
                        }
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                GYv[2 * i] = GY2[i].x;
                GYv[2 * i + 1] = GY2[i].y;
            }
            float du[5], dy[3];
            sym_backprop<5>(GU, u, du);
            sym_backprop<3>(GYv, cy, dy);
#pragma unroll
            for (int i = 0; i < 5; ++i) gx[(3 + i) * 128 + row] = du[i] - lin_u[i];
            gx[8 * 128 + row] = fmaf(dy[2], dcy[2], fmaf(dy[1], dcy[1], dy[0] * dcy[0]));   // the angle thread adds -ey.dcy
        } else {
            // all of T -> s[c,d] -> GR, GP -> d/d(pitch, roll); d/d(yaw): the linear part here, the quadratic part on the identity thread
            float GR[6], GP[6], YYk[6];
            float2 sc[18];
            {
                const float kt = __int_as_float((127 - a.s_exp - uu_exp) << 23);   // 2^-(s_exp + uu_exp): the T accumulator's scale off
                scale_packed<6>(YY, kt, YYk);
            }
            if (NLML_DBG_MMA) ttc::mbar_wait(bar, phase);       // T GEMM (launched first, long done)
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            NLML_TSTAMP(3);
            float2 GR2[3];   // GR[d..d+1] as packed pairs (PP_c broadcast); GP[c] stays one scalar chain per c
#pragma unroll
            for (int i = 0; i < 3; ++i) GR2[i] = make_float2(0.f, 0.f);
#pragma unroll
            for (int i = 0; i < 6; ++i) GP[i] = 0.f;
            if (NLML_DBG_READ) {
                tc_reduce_t_b(lane_addr + C::COL_T, YYk, sc);
#pragma unroll
                for (int c = 0; c < 6; ++c)
#pragma unroll
                    for (int d2 = 0; d2 < 3; ++d2) {
                        GR2[d2] = __ffma2_rn(make_float2(PP[c], PP[c]), sc[c * 3 + d2], GR2[d2]);
                        GP[c] = fmaf(RRv[2 * d2], sc[c * 3 + d2].x, GP[c]);
                        GP[c] = fmaf(RRv[2 * d2 + 1], sc[c * 3 + d2].y, GP[c]);
                    }
            }
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                GR[2 * i] = GR2[i].x;
                GR[2 * i + 1] = GR2[i].y;
            }
            float dp[3], dr[3];
            sym_backprop<3>(GP, cp, dp);
            sym_backprop<3>(GR, cr, dr);
            float gy = 0.f, gp = 0.f, gr = 0.f;
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                gy = fmaf(-ey[j], dcy[j], gy);
                gp = fmaf(dp[j] - ep[j], dcp[j], gp);
                gr = fmaf(dr[j] - er[j], dcr[j], gr);
            }
            gx[0 * 128 + row] = gy;
            gx[1 * 128 + row] = gp;
            gx[2 * 128 + row] = gr;
        }
        NLML_TSTAMP(4);   // TMEM read-back + reduction + gradient part
        phase ^= 1;
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();   // all 8 gradient parts in gx
        NLML_TSTAMP(5);   // CTA barrier
        float g[C::NP];
#pragma unroll
        for (int i = 0; i < C::NP; ++i) g[i] = gx[i * 128 + row];
        g[0] += gx[8 * 128 + row];   // d/d(yaw) = linear part (angle thread) + quadratic part (identity thread)
        clip_and_step_fast<C::NP>(p, g, lr, clip);
        NLML_TSTAMP(6);   // clip + step
    }
#ifdef NLML_TC_TIMING
    // rows 0..7 of the CTA's output <- the lane-0 timings of warps 0..7
    if ((tid & 31) == 0 && s0 + 8 <= a.N) {
        float* out = a.P + (s0 + warp) * a.ldp;
        for (int i = 0; i < 8; ++i) out[i] = tacc[i] / (float)a.T;
        return;
    }
    if (tid < 8) return;
#endif
    if (role == 0 && s0 + row < a.N) {
        float* out = a.P + (s0 + row) * a.ldp;
#pragma unroll
        for (int i = 0; i < C::NP; ++i) out[i] = p[i];
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) tmem_free_cols(tmem, C::TMEM_COLS);
}


// ---------------------------------------------------------------------------------------------
// TD_Tester.Test as the reference ships it: scipy Powell over the float64 objective (TD_Tester.py:31-58, :191-194),
// reproduced BIT FOR BIT (powell_math.h).  One CTA per sample: every thread runs the same Powell / Brent control flow
// on identical values (the search is a sequential scalar algorithm), and each objective evaluation -- 135 x 1404
// float64 product chains, the part that costs -- is shared by the CTA's threads in exactly the reference's
// operation order: thread t owns features t, t+128, ...; x_hat accumulates over (i,j,k,l) as np.einsum does; the sum
// of squares follows numpy's pairwise summation (leaf blocks of <= 128 elements with eight strided accumulators, then
// the halving tree; the leaf table and the combine program are prepared on the host for the plan's F).
// Bound by the float64 pipe (5 dependent-free operations per (r, feature) pair).
// ---------------------------------------------------------------------------------------------
constexpr int kPowellThreads = 128;
constexpr int kPowellMaxFeat = 16;     // features per thread: F <= 2048
constexpr int kPowellMaxLeaves = 64;

struct PowellArgs {
    const float* X;
    long long N, ldx;
    const float* W2;
    double* P;            // [N][ldp]
    long long ldp;
    double* fun;          // [N] or null
    int* nfev;            // [N] or null
    int ri, ry, rp, rr, F;
    int ipd;              // X rows are raw landmarks: x is staged through the IPD normalisation (common.cuh)
    int nleaf, nprog;
    short leaf_off[kPowellMaxLeaves], leaf_len[kPowellMaxLeaves];
    signed char prog[2 * kPowellMaxLeaves];   // postfix combine program of the pairwise tree: k >= 0 push leaf k, -1 add
    double rows_y[4 * kMaxModeRank], rows_p[4 * kMaxModeRank], rows_r[4 * kMaxModeRank];
};

struct PowellCoopObjective {
    const PowellArgs& a;
    const float* xs;      // shared: this sample's x
    double* e;            // shared: [F] squared residuals
    double* racc;         // shared: [nleaf][8]
    double* leafsum;      // shared: [nleaf]
    double* result;       // shared: [1]
    __device__ double operator()(const double* p) const {
        const int tid = threadIdx.x;
        powell::TuckerFactors t;
        powell::tucker_factors(p, a.ry, a.rp, a.rr, a.rows_y, a.rows_p, a.rows_r, t);
        const double* u = p + 3;
        // (x - x_hat)^2 per feature; the thread's features advance together over r (independent accumulation chains)
        double acc[kPowellMaxFeat];
#pragma unroll
        for (int k = 0; k < kPowellMaxFeat; ++k) acc[k] = 0.0;
        const float* wrow = a.W2;
        for (int i = 0; i < a.ri; ++i)
            for (int j = 0; j < a.ry; ++j)
                for (int kk = 0; kk < a.rp; ++kk)
                    for (int l = 0; l < a.rr; ++l, wrow += a.F) {
                        const double ui = u[i], fy = t.fy[j], fp = t.fp[kk], fr = t.fr[l];
#pragma unroll
                        for (int k = 0; k < kPowellMaxFeat; ++k) {
                            const int m = tid + k * kPowellThreads;
                            if (m < a.F) {
                                const double term = __dmul_rn(__dmul_rn(__dmul_rn(__dmul_rn((double)__ldg(wrow + m), ui), fy), fp), fr);
                                acc[k] = __dadd_rn(acc[k], term);
                            }
                        }
                    }
#pragma unroll
        for (int k = 0; k < kPowellMaxFeat; ++k) {
            const int m = tid + k * kPowellThreads;
            if (m < a.F) {
                const double d = __dsub_rn((double)xs[m], acc[k]);
                e[m] = __dmul_rn(d, d);
            }
        }
        __syncthreads();
        // numpy pairwise sum, leaves first: accumulator j of leaf k
        for (int w = tid; w < a.nleaf * 8; w += kPowellThreads) {
            const int k = w >> 3, j = w & 7, off = a.leaf_off[k], n = a.leaf_len[k];
            if (n >= 8) {
                double r = e[off + j];
                for (int i = 8; i < n - (n % 8); i += 8) r = __dadd_rn(r, e[off + i + j]);
                racc[w] = r;
            }
        }
        __syncthreads();
        for (int k = tid; k < a.nleaf; k += kPowellThreads) {
            const int off = a.leaf_off[k], n = a.leaf_len[k];
            double res;
            if (n < 8) {
                res = 0.0;
                for (int i = 0; i < n; ++i) res = __dadd_rn(res, e[off + i]);
            } else {
                const double* r = racc + 8 * k;
                res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])), __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
                for (int i = n - (n % 8); i < n; ++i) res = __dadd_rn(res, e[off + i]);
            }
            leafsum[k] = res;
        }
        __syncthreads();
        if (tid == 0) {
            double stack[16];
            int sp = 0;
            for (int i = 0; i < a.nprog; ++i) {
                const int op = a.prog[i];
                if (op >= 0) stack[sp++] = leafsum[op];
                else {
                    --sp;
                    stack[sp - 1] = __dadd_rn(stack[sp - 1], stack[sp]);
                }
            }
            *result = __dmul_rn(0.5, stack[0]);
        }
        __syncthreads();
        const double v = *result;
        __syncthreads();   // everybody has read the value before the next evaluation overwrites it
        return v;
    }
};

__global__ void __launch_bounds__(kPowellThreads) tucker_powell_kernel(const __grid_constant__ PowellArgs a) {
    extern __shared__ __align__(16) uint8_t psm_[];
    double* e = reinterpret_cast<double*>(psm_);
    double* racc = e + a.F;
    double* leafsum = racc + 8 * kPowellMaxLeaves;
    double* result = leafsum + kPowellMaxLeaves;
    float* xs = reinterpret_cast<float*>(result + 2);
    const long long s = blockIdx.x;
    const float* xrow = a.X + s * a.ldx;
    if (a.ipd) {   // raw landmarks: x becomes the float32 vector FE.get_feature_vector(..., normalize=True) returns
        const IpdRow nr = ipd_row(xrow);
        for (int f = threadIdx.x; f < a.F; f += kPowellThreads) xs[f] = ipd_map(__ldg(xrow + f), nr, f % 3);
    } else {
        for (int f = threadIdx.x; f < a.F; f += kPowellThreads) xs[f] = __ldg(xrow + f);
    }
    __syncthreads();
    PowellCoopObjective obj{a, xs, e, racc, leafsum, result};
    const int NP = 3 + a.ri;
    double x[powell::kMaxN], direc[powell::kMaxN * powell::kMaxN];
    for (int i = 0; i < NP; ++i) x[i] = 0.0;   // initial_guess = zeros (TD_Tester.py:166)
    const powell::Result res = powell::minimize(obj, NP, x, direc);
    if (threadIdx.x == 0) {
        for (int i = 0; i < NP; ++i) a.P[s * a.ldp + i] = x[i];
        if (a.fun) a.fun[s] = res.fun;
        if (a.nfev) a.nfev[s] = res.nfev;
    }
}

// test hook: the cooperative objective alone, at given parameter points of ONE sample (checked bitwise against the host build)
__global__ void __launch_bounds__(kPowellThreads) tucker_powell_objective_kernel(const __grid_constant__ PowellArgs a, const double* __restrict__ pts,
                                                                                 int npts, double* __restrict__ out) {
    extern __shared__ __align__(16) uint8_t psm_[];
    double* e = reinterpret_cast<double*>(psm_);
    double* racc = e + a.F;
    double* leafsum = racc + 8 * kPowellMaxLeaves;
    double* result = leafsum + kPowellMaxLeaves;
    float* xs = reinterpret_cast<float*>(result + 2);
    for (int f = threadIdx.x; f < a.F; f += kPowellThreads) xs[f] = __ldg(a.X + f);
    __syncthreads();
    PowellCoopObjective obj{a, xs, e, racc, leafsum, result};
    const int NP = 3 + a.ri;
    for (int i = 0; i < npts; ++i) {
        double x[powell::kMaxN];
        for (int k = 0; k < NP; ++k) x[k] = pts[i * NP + k];
        const double v = obj(x);
        if (threadIdx.x == 0) out[i] = v;
    }
}

// TD_Trainer.Train for the columns of one factor matrix (TD_Trainer.py:232-351 -> :125-148 Fourier initial guess, :60-93
// scipy Powell per column): one thread per column, float64, the statements of powell_math.h.
__global__ void cosine_fit_kernel(const double* __restrict__ U, int n_rows, int n_cols, const double* __restrict__ w_rad,
                                  double* __restrict__ init, double* __restrict__ out, double* __restrict__ fun, int* __restrict__ nfev) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_cols) return;
    double x[powell::kMaxN], direc[16], g[4];
    powell::fourier_init(U + j, n_cols, w_rad, n_rows, g);
    for (int i = 0; i < 4; ++i) {
        x[i] = g[i];
        if (init) init[4 * j + i] = g[i];
    }
    powell::CosineObjective obj{U + j, w_rad, n_rows, n_cols};
    const powell::Result res = powell::minimize(obj, 4, x, direc);
    for (int i = 0; i < 4; ++i) out[4 * j + i] = x[i];
    if (fun) fun[j] = res.fun;
    if (nfev) nfev[j] = res.nfev;
}

// ---------------------------------------------------------------------------------------------
// Phase A on the tensor cores: q = W2 x for a whole batch as a 3xTF32 tcgen05 GEMM  [N x F] x [F x 136]  (SURVEY.md
// section 7: at 67 flop/B this projection needs tensor cores to outrun HBM; on CUDA cores it was 37 % of the converged
// solve).  Persistent, one CTA per SM, 128 samples per tile:
//   warp 0       TMA producer: the raw FP32 tile of X (2-D tensor map, 128 rows x 32 features, 128-byte swizzle, rows / columns
//                beyond the batch / F zero-filled by the TMA unit) and the k-block's W2 tile image (1-D bulk copy)
//   warp 1       MMA issuer (converged warp, elected lane): per k-block 4 k-steps x (lo*hi, hi*lo, hi*hi), FP32 TMEM accumulator
//   warps 4-7    converters: split the landed X tile in place into hi = tf32(x) and lo = x - hi (the planes the MMAs read)
//   warps 8-11   promotion + epilogue: tcgen05.ld every group's partial 128 x 136 tile (double-buffered in TMEM), add it into
//                FP32 registers with round-to-nearest, store the finished tile as the CTA-blocked slab [136][128] the fit /
//                solve kernels copy into shared memory with coalesced loads
// ---------------------------------------------------------------------------------------------
struct ProjCfg {
    static constexpr int BM = 128, BK = 32, NQ = 144;           // samples per tile, features per k-block, q rows padded to 16
    static constexpr int STAGES = 3;
    static constexpr int GROUP = 1;                              // k-blocks summed in one TMEM accumulator (12 MMAs) before the partial
                                                                 // tile is promoted into FP32 registers: the tensor core's accumulate
                                                                 // truncates -- a 528-MMA chain left q 3e-5 low (0.1 degrees after the
                                                                 // solve), 48-MMA chains 9e-7; per k-block it is FP32-grade
    static constexpr int X_BYTES = BM * BK * 4;                  // one plane of the X tile (128-byte rows, swizzled)
    static constexpr int W_BYTES = 2 * NQ * BK * 4;              // hi + lo planes of the W2 tile (UMMA no-swizzle image)
    static constexpr int STAGE_BYTES = 2 * X_BYTES + W_BYTES;    // X hi (lands raw) + X lo + W
    static constexpr int OFF_BAR = STAGES * STAGE_BYTES;
    static constexpr size_t SMEM_BYTES = 1024 + OFF_BAR + 256;
    static constexpr int THREADS = 384;
};
struct ProjArgs {
    long long N;
    int F, RPAD, num_kb;
    const uint8_t* wtiles;   // [num_kb][W_BYTES]
    float* Q;                // [tiles][RPAD][128]
    int ipd;                 // X rows are raw landmarks: the converters apply the IPD normalisation before the split
    const float* X;          // ... and read each row's (ref, ipd) from here (the tensor map's base, row pitch ldx floats)
    long long ldx;
};
__device__ __forceinline__ uint64_t proj_desc_sw128(uint32_t smem_addr) {   // K-major, 128-byte swizzle, 8-row groups 1024 B apart
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
__global__ void __launch_bounds__(ProjCfg::THREADS, 1) tucker_project_tc_kernel(const __grid_constant__ CUtensorMap xmap, const __grid_constant__ ProjArgs a) {
    using C = ProjCfg;
    extern __shared__ uint8_t proj_raw[];
    uint8_t* sm = proj_raw + ((1024u - (ttc::smem_u32(proj_raw) & 1023u)) & 1023u);
    uint64_t* bars = reinterpret_cast<uint64_t*>(sm + C::OFF_BAR);
    uint64_t* full = bars;                 // [STAGES] X tile and W tile landed
    uint64_t* conv = bars + C::STAGES;     // [STAGES] hi / lo planes written
    uint64_t* empty = conv + C::STAGES;    // [STAGES] consumed by the MMAs
    uint64_t* tfull = empty + C::STAGES;   // [2] accumulator complete
    uint64_t* tempty = tfull + 2;          // [2] accumulator stored
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
    const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
    const long long tiles = (a.N + C::BM - 1) / C::BM;
    if (tid == 0) {
        for (int i = 0; i < C::STAGES; ++i) { ttc::mbar_init(&full[i], 1); ttc::mbar_init(&conv[i], 4); ttc::mbar_init(&empty[i], 1); }
        for (int i = 0; i < 2; ++i) { ttc::mbar_init(&tfull[i], 1); ttc::mbar_init(&tempty[i], 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&xmap)) : "memory");
    }
    if (warp == 1) tmem_alloc_cols(tmem_slot, 512);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(40));
        if (lane == 0) {
            int s = 0; uint32_t ph = 0;
            for (long long t = blockIdx.x; t < tiles; t += gridDim.x)
                for (int kb = 0; kb < a.num_kb; ++kb) {
                    ttc::mbar_wait(&empty[s], ph ^ 1u);
                    uint8_t* st = sm + (size_t)s * C::STAGE_BYTES;
                    tgen::mbar_expect_tx(&full[s], (uint32_t)(C::X_BYTES + C::W_BYTES));
                    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                                 ::"r"(ttc::smem_u32(st)), "l"(reinterpret_cast<uint64_t>(&xmap)), "r"(kb * C::BK), "r"((int)(t * C::BM)),
                                   "r"(ttc::smem_u32(&full[s])) : "memory");
                    tgen::bulk_load(st + 2 * C::X_BYTES, a.wtiles + (size_t)kb * C::W_BYTES, (uint32_t)C::W_BYTES, &full[s]);
                    if (++s == C::STAGES) { s = 0; ph ^= 1u; }
                }
        }
    } else if (warp == 1) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(40));
        const uint32_t idesc = ttc::make_idesc_tf32(128, C::NQ);
        int s = 0; uint32_t ph = 0; int acc = 0; uint32_t aph = 0;
        for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
            for (int kb = 0; kb < a.num_kb; ++kb) {
                const bool g_first = kb % C::GROUP == 0, g_last = (kb % C::GROUP == C::GROUP - 1) || kb == a.num_kb - 1;
                if (g_first) ttc::mbar_wait(&tempty[acc], aph ^ 1u);
                ttc::mbar_wait(&conv[s], ph);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t st = ttc::smem_u32(sm) + (uint32_t)s * (uint32_t)C::STAGE_BYTES;
                const uint64_t xh = proj_desc_sw128(st), xl = proj_desc_sw128(st + C::X_BYTES);
                uint64_t wh = ttc::make_desc_noswz(st + 2 * C::X_BYTES, C::BK, 0), wl = ttc::make_desc_noswz(st + 2 * C::X_BYTES + C::W_BYTES / 2, C::BK, 0);
#pragma unroll
                for (int k = 0; k < C::BK / 8; ++k) {
                    ttc::mma3_ss(tmem + acc * C::NQ, xh + 2 * k, xl + 2 * k, wh, wl, idesc, (!g_first || k > 0) ? 1u : 0u);   // 8 floats = 32 B per k-step
                    wh += 16; wl += 16;
                }
                ttc::umma_commit_elect(&empty[s]);
                if (++s == C::STAGES) { s = 0; ph ^= 1u; }
                if (g_last) {
                    ttc::umma_commit_elect(&tfull[acc]);
                    if (++acc == 2) { acc = 0; aph ^= 1u; }
                }
            }
        }
    } else if (warp < 4) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(40));   // idle warps of group 0
    } else if (warp < 8) {
        // converters: thread = row of the tile; a row is 128 B = 8 chunks of 16 B, chunk c of row r at position c ^ (r % 8)
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(64));
        const int r = tid - 128;
        int s = 0; uint32_t ph = 0;
        for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
            // raw landmarks: this row's (ref, ipd) once per tile (nine L2 hits), kept in registers across the k-blocks; rows
            // past N are the tensor map's zero fill and stay zero
            const long long grow = t * C::BM + r;
            const bool map = a.ipd && grow < a.N;
            IpdRow nr{};
            if (map) nr = ipd_row(a.X + grow * a.ldx);
            for (int kb = 0; kb < a.num_kb; ++kb) {
                ttc::mbar_wait(&full[s], ph);
                uint8_t* xh = sm + (size_t)s * C::STAGE_BYTES + r * 128;
                uint8_t* xl = xh + C::X_BYTES;
#pragma unroll
                for (int cc = 0; cc < 8; ++cc) {
                    // the swizzle permutes whole 16-byte chunks, so position-wise processing is enough; the threads of 8
                    // consecutive rows take different chunk positions at a time (rows are 128 B apart: all on the same banks otherwise)
                    // (position c holds logical chunk c ^ (r & 7) = cc: features kb*32 + 4cc .. +3)
                    const int c = cc ^ (r & 7);
                    float4 v = *reinterpret_cast<float4*>(xh + 16 * c);
                    if (map) v = ipd_map4(v, nr, kb * C::BK + 4 * cc, a.F);
                    float4 h, l;
                    ttc::split_tf32_bits(v.x, h.x, l.x); ttc::split_tf32_bits(v.y, h.y, l.y);
                    ttc::split_tf32_bits(v.z, h.z, l.z); ttc::split_tf32_bits(v.w, h.w, l.w);
                    *reinterpret_cast<float4*>(xh + 16 * c) = h;
                    *reinterpret_cast<float4*>(xl + 16 * c) = l;
                }
                ttc::fence_async_smem();
                __syncwarp();
                if (lane == 0) tgen::mbar_arrive(&conv[s]);
                if (++s == C::STAGES) { s = 0; ph ^= 1u; }
            }
        }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(232));
        const int row = tid - 256;
        const uint32_t lane_addr = tmem + ((uint32_t)((warp & 3) * 32) << 16);
        int acc = 0; uint32_t aph = 0;
        for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
            float sum[C::NQ];
#pragma unroll
            for (int j = 0; j < C::NQ; ++j) sum[j] = 0.f;
            for (int kb = 0; kb < a.num_kb; kb += C::GROUP) {
                ttc::mbar_wait(&tfull[acc], aph);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
                for (int c0 = 0; c0 < C::NQ; c0 += 48) {
                    uint32_t v[48];
#pragma unroll
                    for (int x = 0; x < 6; ++x) tgen::tmem_ld8(lane_addr + acc * C::NQ + c0 + 8 * x, v + 8 * x);
                    tmem_load_wait();
#pragma unroll
                    for (int e = 0; e < 48; ++e) sum[c0 + e] += __uint_as_float(v[e]);
                }
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) tgen::mbar_arrive(&tempty[acc]);
                if (++acc == 2) { acc = 0; aph ^= 1u; }
            }
            float* slab = a.Q + (size_t)t * a.RPAD * 128 + row;
#pragma unroll
            for (int j = 0; j < C::NQ; ++j)
                if (j < a.RPAD) slab[(size_t)j * 128] = sum[j];
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) tmem_free_cols(tmem, 512);
}

// W2 tile images for the projection GEMM: k-block kb = rows r < NQ (zero beyond R), features kb*32 .. +31 (zero beyond F),
// hi plane then lo plane, UMMA no-swizzle K-major layout
__global__ void build_proj_tiles_kernel(const float* __restrict__ W2, int R, int F, int num_kb, uint8_t* __restrict__ img) {
    using C = ProjCfg;
    const long long total = (long long)num_kb * C::NQ * C::BK;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int kb = (int)(idx / (C::NQ * C::BK)), e = (int)(idx % (C::NQ * C::BK));
        const int r = e / C::BK, k = e % C::BK, f = kb * C::BK + k;
        const float v = (r < R && f < F) ? W2[(long long)r * F + f] : 0.f;
        float hi, lo;
        ttc::split_tf32(v, hi, lo);
        uint8_t* base = img + (size_t)kb * C::W_BYTES;
        *reinterpret_cast<float*>(base + ttc::op_offset(r, k, C::BK)) = hi;
        *reinterpret_cast<float*>(base + C::W_BYTES / 2 + ttc::op_offset(r, k, C::BK)) = lo;
    }
}

// register-only FFMA loop: measures the sustained FP32 FMA rate used as a roofline denominator
__global__ void __launch_bounds__(256) ffma_peak_kernel(float* out, int iters) {
    float a0 = threadIdx.x * 1e-3f, a1 = a0 + 1.f, a2 = a0 + 2.f, a3 = a0 + 3.f, a4 = a0 + 4.f, a5 = a0 + 5.f,
          a6 = a0 + 6.f, a7 = a0 + 7.f;
    const float b = 0.999f, c = 1e-3f;
#pragma unroll 1
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            a0 = fmaf(a0, b, c); a1 = fmaf(a1, b, c); a2 = fmaf(a2, b, c); a3 = fmaf(a3, b, c);
            a4 = fmaf(a4, b, c); a5 = fmaf(a5, b, c); a6 = fmaf(a6, b, c); a7 = fmaf(a7, b, c);
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

// same loop with three register operands per FFMA (multiplier and addend are run-time values held in registers,
// as in the fit kernel's inner loop): measures the register-file-limited FFMA rate
__global__ void __launch_bounds__(256) ffma_3reg_kernel(float* out, const float* in, int iters) {
    float a[8], b[8], c[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        a[k] = threadIdx.x * 1e-3f + k;
        b[k] = in[(threadIdx.x + k) & 255];
        c[k] = in[(threadIdx.x + 8 + k) & 255];
    }
#pragma unroll 1
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
#pragma unroll
            for (int k = 0; k < 8; ++k) a[k] = fmaf(a[k], b[(k + j) & 7], c[(k + 3 * j) & 7]);
        }
    }
    float r = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) r += a[k];
    out[blockIdx.x * blockDim.x + threadIdx.x] = r;
}

// back-to-back tcgen05.mma.kind::tf32 (M = 128, N = 256, K = 8, operands in shared memory, two TMEM accumulators):
// measures the dense TF32 tensor rate of the device, the denominator of the Tucker kernels' tensor roofline
__global__ void __launch_bounds__(128, 1) tf32_peak_kernel(int iters) {
    extern __shared__ __align__(1024) uint8_t psm[];
    constexpr int K = 64;
    uint8_t* a_t = psm;                                  // [128][64]
    uint8_t* b_t = psm + ttc::op_bytes(128, K);           // [256][64]
    uint64_t* bar = reinterpret_cast<uint64_t*>(b_t + ttc::op_bytes(256, K));
    uint32_t* slot = reinterpret_cast<uint32_t*>(bar + 1);
    const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    for (int i = tid; i < (ttc::op_bytes(128, K) + ttc::op_bytes(256, K)) / 4; i += 128) reinterpret_cast<float*>(psm)[i] = 1.0f + 1e-3f * (float)(i & 63);
    if (tid == 0) {
        ttc::mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) tmem_alloc_cols(slot, 512);
    ttc::fence_async_smem();
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *slot;
    if (warp == 0) {
        const uint32_t idesc = ttc::make_idesc_tf32(128, 256);
        for (int it = 0; it < iters; ++it) {
            uint64_t da = ttc::make_desc_noswz(ttc::smem_u32(a_t), K, 0), db = ttc::make_desc_noswz(ttc::smem_u32(b_t), K, 0);
#pragma unroll
            for (int k = 0; k < K / 8; ++k) {
                asm volatile(
                    "{\n\t.reg .pred p, e;\n\t"
                    "elect.sync _|e, 0xffffffff;\n\t"
                    "setp.ne.b32 p, %4, 0;\n\t"
                    "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                    ::"r"(tmem + (uint32_t)((k & 1) * 256)), "l"(da), "l"(db), "r"(idesc), "r"((uint32_t)(it > 0 || k > 1)) : "memory");
                da += 16; db += 16;
            }
        }
        ttc::umma_commit_elect(bar);
    }
    ttc::mbar_wait(bar, 0);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) tmem_free_cols(tmem, 512);
}

}  // namespace nlml

// =============================================================================================
// C ABI
// =============================================================================================
using namespace nlml;

struct nlml_tucker_plan {
    int device = 0;
    int ri = 0, ry = 0, rp = 0, rr = 0, F = 0, R = 0;
    int nA = 0, NAP = 0, nBCD = 0, nBCDp = 0;
    float* W2 = nullptr;
    float* S = nullptr;
    float* St = nullptr;
    TuckerArgs base{};
    bool fast = false;        // ranks (5,3,3,3): thread-per-sample kernel available
    bool cta_ok = false;      // CTA-per-sample kernel usable (its working set fits shared memory)
    bool gen_ok = false;      // run-time-rank tensor-core kernel usable (tucker_gen.cuh)
    tgen::GenCfg gen{};
    uint8_t* proj_tiles = nullptr;          // (5,3,3,3): W2 tile images of the tensor-core projection GEMM
    float* q_pre = nullptr;                 // its output for the batch in flight (CTA-blocked slabs), grown on demand
    int64_t q_pre_rows = 0;
    cudaEvent_t q_pre_done = nullptr;
    double rows64[3][4 * kMaxModeRank] = {};   // the cosine rows in float64, as the reference's Powell objective uses them
    uint8_t* tc_ops = nullptr;              // (5,3,3,3) tensor-core kernel: image of its two constant B operands
    uint8_t* gen_tiles = nullptr;           // tile images of S (hi/lo, UMMA layout), streamed by TMA
    float* q_ws[3] = {nullptr, nullptr, nullptr};   // q = W2 x slabs: [0],[1] host-pipeline slots, [2] device-buffer calls
    int64_t q_rows[3] = {0, 0, 0};
    cudaEvent_t q_done = nullptr;           // orders device-buffer calls issued on different streams over q_ws[2]
    bool st_in_smem = false;  // CTA kernel keeps St in shared memory
    size_t cta_smem = 0;
    int num_sms = 148;
    int64_t launches = 0;
    // host-buffer path
    cudaStream_t streams[2] = {nullptr, nullptr};
    float* x_dev[2] = {nullptr, nullptr};
    float* p_dev[2] = {nullptr, nullptr};
    float* p_stage[2] = {nullptr, nullptr};   // pinned: a D2H copy into pageable user memory would block the host
                                              // thread until the chunk's kernel is done and serialise the pipeline
    int64_t chunk = 0;
    int64_t host_rows = 0;   // capacity of x_dev / p_dev / p_stage
};

namespace {
constexpr int kTpsThreads = 128;   // threads per CTA of the thread-per-sample kernel
constexpr int kTpsSamples = 1;     // samples per thread.  2 halves the shared-memory wavefronts per sample but the q
                                   // buffer then limits the SM to 4 warps: measured 740 k poses/s against 919 k at 1.
constexpr int kTpsMinBlocks = 2;
constexpr int kSolveMinBlocks = 2;   // converged-solve variant of the same kernel
constexpr int kTpsBigThreads = 384;  // TMEM-resident-q variant: one 12-warp CTA per SM
// measured: 913 k poses/s with q in TMEM (12 warps/SM) vs 912 k with q in shared memory (8 warps/SM) -- the kernel
// is bound by the 3-register-operand FFMA rate, not by latency -- so the variant is opt-in (kernel_hint 4) only
constexpr int kCtaThreads = 128;
constexpr int kWpsWarps = 4;
// The tensor-core kernel runs a whole wave (up to 128 samples on each SM) in the time of its 3000-step chain: 4.4-4.7 ms for
// ANY batch up to 18 944 samples on a 148-SM B200 (round 2 kernel), against 2.8 / 3.6 / 7.2 / 14.4 ms for 256 / 1024 / 2048 /
// 4096 samples in the warp-per-sample kernel and 23.5 ms per wave in the FP32 thread-per-sample kernel.  So it takes over
// from 1536 samples (round 1: from two full waves, when its wave took 17 ms); below that the warp-per-sample kernel
// finishes sooner, and the thread-per-sample kernel is the FP32 reference on request (kernel_hint 1).
inline int64_t tc_crossover(const nlml_tucker_plan*) { return 1536; }
constexpr int64_t kWpsCrossover = 8192;  // (only reachable when the tensor-core kernel is not eligible)
using TpsDefault = TpsCfg<5, 3, 3, 3, kTpsThreads, kTpsSamples>;
using TpsBig = TpsCfg<5, 3, 3, 3, kTpsBigThreads, 1, true>;
size_t wps_smem_bytes(int F) { return sizeof(float) * kWpsWarps * ((F + 3) / 4 * 4 + 64); }

// ---- run-time-rank tensor-core kernel: per-plan configuration (TMEM columns, shared-memory ring, block size) ----
constexpr int kGenSmemMax = 232448;   // 227 KB of dynamic shared memory per CTA
// ranks: roll <= 8, others <= tgen::kMaxRank (checked by gen_config_for)
bool choose_gen_config(int ri, int ry, int rp, int rr, tgen::GenCfg& best) {
    tgen::GenCfg b{};
    b.ri = ri; b.ry = ry; b.rp = rp; b.rr = rr; b.R = ri * ry * rp * rr;
    b.rrmax = rr <= 5 ? 5 : 8;
    b.nA = tri(ri); b.KA = (b.nA + 15) / 16 * 16; b.NA16 = b.KA;   // FP16 MMAs: K in steps of 16
    b.nC = tri(rp); b.nBC = tri(ry) * tri(rp);
    b.nDp = (tri(b.rrmax) + 7) / 8 * 8;
    b.NP = 3 + ri;
    b.t_p = 0; b.t_gx = b.NP; b.t_gl = 2 * b.NP; b.t_cy = 3 * b.NP; b.t_dcy = b.t_cy + ry; b.t_cp = b.t_dcy + ry;
    b.t_dcp = b.t_cp + rp; b.t_rows = b.t_dcp + rp;
    const int tab_bytes = b.t_rows * tgen::kSamples * 4, bar_bytes = 1024;
    // the highest-scoring feasible candidate, whatever its sign: roll rank 1 fills 1 of every 16 columns, so all of its
    // candidates score below zero (ties keep the first candidate)
    double best_score = -HUGE_VAL;
    bool found = false;
#ifdef NLML_GEN_TUNE
    // development build only (-DNLML_GEN_TUNE): pin parts of the configuration from the environment for sweeps
    auto pin = [](const char* name) { const char* e = std::getenv(name); return e ? std::atoi(e) : 0; };
    const int pin_bcp = pin("NLML_GEN_BCP"), pin_tb = pin("NLML_GEN_TB"), pin_gb = pin("NLML_GEN_GB"), pin_yb = pin("NLML_GEN_YB"),
              pin_slots = pin("NLML_GEN_SLOTS"), pin_ytm = pin("NLML_GEN_YTM");   // YTM: 1 = shared memory, 2 = tensor memory
#else
    constexpr int pin_bcp = 0, pin_tb = 0, pin_gb = 0, pin_yb = 0, pin_slots = 0, pin_ytm = 0;
#endif
    for (int BCP = 1; BCP <= 32; ++BCP) {
        if (pin_bcp && BCP != pin_bcp) continue;
        const int NB = (BCP * b.nDp + 15) / 16 * 16;   // MMA N granularity; pad columns hold zeros in the tiles and the operand
        if (NB > 256) continue;
        const int nblocks = (b.nBC + BCP - 1) / BCP;
        for (int ytm = 1; ytm >= 0; --ytm)   // the YPR operand in tensor memory (preferred: shared-memory bandwidth is the scarce resource) or in shared memory
        for (int tbufs = 2; tbufs >= 1; --tbufs)
            for (int gbufs = 2; gbufs >= 1; --gbufs) {
                if ((pin_tb && tbufs != pin_tb) || (pin_gb && gbufs != pin_gb)) continue;
                for (int ybufs = 2; ybufs >= 1; --ybufs) {
                    // tensor-memory columns: D_G buffers, UU operand (KA/2 packed hi + KA/2 lo), D_T buffers, YPR operand (NB/2 + NB/2)
                    const int cols = gbufs * b.NA16 + b.KA + tbufs * NB + (ytm ? ybufs * NB : 0);
                    if (cols > 512) continue;
                    // FP16 hi + lo planes: 4 bytes per element
                    const int tt = NB * b.KA * 4, gt = b.NA16 * NB * 4, ypr = ytm ? 0 : ybufs * NB * tgen::kSamples * 4;
                    const int avail = kGenSmemMax - 1024 - ypr - tab_bytes - bar_bytes;
                    if (avail < tt + gt) continue;
                    if (pin_yb && ybufs != pin_yb) continue;
                    if (pin_ytm && ytm != pin_ytm - 1) continue;
                    const bool resident = !pin_slots && nblocks <= tgen::kMaxSlots && (long long)nblocks * (tt + gt) <= avail;
                    int slots = resident ? nblocks : std::min(4, avail / (tt + gt));
                    if (pin_slots) slots = std::min(slots, pin_slots);
                    const double waste = (double)nblocks * NB / ((double)b.nBC * tri(rr)) - 1.0;   // padded columns issued per useful one
                    // (streamed tiles: the per-block handshakes and TMA round trips amortise over wider blocks -- measured on
                    // (16,8,8,8): NB = 80 with two ring slots 3226 poses/s, NB = 48 with three 2370)
                    const double score = (resident ? 40.0 : 10.0 * std::min(slots, 3)) + 6.0 * ybufs + 4.0 * tbufs + 3.0 * gbufs + 30.0 * ytm +
                                         (resident ? 0.25 : 0.6) * std::min(NB, 128) - 20.0 * waste;
                    if (found && score <= best_score) continue;
                    found = true;
                    best_score = score;
                    best = b;
                    best.BCP = BCP; best.NB = NB; best.nblocks = nblocks;
                    best.tbufs = tbufs; best.gbufs = gbufs; best.ybufs = ybufs; best.ypr_tmem = ytm;
                    best.tslots = best.gslots = slots; best.resident = resident ? 1 : 0;
                    best.tt_bytes = tt; best.gt_bytes = gt;
                    best.col_g = 0; best.col_a = gbufs * b.NA16; best.col_t = best.col_a + b.KA; best.col_y = best.col_t + tbufs * NB;
                    best.off_tring = 0;
                    best.off_gring = slots * tt;
                    best.off_ypr = best.off_gring + slots * gt;
                    best.off_tab = best.off_ypr + ypr;
                    best.off_bar = best.off_tab + tab_bytes;
                    best.smem_bytes = best.off_bar + bar_bytes;
                }
            }
    }
    return found;
}

// Configuration of the run-time-rank tensor-core kernel for a rank set, or why it has none (nullptr on success).  Plan
// creation and nlml_debug_gen_config both decide through this function.
constexpr double kGenMaxTileBytes = 3.0e9;   // tile images of S kept on the device
const char* gen_config_for(int ri, int ry, int rp, int rr, tgen::GenCfg& cfg) {
    static thread_local char why[160];
    if (rr > 8 || ri > tgen::kMaxRank || ry > tgen::kMaxRank || rp > tgen::kMaxRank) {
        std::snprintf(why, sizeof(why), "the run-time-rank tensor-core kernel serves roll ranks <= 8 and other ranks <= %d "
                      "(ranks %d,%d,%d,%d)", tgen::kMaxRank, ri, ry, rp, rr);
        return why;
    }
    if (!choose_gen_config(ri, ry, rp, rr, cfg)) {
        std::snprintf(why, sizeof(why), "no block size of the run-time-rank tensor-core kernel fits tensor memory and "
                      "shared memory for ranks %d,%d,%d,%d", ri, ry, rp, rr);
        return why;
    }
    const double tile_bytes = (double)cfg.nblocks * ((double)cfg.tt_bytes + cfg.gt_bytes);
    if (tile_bytes > kGenMaxTileBytes) {
        std::snprintf(why, sizeof(why), "the run-time-rank tensor-core kernel's tile images of ranks %d,%d,%d,%d would "
                      "take %.2f GB (limit %.1f GB)", ri, ry, rp, rr, tile_bytes * 1e-9, kGenMaxTileBytes * 1e-9);
        return why;
    }
    return nullptr;
}

template <int RRMAX, int NA16MAX>
int launch_gen_instance(const tgen::GenArgs& a, unsigned grid, cudaStream_t st, bool set_attr) {
    auto kern = tgen::tucker_fit_gen_kernel<RRMAX, NA16MAX>;
    if (set_attr) {
        NLML_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, a.c.smem_bytes));
        return 0;
    }
    kern<<<grid, tgen::kThreads, a.c.smem_bytes, st>>>(a);
    return 0;
}
int dispatch_gen(const tgen::GenArgs& a, unsigned grid, cudaStream_t st, bool set_attr) {
    const bool small_a = a.c.NA16 <= 48;
    if (a.c.rrmax == 5) return small_a ? launch_gen_instance<5, 48>(a, grid, st, set_attr) : launch_gen_instance<5, 144>(a, grid, st, set_attr);
    return small_a ? launch_gen_instance<8, 48>(a, grid, st, set_attr) : launch_gen_instance<8, 144>(a, grid, st, set_attr);
}

// samples per pass of the generic kernel: whole waves of 128-sample CTAs, q slabs of at most ~1.5 GB
int64_t gen_chunk(const nlml_tucker_plan* pl) {
    const int64_t wave = (int64_t)pl->num_sms * tgen::kSamples;
    const int64_t waves = std::max<int64_t>(1, (int64_t)(1.5e9 / ((double)pl->R * 4.0 * (double)wave)));
    return std::min<int64_t>(waves, 8) * wave;
}

int launch_gen(nlml_tucker_plan* pl, const float* X, int64_t N, int64_t ldx, int ipd, int iters, float lr, float clip, float* P,
               int64_t ldp, int ws_slot, cudaStream_t st) {
    const int64_t chunk = gen_chunk(pl);
    const int64_t want = std::min<int64_t>(chunk, ceil_div(N, tgen::kSamples) * tgen::kSamples);
    if (pl->q_rows[ws_slot] < want) {
        if (pl->q_rows[ws_slot]) NLML_CUDA(cudaDeviceSynchronize());
        pl->q_rows[ws_slot] = 0;
        cudaFree(pl->q_ws[ws_slot]);
        pl->q_ws[ws_slot] = nullptr;
        NLML_CUDA(cudaMalloc(&pl->q_ws[ws_slot], sizeof(float) * (size_t)want * pl->R));
        pl->q_rows[ws_slot] = want;
    }
    if (ws_slot == 2) {   // device-buffer calls may come from different streams: they share one q workspace
        if (!pl->q_done) NLML_CUDA(cudaEventCreateWithFlags(&pl->q_done, cudaEventDisableTiming));
        else NLML_CUDA(cudaStreamWaitEvent(st, pl->q_done, 0));
    }
    tgen::GenArgs a{};
    a.q = pl->q_ws[ws_slot];
    a.tiles = pl->gen_tiles;
    a.ldp = ldp;
    a.T = iters; a.lr = lr; a.clip = clip;
    a.c = pl->gen;
    std::memcpy(a.rows_y, pl->base.rows_y, sizeof(a.rows_y));
    std::memcpy(a.rows_p, pl->base.rows_p, sizeof(a.rows_p));
    std::memcpy(a.rows_r, pl->base.rows_r, sizeof(a.rows_r));
    for (int64_t s0 = 0; s0 < N; s0 += chunk) {
        const int64_t n = std::min<int64_t>(chunk, N - s0);
        const float* x = X + s0 * ldx;
        const int vec_ok = (pl->F % 4 == 0) && (ldx % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
        const unsigned ctas = (unsigned)ceil_div(n, tgen::kSamples);
        tgen::tucker_project_kernel<<<dim3(ctas, (unsigned)ceil_div(pl->R, 64)), 256, ipd ? sizeof(IpdRow) * tgen::kSamples : 0, st>>>(x, n, ldx, pl->W2, pl->R, pl->F, vec_ok, pl->q_ws[ws_slot], ipd);
        a.P = P + s0 * ldp;
        a.N = n;
        if (int rc = dispatch_gen(a, ctas, st, false)) return rc;
        NLML_CUDA(cudaGetLastError());
        pl->launches += 2;
    }
    if (ws_slot == 2) NLML_CUDA(cudaEventRecord(pl->q_done, st));
    return 0;
}

constexpr int64_t kProjMinRows = 4096;   // below this the consumer's own phase A is as fast (one partial wave)
int project_tc(nlml_tucker_plan* pl, const float* X, int64_t N, int64_t ldx, int ipd, cudaStream_t st, const float** Qout,
               int64_t min_rows = kProjMinRows);

// ipd: X holds raw landmarks; every phase A below reads it through the IPD normalisation (common.cuh)
int launch_fit(nlml_tucker_plan* pl, const float* X, int64_t N, int64_t ldx, int ipd, int iters, float lr, float clip,
               float* P, int64_t ldp, int hint, cudaStream_t st, int ws_slot = 2, int64_t proj_min_rows = kProjMinRows) {
    if (N == 0) return 0;
    // run-time-rank tensor-core kernel: asked for, or the default for every rank set without compiled kernels
    if (hint == 6 && !pl->gen_ok) {
        tgen::GenCfg unused{};
        return set_error(NLML_E_UNSUPPORTED, "%s", gen_config_for(pl->ri, pl->ry, pl->rp, pl->rr, unused));
    }
    if (hint == 2 && !pl->cta_ok)
        return set_error(NLML_E_UNSUPPORTED, "core too large for the CTA-per-sample kernel's shared-memory working set");
    if (hint == 6 || (hint == 0 && !pl->fast && pl->gen_ok && (N >= 32 || !pl->cta_ok)))
        return launch_gen(pl, X, N, ldx, ipd, iters, lr, clip, P, ldp, ws_slot, st);
    TuckerArgs a = pl->base;
    a.X = X;
    a.N = N;
    a.ldx = ldx;
    a.ipd = ipd;
    a.P = P;
    a.ldp = ldp;
    a.T = iters;
    a.lr = lr;
    a.clip = clip;
    a.vec_ok = (pl->F % 4 == 0) && (ldx % 4 == 0) && ((reinterpret_cast<uintptr_t>(X) & 15) == 0);
#ifdef NLML_TC_DBG
    if (const char* e = std::getenv("NLML_TUCKER_DBG")) a.dbg = std::atoi(e);   // development build only
#endif
    // crossover: below ~one thread-per-sample wave the 3000-step chain is latency bound and the
    // CTA-per-sample kernel finishes sooner
    // large batches: the tensor-core iteration kernel (2.6 M poses/s) beats the FP32 thread-per-sample kernel (0.92 M)
    const bool use_tc = pl->fast && (hint == 5 || (hint == 0 && N >= tc_crossover(pl)));
    const bool use_tps = pl->fast && !use_tc && (hint == 1 || hint == 4 || (hint == 0 && N >= kWpsCrossover));
    const bool use_wps = pl->fast && !use_tc && (hint == 3 || (hint == 0 && N < kWpsCrossover));
    if (!pl->fast && !pl->cta_ok)
        return set_error(NLML_E_UNSUPPORTED, "core too large for the CTA-per-sample kernel's shared-memory working set");
    if ((hint == 1 || hint == 3 || hint == 4 || hint == 5) && !pl->fast)
        return set_error(NLML_E_UNSUPPORTED, "thread/warp-per-sample kernels are built for ranks (5,3,3,3) only");
    if (use_tc) {
        // phase A (q = W2 x) as a 3xTF32 tcgen05 GEMM of its own when the layout allows TMA; the kernel then only copies its slab
        if (int rc = project_tc(pl, X, N, ldx, ipd, st, &a.Qpre, proj_min_rows)) return rc;
        tucker_fit_tc_kernel<<<(unsigned)ceil_div(N, TcFitCfg::THREADS), 2 * TcFitCfg::THREADS, TcFitCfg::SMEM_BYTES, st>>>(a);
        if (a.Qpre) NLML_CUDA(cudaEventRecord(pl->q_pre_done, st));
    } else if (use_wps) {
        auto kern = tucker_fit_wps_kernel<5, 3, 3, 3, kWpsWarps>;
        const unsigned grid = (unsigned)ceil_div(N, kWpsWarps);
        // the shared-memory limit is a property of the function, not of the plan: a plan with a smaller F created since
        // may have lowered it (as for the Powell kernel, it is set at each launch)
        NLML_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wps_smem_bytes(pl->F)));
        kern<<<grid, 32 * kWpsWarps, wps_smem_bytes(pl->F), st>>>(a);
    } else if (use_tps) {
        if (hint == 4) {
            auto kern = tucker_fit_tps_kernel<5, 3, 3, 3, kTpsBigThreads, 1, 1, true>;
            kern<<<(unsigned)ceil_div(N, TpsBig::SAMPLES), kTpsBigThreads, TpsBig::SMEM_BYTES, st>>>(a);
        } else {
            auto kern = tucker_fit_tps_kernel<5, 3, 3, 3, kTpsThreads, kTpsSamples, kTpsMinBlocks, false>;
            kern<<<(unsigned)ceil_div(N, TpsDefault::SAMPLES), kTpsThreads, TpsDefault::SMEM_BYTES, st>>>(a);
        }
    } else {
        auto kern = tucker_fit_cta_kernel<kCtaThreads>;
        NLML_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl->cta_smem));   // as above
        kern<<<(unsigned)N, kCtaThreads, pl->cta_smem, st>>>(a, pl->st_in_smem ? 1 : 0);
    }
    NLML_CUDA(cudaGetLastError());
    pl->launches += 1;
    return 0;
}

// q = W2 x for the batch through tucker_project_tc_kernel.  *Qout stays null (the consumer runs its own phase A) when X
// cannot be described by a tensor map (row pitch or base not 16-byte aligned) or the batch is small.
typedef CUresult (*EncodeTiledFnT)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
int project_tc(nlml_tucker_plan* pl, const float* X, int64_t N, int64_t ldx, int ipd, cudaStream_t st, const float** Qout, int64_t min_rows) {
    *Qout = nullptr;
    if (!pl->fast || !pl->proj_tiles || N < min_rows || (ldx % 4) != 0 || (reinterpret_cast<uintptr_t>(X) & 15) != 0) return 0;
    static EncodeTiledFnT encode = nullptr;
    if (!encode) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) return 0;
        encode = reinterpret_cast<EncodeTiledFnT>(p);
    }
    const int64_t tiles = ceil_div(N, ProjCfg::BM);
    if (pl->q_pre_rows < tiles * ProjCfg::BM) {
        if (pl->q_pre_rows) NLML_CUDA(cudaDeviceSynchronize());
        pl->q_pre_rows = 0;
        cudaFree(pl->q_pre);
        pl->q_pre = nullptr;
        NLML_CUDA(cudaMalloc(&pl->q_pre, sizeof(float) * (size_t)tiles * ProjCfg::BM * 136));
        pl->q_pre_rows = tiles * ProjCfg::BM;
    }
    if (!pl->q_pre_done) NLML_CUDA(cudaEventCreateWithFlags(&pl->q_pre_done, cudaEventDisableTiming));
    else NLML_CUDA(cudaStreamWaitEvent(st, pl->q_pre_done, 0));   // one q buffer per plan: calls on other streams wait for its last reader
    CUtensorMap xmap;
    cuuint64_t dims[2] = {(cuuint64_t)pl->F, (cuuint64_t)N};
    cuuint64_t strides[1] = {(cuuint64_t)ldx * 4};
    cuuint32_t box[2] = {(cuuint32_t)ProjCfg::BK, (cuuint32_t)ProjCfg::BM};
    cuuint32_t estr[2] = {1, 1};
    if (encode(&xmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(X), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
        return 0;
    ProjArgs pa{};
    pa.N = N; pa.F = pl->F; pa.RPAD = 136; pa.num_kb = (pl->F + ProjCfg::BK - 1) / ProjCfg::BK;
    pa.wtiles = pl->proj_tiles; pa.Q = pl->q_pre;
    pa.ipd = ipd; pa.X = X; pa.ldx = ldx;
    const unsigned grid = (unsigned)std::min<int64_t>(tiles, pl->num_sms);
    tucker_project_tc_kernel<<<grid, ProjCfg::THREADS, ProjCfg::SMEM_BYTES, st>>>(xmap, pa);
    NLML_CUDA(cudaGetLastError());
    pl->launches += 1;
    *Qout = pl->q_pre;
    return 0;
}

// converged fit (SURVEY.md section 8f row 1): thread-per-sample kernel, phase B' = tucker_lm_solve
int launch_solve(nlml_tucker_plan* pl, const float* X, int64_t N, int64_t ldx, int ipd, int max_evals, float* P, int64_t ldp,
                 int* evals, cudaStream_t st, int64_t proj_min_rows = kProjMinRows) {
    if (N == 0) return 0;
    if (!pl->fast) return set_error(NLML_E_UNSUPPORTED, "the converged solve is built for ranks (5,3,3,3) only");
    TuckerArgs a = pl->base;
    a.X = X;
    a.N = N;
    a.ldx = ldx;
    a.ipd = ipd;
    a.P = P;
    a.ldp = ldp;
    a.vec_ok = (pl->F % 4 == 0) && (ldx % 4 == 0) && ((reinterpret_cast<uintptr_t>(X) & 15) == 0);
    a.lm = lm_default_options();
    if (max_evals > 0) a.lm.max_evals = max_evals;
    a.evals = evals;
    if (int rc = project_tc(pl, X, N, ldx, ipd, st, &a.Qpre, proj_min_rows)) return rc;   // phase A as a tensor-core GEMM when the layout allows TMA
    auto kern = tucker_fit_tps_kernel<5, 3, 3, 3, kTpsThreads, 1, kSolveMinBlocks, false, true>;
    kern<<<(unsigned)ceil_div(N, TpsDefault::SAMPLES), kTpsThreads, TpsDefault::SMEM_BYTES, st>>>(a);
    NLML_CUDA(cudaGetLastError());
    if (a.Qpre) NLML_CUDA(cudaEventRecord(pl->q_pre_done, st));
    pl->launches += 1;
    return 0;
}

// HOST buffers: chunk the batch and overlap H2D copy / kernel / D2H copy on two internal streams.
template <class Launch>
int host_pipeline(nlml_tucker_plan* pl, const float* X_host, int64_t N, int64_t ldx, float* P_out_host, int64_t ldp,
                  Launch&& launch) {
    const int np = 3 + pl->ri;
    if (!pl->streams[0]) {
        pl->chunk = (int64_t)pl->num_sms * TcFitCfg::THREADS * 8;   // 8 waves of the tensor-core kernel per chunk
        if (!pl->fast && pl->gen_ok) pl->chunk = gen_chunk(pl);
        for (int i = 0; i < 2; ++i) NLML_CUDA(cudaStreamCreateWithFlags(&pl->streams[i], cudaStreamNonBlocking));
    }
    // staging grows to the largest chunk seen (single-sample calls through TD_Tester.Test stay small)
    const int64_t want = std::min<int64_t>(pl->chunk, ceil_div(std::max<int64_t>(N, 1), 128) * 128);
    if (pl->host_rows < want) {
        if (pl->host_rows) NLML_CUDA(cudaDeviceSynchronize());
        pl->host_rows = 0;   // nothing below is usable until every allocation has succeeded
        for (int i = 0; i < 2; ++i) {
            cudaFree(pl->x_dev[i]);
            cudaFree(pl->p_dev[i]);
            if (pl->p_stage[i]) cudaFreeHost(pl->p_stage[i]);
            pl->x_dev[i] = pl->p_dev[i] = pl->p_stage[i] = nullptr;
        }
        for (int i = 0; i < 2; ++i) {
            NLML_CUDA(cudaMalloc(&pl->x_dev[i], sizeof(float) * (size_t)want * pl->F));
            NLML_CUDA(cudaMalloc(&pl->p_dev[i], sizeof(float) * (size_t)want * np));
            NLML_CUDA(cudaMallocHost(&pl->p_stage[i], sizeof(float) * (size_t)want * np));
        }
        pl->host_rows = want;
    }
    // results land in pinned staging and are handed to the caller's buffer when the slot comes round again
    struct Pending { int64_t s0 = 0, n = 0; } pending[2];
    auto drain = [&](int slot) -> int {
        if (!pending[slot].n) return 0;
        NLML_CUDA(cudaStreamSynchronize(pl->streams[slot]));
        const float* src = pl->p_stage[slot];
        float* dst = P_out_host + pending[slot].s0 * ldp;
        if (ldp == np) {
            std::memcpy(dst, src, sizeof(float) * np * pending[slot].n);
        } else {
            for (int64_t r = 0; r < pending[slot].n; ++r) std::memcpy(dst + r * ldp, src + r * np, sizeof(float) * np);
        }
        pending[slot].n = 0;
        return 0;
    };
    // Chunk sizes ramp up (1, 2, 4 waves, then the full 8): only the first, small copy is exposed; every later copy is
    // shorter than the kernel of the chunk before it (a wave is ~2 ms of PCIe against ~7 ms of fit at T = 3000).
    int slot = 0, k = 0;
    const int64_t wave = (int64_t)pl->num_sms * TcFitCfg::THREADS;
    for (int64_t s0 = 0, n = 0; s0 < N; s0 += n, slot ^= 1, ++k) {
        n = std::min<int64_t>(k < 3 ? std::min<int64_t>(pl->chunk, wave << k) : pl->chunk, N - s0);
        cudaStream_t st = pl->streams[slot];
        if (int rc = drain(slot)) return rc;   // also makes the reuse of this slot's device buffers safe
        if (ldx == pl->F)   // contiguous rows: one linear DMA instead of a pitched copy
            NLML_CUDA(cudaMemcpyAsync(pl->x_dev[slot], X_host + s0 * ldx, sizeof(float) * pl->F * n, cudaMemcpyHostToDevice, st));
        else
            NLML_CUDA(cudaMemcpy2DAsync(pl->x_dev[slot], sizeof(float) * pl->F, X_host + s0 * ldx, sizeof(float) * ldx,
                                        sizeof(float) * pl->F, (size_t)n, cudaMemcpyHostToDevice, st));
        if (int rc = launch(pl->x_dev[slot], n, pl->p_dev[slot], st, slot)) return rc;
        NLML_CUDA(cudaMemcpyAsync(pl->p_stage[slot], pl->p_dev[slot], sizeof(float) * np * n, cudaMemcpyDeviceToHost, st));
        pending[slot].s0 = s0;
        pending[slot].n = n;
    }
    if (int rc = drain(slot)) return rc;        // older chunk first
    if (int rc = drain(slot ^ 1)) return rc;
    return 0;
}
}  // namespace

extern "C" int nlml_abi_version(void) { return NLML_ABI_VERSION; }
extern "C" const char* nlml_last_error(void) { return last_error_buf(); }

extern "C" int nlml_tucker_plan_create(const float* W_host, int r_id, int r_y, int r_p, int r_r, int F,
                                       const double* rows_y, const double* rows_p, const double* rows_r,
                                       int device, nlml_tucker_plan** plan_out) {
    if (!W_host || !rows_y || !rows_p || !rows_r || !plan_out)
        return set_error(NLML_E_INVALID, "null pointer argument");
    if (r_id < 1 || r_y < 1 || r_p < 1 || r_r < 1 || F < 1)
        return set_error(NLML_E_INVALID, "ranks and F must be positive");
    if (r_id > kMaxModeRank || r_y > kMaxModeRank || r_p > kMaxModeRank || r_r > kMaxModeRank)
        return set_error(NLML_E_UNSUPPORTED, "per-mode rank limit is %d", kMaxModeRank);
    if (int rc = check_device(device)) return rc;
    DeviceGuard guard(device);
    if (!guard.ok) return set_error(NLML_E_NO_DEVICE, "cudaSetDevice(%d) failed", device);

    // owned until the end of this function: every early error return below frees the plan and its device buffers
    struct PlanOwner {
        nlml_tucker_plan* p;
        ~PlanOwner() { if (p) nlml_tucker_plan_destroy(p); }
    } owner{new nlml_tucker_plan()};
    nlml_tucker_plan* pl = owner.p;
    pl->device = device;
    pl->ri = r_id; pl->ry = r_y; pl->rp = r_p; pl->rr = r_r; pl->F = F;
    pl->R = r_id * r_y * r_p * r_r;
    pl->nA = tri(r_id);
    pl->NAP = (pl->nA + 3) / 4 * 4;
    pl->nBCD = tri(r_y) * tri(r_p) * tri(r_r);
    pl->nBCDp = (pl->nBCD + 31) / 32 * 32;
    const char* gen_why = gen_config_for(r_id, r_y, r_p, r_r, pl->gen);
    pl->gen_ok = gen_why == nullptr;
    if (pl->nBCD > kMaxBCD && !pl->gen_ok) {
        return set_error(NLML_E_UNSUPPORTED, "angle-mode ranks (%d,%d,%d) give %d folded entries per identity pair, above the "
                         "CTA-per-sample kernel's limit %d, and %s", r_y, r_p, r_r, pl->nBCD, kMaxBCD, gen_why);
    }
    cudaDeviceProp prop;
    NLML_CUDA(cudaGetDeviceProperties(&prop, device));
    pl->num_sms = prop.multiProcessorCount;

    const size_t w_bytes = sizeof(float) * (size_t)pl->R * F;
    struct DevScratch {   // the float64 Gram matrix is only needed while the folded tensor is built
        double* p = nullptr;
        ~DevScratch() { cudaFree(p); }
    } gram;
    double*& M = gram.p;
    NLML_CUDA(cudaMalloc(&pl->W2, w_bytes));
    NLML_CUDA(cudaMalloc(&pl->S, sizeof(float) * (size_t)pl->nBCD * pl->NAP));
    NLML_CUDA(cudaMalloc(&pl->St, sizeof(float) * (size_t)pl->nA * pl->nBCDp));
    NLML_CUDA(cudaMalloc(&M, sizeof(double) * (size_t)pl->R * pl->R));
    NLML_CUDA(cudaMemcpy(pl->W2, W_host, w_bytes, cudaMemcpyHostToDevice));
    NLML_CUDA(cudaMemset(pl->S, 0, sizeof(float) * (size_t)pl->nBCD * pl->NAP));
    NLML_CUDA(cudaMemset(pl->St, 0, sizeof(float) * (size_t)pl->nA * pl->nBCDp));
    {
        const int n = pl->R * pl->R;
        if (pl->R > 512) {
            const unsigned nb = (unsigned)ceil_div(pl->R, 64);
            tgen::gram_tiled_kernel<<<dim3(nb, nb), 256>>>(pl->W2, pl->R, F, M);
        } else {
            gram_kernel<<<(n + 127) / 128, 128>>>(pl->W2, pl->R, F, M);
        }
        const int m = pl->nA * pl->nBCD;
        fold_kernel<<<(m + 127) / 128, 128>>>(M, r_id, r_y, r_p, r_r, pl->NAP, pl->nBCDp, pl->S, pl->St);
        NLML_CUDA(cudaGetLastError());
        NLML_CUDA(cudaDeviceSynchronize());
        pl->launches += 2;
    }

    TuckerArgs& a = pl->base;
    a.W2 = pl->W2; a.S = pl->S; a.St = pl->St;
    a.F = F; a.ri = r_id; a.ry = r_y; a.rp = r_p; a.rr = r_r; a.nBCDp = pl->nBCDp;
    for (int j = 0; j < 4 * r_y; ++j) pl->rows64[0][j] = rows_y[j];
    for (int j = 0; j < 4 * r_p; ++j) pl->rows64[1][j] = rows_p[j];
    for (int j = 0; j < 4 * r_r; ++j) pl->rows64[2][j] = rows_r[j];
    for (int j = 0; j < 4 * r_y; ++j) a.rows_y[j] = (float)rows_y[j];  // f64 -> f32, TD_Tester.py:172-174
    for (int j = 0; j < 4 * r_p; ++j) a.rows_p[j] = (float)rows_p[j];
    for (int j = 0; j < 4 * r_r; ++j) a.rows_r[j] = (float)rows_r[j];

    pl->fast = (r_id == 5 && r_y == 3 && r_p == 3 && r_r == 3);
    if (pl->fast) {
        auto kern = tucker_fit_tps_kernel<5, 3, 3, 3, kTpsThreads, kTpsSamples, kTpsMinBlocks, false>;
        NLML_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TpsDefault::SMEM_BYTES));
        NLML_CUDA(cudaFuncSetAttribute(tucker_fit_tps_kernel<5, 3, 3, 3, kTpsThreads, 1, kSolveMinBlocks, false, true>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TpsDefault::SMEM_BYTES));
        NLML_CUDA(cudaFuncSetAttribute(tucker_fit_tps_kernel<5, 3, 3, 3, kTpsBigThreads, 1, 1, true>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TpsBig::SMEM_BYTES));
        NLML_CUDA(cudaFuncSetAttribute(tucker_fit_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TcFitCfg::SMEM_BYTES));
        NLML_CUDA(cudaMalloc(&pl->tc_ops, TcFitCfg::OFF_AV));
        {   // power-of-two scale of the S operand image: the largest |S| lands in [2^13, 2^14) of FP16's range
            std::vector<float> Sh((size_t)pl->nBCD * pl->NAP);
            NLML_CUDA(cudaMemcpy(Sh.data(), pl->S, sizeof(float) * Sh.size(), cudaMemcpyDeviceToHost));
            float smax = 0.f;
            for (float v : Sh) smax = std::max(smax, std::fabs(v));
            int e = 0;
            if (smax > 0.f && std::isfinite(smax)) e = 13 - (int)std::floor(std::log2(smax));
            a.s_exp = std::max(-20, std::min(e, 20));
            // |PP_c RR_D| <= (max_j |a_j| + |d_j|)^2 of the pitch rows times the same of the roll rows: keep it below 2^14
            double bp = 0.0, br = 0.0;
            for (int j = 0; j < r_p; ++j) bp = std::max(bp, std::fabs(rows_p[4 * j]) + std::fabs(rows_p[4 * j + 3]));
            for (int j = 0; j < r_r; ++j) br = std::max(br, std::fabs(rows_r[4 * j]) + std::fabs(rows_r[4 * j + 3]));
            const double bound = std::max(bp * bp * br * br, 1e-30);
            a.pr_exp = std::max(-20, std::min(14 - (int)std::ceil(std::log2(bound)), 14));
        }
        build_tc_operands_kernel<<<32, 256>>>(pl->S, std::ldexp(1.0f, a.s_exp), pl->tc_ops);
        NLML_CUDA(cudaGetLastError());
        NLML_CUDA(cudaDeviceSynchronize());
        pl->launches += 1;
        a.tc_ops = pl->tc_ops;
        {
            const int num_kb = (F + ProjCfg::BK - 1) / ProjCfg::BK;
            NLML_CUDA(cudaMalloc(&pl->proj_tiles, (size_t)num_kb * ProjCfg::W_BYTES));
            build_proj_tiles_kernel<<<64, 256>>>(pl->W2, pl->R, F, num_kb, pl->proj_tiles);
            NLML_CUDA(cudaGetLastError());
            NLML_CUDA(cudaDeviceSynchronize());
            NLML_CUDA(cudaFuncSetAttribute(tucker_project_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ProjCfg::SMEM_BYTES));
            pl->launches += 1;
        }
        if (wps_smem_bytes(F) > 200 * 1024) pl->fast = false;
        else
            NLML_CUDA(cudaFuncSetAttribute(tucker_fit_wps_kernel<5, 3, 3, 3, kWpsWarps>,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wps_smem_bytes(F)));
    }
    {
        const size_t with_st = sizeof(float) * cta_layout(F, pl->R, pl->nBCD, pl->nA, pl->nBCDp, true).total;
        pl->st_in_smem = with_st <= 96 * 1024;
        pl->cta_smem = sizeof(float) * cta_layout(F, pl->R, pl->nBCD, pl->nA, pl->nBCDp, pl->st_in_smem).total;
        pl->cta_ok = pl->nBCD <= kMaxBCD && pl->cta_smem <= 220 * 1024;
        if (!pl->cta_ok && !pl->gen_ok)   // (PlanOwner frees the plan)
            return set_error(NLML_E_UNSUPPORTED, "core too large for the CTA kernel's shared-memory working set");
        if (pl->cta_ok)
            NLML_CUDA(cudaFuncSetAttribute(tucker_fit_cta_kernel<kCtaThreads>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)pl->cta_smem));
    }
    if (pl->gen_ok) {
        // power-of-two scale of the tile images (FP16 range): the largest |S| lands in [2^13, 2^14)
        {
            std::vector<float> Sh((size_t)pl->nBCD * pl->NAP);
            NLML_CUDA(cudaMemcpy(Sh.data(), pl->S, sizeof(float) * Sh.size(), cudaMemcpyDeviceToHost));
            float smax = 0.f;
            for (float v : Sh) smax = std::max(smax, std::fabs(v));
            int e = 0;
            if (smax > 0.f && std::isfinite(smax)) e = 13 - (int)std::floor(std::log2(smax));
            pl->gen.s_exp = std::max(-40, std::min(e, 40));
        }
        // tile images of S for the run-time-rank tensor-core kernel (FP16 hi/lo planes in the UMMA operand layout)
        const size_t bytes = (size_t)pl->gen.nblocks * ((size_t)pl->gen.tt_bytes + pl->gen.gt_bytes);
        NLML_CUDA(cudaMalloc(&pl->gen_tiles, bytes));
        const long long elems = (long long)pl->gen.nblocks * ((long long)pl->gen.NB * pl->gen.KA + (long long)pl->gen.NA16 * pl->gen.NB);
        const unsigned grid = (unsigned)std::min<long long>((elems + 255) / 256, (long long)pl->num_sms * 32);
        tgen::build_tiles_kernel<<<grid, 256>>>(pl->S, pl->NAP, pl->gen, pl->gen_tiles);
        NLML_CUDA(cudaGetLastError());
        NLML_CUDA(cudaDeviceSynchronize());
        pl->launches += 1;
        tgen::GenArgs ga{};
        ga.c = pl->gen;
        if (int rc = dispatch_gen(ga, 1, nullptr, true)) return rc;
    }
    owner.p = nullptr;
    *plan_out = pl;
    return 0;
}

extern "C" void nlml_tucker_plan_destroy(nlml_tucker_plan* pl) {
    if (!pl) return;
    DeviceGuard guard(pl->device);
    for (int i = 0; i < 2; ++i) {
        if (pl->streams[i]) cudaStreamDestroy(pl->streams[i]);
        cudaFree(pl->x_dev[i]);
        cudaFree(pl->p_dev[i]);
        if (pl->p_stage[i]) cudaFreeHost(pl->p_stage[i]);
    }
    cudaFree(pl->W2);
    cudaFree(pl->S);
    cudaFree(pl->St);
    cudaFree(pl->gen_tiles);
    cudaFree(pl->tc_ops);
    cudaFree(pl->proj_tiles);
    cudaFree(pl->q_pre);
    if (pl->q_pre_done) cudaEventDestroy(pl->q_pre_done);
    for (int i = 0; i < 3; ++i) cudaFree(pl->q_ws[i]);
    if (pl->q_done) cudaEventDestroy(pl->q_done);
    delete pl;
}

namespace {
// the raw-landmark entry points (ipd = 1) read landmarks 1, 33 and 263: columns 3..5, 99..101 and 789..791
int check_landmark_plan(const nlml_tucker_plan* pl, int ipd) {
    if (ipd && pl->F < 3 * 264)
        return set_error(NLML_E_INVALID, "IPD normalisation needs x,y,z triples up to landmark 263 (F=%d)", pl->F);
    return 0;
}

int fit_device(nlml_tucker_plan* pl, const float* X_dev, int64_t N, int64_t ldx, int ipd, int iters, float lr, float clip,
               float* P_out_dev, int64_t ldp, int kernel_hint, void* stream) {
    if (!pl || (N > 0 && (!X_dev || !P_out_dev))) return set_error(NLML_E_INVALID, "null pointer argument");
    if (N < 0 || ldx < pl->F || ldp < 3 + pl->ri || iters < 0)
        return set_error(NLML_E_INVALID, "bad sizes: N=%lld ldx=%lld (F=%d) ldp=%lld (need >= %d) iters=%d",
                         (long long)N, (long long)ldx, pl->F, (long long)ldp, 3 + pl->ri, iters);
    if (kernel_hint < 0 || kernel_hint > 6) return set_error(NLML_E_INVALID, "kernel_hint must be 0..6");
    if (int rc = check_landmark_plan(pl, ipd)) return rc;
    DeviceGuard guard(pl->device);
    return launch_fit(pl, X_dev, N, ldx, ipd, iters, lr, clip, P_out_dev, ldp, kernel_hint, (cudaStream_t)stream);
}

int fit_host(nlml_tucker_plan* pl, const float* X_host, int64_t N, int64_t ldx, int ipd, int iters, float lr, float clip,
             float* P_out_host, int64_t ldp) {
    if (!pl || (N > 0 && (!X_host || !P_out_host))) return set_error(NLML_E_INVALID, "null pointer argument");
    if (N < 0 || ldx < pl->F || ldp < 3 + pl->ri || iters < 0) return set_error(NLML_E_INVALID, "bad sizes");
    if (int rc = check_landmark_plan(pl, ipd)) return rc;
    DeviceGuard guard(pl->device);
    const int np = 3 + pl->ri;
    // every chunk runs the kernel the whole batch would get (the first chunks of the ramp are below the cross-over)
    const int hint = (pl->fast && N >= tc_crossover(pl)) ? 5 : 0;
    const int64_t proj_min = hint == 5 ? 1 : kProjMinRows;   // ... and the phase A the whole batch would get
    return host_pipeline(pl, X_host, N, ldx, P_out_host, ldp, [&](const float* x, int64_t n, float* p, cudaStream_t st, int slot) {
        return launch_fit(pl, x, n, pl->F, ipd, iters, lr, clip, p, np, hint, st, slot, proj_min);
    });
}

int solve_device(nlml_tucker_plan* pl, const float* X_dev, int64_t N, int64_t ldx, int ipd, int max_evals, float* P_out_dev,
                 int64_t ldp, int32_t* evals_out_dev, void* stream) {
    if (!pl || (N > 0 && (!X_dev || !P_out_dev))) return set_error(NLML_E_INVALID, "null pointer argument");
    if (N < 0 || ldx < pl->F || ldp < 3 + pl->ri || max_evals < 0 || max_evals == 1)
        return set_error(NLML_E_INVALID, "bad sizes: N=%lld ldx=%lld (F=%d) ldp=%lld (need >= %d) max_evals=%d (0 = default, else >= 2)",
                         (long long)N, (long long)ldx, pl->F, (long long)ldp, 3 + pl->ri, max_evals);
    if (int rc = check_landmark_plan(pl, ipd)) return rc;
    DeviceGuard guard(pl->device);
    return launch_solve(pl, X_dev, N, ldx, ipd, max_evals, P_out_dev, ldp, evals_out_dev, (cudaStream_t)stream);
}

int solve_host(nlml_tucker_plan* pl, const float* X_host, int64_t N, int64_t ldx, int ipd, int max_evals, float* P_out_host,
               int64_t ldp) {
    if (!pl || (N > 0 && (!X_host || !P_out_host))) return set_error(NLML_E_INVALID, "null pointer argument");
    if (N < 0 || ldx < pl->F || ldp < 3 + pl->ri || max_evals < 0 || max_evals == 1) return set_error(NLML_E_INVALID, "bad sizes");
    if (!pl->fast) return set_error(NLML_E_UNSUPPORTED, "the converged solve is built for ranks (5,3,3,3) only");
    if (int rc = check_landmark_plan(pl, ipd)) return rc;
    DeviceGuard guard(pl->device);
    const int np = 3 + pl->ri;
    // every chunk takes the phase A the whole batch would get (the last chunk of the ramp may be below the threshold)
    const int64_t proj_min = N >= kProjMinRows ? 1 : kProjMinRows;
    return host_pipeline(pl, X_host, N, ldx, P_out_host, ldp, [&](const float* x, int64_t n, float* p, cudaStream_t st, int) {
        return launch_solve(pl, x, n, pl->F, ipd, max_evals, p, np, nullptr, st, proj_min);
    });
}
}  // namespace

extern "C" int nlml_tucker_fit_f32(nlml_tucker_plan* pl, const float* X_dev, int64_t N, int64_t ldx, int iters,
                                   float lr, float clip, float* P_out_dev, int64_t ldp, int kernel_hint,
                                   void* stream) {
    return fit_device(pl, X_dev, N, ldx, 0, iters, lr, clip, P_out_dev, ldp, kernel_hint, stream);
}
extern "C" int nlml_tucker_fit_landmarks_f32(nlml_tucker_plan* pl, const float* LM_dev, int64_t N, int64_t ldx, int iters,
                                             float lr, float clip, float* P_out_dev, int64_t ldp, int kernel_hint,
                                             void* stream) {
    return fit_device(pl, LM_dev, N, ldx, 1, iters, lr, clip, P_out_dev, ldp, kernel_hint, stream);
}

extern "C" int nlml_tucker_fit_host_f32(nlml_tucker_plan* pl, const float* X_host, int64_t N, int64_t ldx,
                                        int iters, float lr, float clip, float* P_out_host, int64_t ldp) {
    return fit_host(pl, X_host, N, ldx, 0, iters, lr, clip, P_out_host, ldp);
}
extern "C" int nlml_tucker_fit_landmarks_host_f32(nlml_tucker_plan* pl, const float* LM_host, int64_t N, int64_t ldx,
                                                  int iters, float lr, float clip, float* P_out_host, int64_t ldp) {
    return fit_host(pl, LM_host, N, ldx, 1, iters, lr, clip, P_out_host, ldp);
}

extern "C" int nlml_tucker_solve_f32(nlml_tucker_plan* pl, const float* X_dev, int64_t N, int64_t ldx, int max_evals,
                                     float* P_out_dev, int64_t ldp, int32_t* evals_out_dev, void* stream) {
    return solve_device(pl, X_dev, N, ldx, 0, max_evals, P_out_dev, ldp, evals_out_dev, stream);
}
extern "C" int nlml_tucker_solve_landmarks_f32(nlml_tucker_plan* pl, const float* LM_dev, int64_t N, int64_t ldx, int max_evals,
                                               float* P_out_dev, int64_t ldp, int32_t* evals_out_dev, void* stream) {
    return solve_device(pl, LM_dev, N, ldx, 1, max_evals, P_out_dev, ldp, evals_out_dev, stream);
}

extern "C" int nlml_tucker_solve_host_f32(nlml_tucker_plan* pl, const float* X_host, int64_t N, int64_t ldx,
                                          int max_evals, float* P_out_host, int64_t ldp) {
    return solve_host(pl, X_host, N, ldx, 0, max_evals, P_out_host, ldp);
}
extern "C" int nlml_tucker_solve_landmarks_host_f32(nlml_tucker_plan* pl, const float* LM_host, int64_t N, int64_t ldx,
                                                    int max_evals, float* P_out_host, int64_t ldp) {
    return solve_host(pl, LM_host, N, ldx, 1, max_evals, P_out_host, ldp);
}

#ifdef NLML_GEN_TIMING
extern "C" int nlml_debug_gen_timing(float* host_out /*[64]*/) {   // development build only
    NLML_CUDA(cudaDeviceSynchronize());
    NLML_CUDA(cudaMemcpyFromSymbol(host_out, tgen::g_gen_timing, sizeof(float) * 64));
    return 0;
}
#endif


// numpy's pairwise-summation tree for n elements: leaves (offset, length) in order and the postfix combine program
static void pairwise_plan(int off, int n, std::vector<short>& loff, std::vector<short>& llen, std::vector<signed char>& prog) {
    if (n <= 128) {
        prog.push_back((signed char)loff.size());
        loff.push_back((short)off);
        llen.push_back((short)n);
        return;
    }
    int n2 = n / 2;
    n2 -= n2 % 8;
    pairwise_plan(off, n2, loff, llen, prog);
    pairwise_plan(off + n2, n - n2, loff, llen, prog);
    prog.push_back(-1);
}

static int powell_launch(nlml_tucker_plan* pl, const float* X_dev, int64_t N, int64_t ldx, int ipd, double* P_out_dev, int64_t ldp,
                         double* fun_out_dev, int32_t* nfev_out_dev, void* stream, const double* pts, int npts, double* vals);

extern "C" int nlml_tucker_powell_f64(nlml_tucker_plan* pl, const float* X_dev, int64_t N, int64_t ldx, double* P_out_dev,
                                      int64_t ldp, double* fun_out_dev, int32_t* nfev_out_dev, void* stream) {
    if (!pl || (N > 0 && (!X_dev || !P_out_dev))) return set_error(NLML_E_INVALID, "null pointer argument");
    return powell_launch(pl, X_dev, N, ldx, 0, P_out_dev, ldp, fun_out_dev, nfev_out_dev, stream, nullptr, 0, nullptr);
}
extern "C" int nlml_tucker_powell_landmarks_f64(nlml_tucker_plan* pl, const float* LM_dev, int64_t N, int64_t ldx, double* P_out_dev,
                                                int64_t ldp, double* fun_out_dev, int32_t* nfev_out_dev, void* stream) {
    if (!pl || (N > 0 && (!LM_dev || !P_out_dev))) return set_error(NLML_E_INVALID, "null pointer argument");
    return powell_launch(pl, LM_dev, N, ldx, 1, P_out_dev, ldp, fun_out_dev, nfev_out_dev, stream, nullptr, 0, nullptr);
}
/* test hook: q = W2 x of the tensor-core projection GEMM for N >= 4096 samples, CTA-blocked: Q_out_dev [ceil(N/128)][136][128] */
extern "C" int nlml_debug_gen_config(int r_id, int r_y, int r_p, int r_r, int32_t* out, int n_out) {
    constexpr int kFields = 23;
    if (!out || n_out < kFields) return set_error(NLML_E_INVALID, "out needs room for %d fields", kFields);
    if (r_id < 1 || r_y < 1 || r_p < 1 || r_r < 1) return set_error(NLML_E_INVALID, "ranks must be positive");
    tgen::GenCfg c{};
    if (const char* why = gen_config_for(r_id, r_y, r_p, r_r, c)) return set_error(NLML_E_UNSUPPORTED, "%s", why);
    const int32_t v[kFields] = {c.rrmax, c.nA, c.KA, c.NA16, c.nBC, c.nDp, c.BCP, c.NB, c.nblocks, c.resident, c.tslots,
                                c.gslots, c.ypr_tmem, c.tbufs, c.gbufs, c.ybufs, c.col_g, c.col_a, c.col_t, c.col_y,
                                c.smem_bytes, c.tt_bytes, c.gt_bytes};
    std::memcpy(out, v, sizeof(v));
    return 0;
}

extern "C" int nlml_debug_project_tc(nlml_tucker_plan* pl, const float* X_dev, int64_t N, int64_t ldx, float* Q_out_dev) {
    if (!pl || !X_dev || !Q_out_dev) return set_error(NLML_E_INVALID, "null pointer argument");
    DeviceGuard guard(pl->device);
    const float* q = nullptr;
    if (int rc = project_tc(pl, X_dev, N, ldx, 0, nullptr, &q)) return rc;
    if (!q) return set_error(NLML_E_UNSUPPORTED, "the tensor-core projection needs ranks (5,3,3,3), N >= 4096 and 16-byte aligned rows");
    NLML_CUDA(cudaEventRecord(pl->q_pre_done, nullptr));
    NLML_CUDA(cudaMemcpy(Q_out_dev, q, sizeof(float) * (size_t)ceil_div(N, 128) * 136 * 128, cudaMemcpyDeviceToDevice));
    return 0;
}
/* test hook: TD_Tester.objective (float64, the reference's operation order) of ONE sample x at npts parameter points */
extern "C" int nlml_debug_powell_objective(nlml_tucker_plan* pl, const float* x_dev, const double* pts_dev, int npts, double* vals_dev) {
    if (!pl || !x_dev || !pts_dev || !vals_dev || npts < 1) return set_error(NLML_E_INVALID, "null pointer argument");
    return powell_launch(pl, x_dev, 1, pl->F, 0, nullptr, 3 + pl->ri, nullptr, nullptr, nullptr, pts_dev, npts, vals_dev);
}
static int powell_launch(nlml_tucker_plan* pl, const float* X_dev, int64_t N, int64_t ldx, int ipd, double* P_out_dev, int64_t ldp,
                         double* fun_out_dev, int32_t* nfev_out_dev, void* stream, const double* pts, int npts, double* vals) {
    if (N < 0 || ldx < pl->F || ldp < 3 + pl->ri)
        return set_error(NLML_E_INVALID, "bad sizes: N=%lld ldx=%lld (F=%d) ldp=%lld (need >= %d)", (long long)N, (long long)ldx, pl->F,
                         (long long)ldp, 3 + pl->ri);
    if (int rc = check_landmark_plan(pl, ipd)) return rc;
    if (pl->F > kPowellThreads * kPowellMaxFeat || pl->F > 32000)
        return set_error(NLML_E_UNSUPPORTED, "the Powell fit serves F <= %d", kPowellThreads * kPowellMaxFeat);
    if (N == 0) return 0;
    DeviceGuard guard(pl->device);
    PowellArgs a{};
    a.X = X_dev; a.N = N; a.ldx = ldx; a.W2 = pl->W2; a.P = P_out_dev; a.ldp = ldp; a.fun = fun_out_dev; a.nfev = nfev_out_dev;
    a.ri = pl->ri; a.ry = pl->ry; a.rp = pl->rp; a.rr = pl->rr; a.F = pl->F; a.ipd = ipd;
    std::vector<short> loff, llen;
    std::vector<signed char> prog;
    pairwise_plan(0, pl->F, loff, llen, prog);
    if ((int)loff.size() > kPowellMaxLeaves) return set_error(NLML_E_UNSUPPORTED, "pairwise-sum tree too large");
    a.nleaf = (int)loff.size(); a.nprog = (int)prog.size();
    std::memcpy(a.leaf_off, loff.data(), sizeof(short) * loff.size());
    std::memcpy(a.leaf_len, llen.data(), sizeof(short) * llen.size());
    std::memcpy(a.prog, prog.data(), prog.size());
    std::memcpy(a.rows_y, pl->rows64[0], sizeof(a.rows_y));
    std::memcpy(a.rows_p, pl->rows64[1], sizeof(a.rows_p));
    std::memcpy(a.rows_r, pl->rows64[2], sizeof(a.rows_r));
    const size_t smem = sizeof(double) * ((size_t)pl->F + 9 * kPowellMaxLeaves + 2) + sizeof(float) * pl->F + 16;
    if (pts) {
        NLML_CUDA(cudaFuncSetAttribute(tucker_powell_objective_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tucker_powell_objective_kernel<<<1, kPowellThreads, smem, (cudaStream_t)stream>>>(a, pts, npts, vals);
        NLML_CUDA(cudaGetLastError());
        return 0;
    }
    NLML_CUDA(cudaFuncSetAttribute(tucker_powell_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    tucker_powell_kernel<<<(unsigned)N, kPowellThreads, smem, (cudaStream_t)stream>>>(a);
    NLML_CUDA(cudaGetLastError());
    pl->launches += 1;
    return 0;
}

extern "C" int nlml_cosine_fit_f64(const double* U_host, int n_rows, int n_cols, const double* w_deg_host, double* params_out_host,
                                   double* init_out_host, double* fun_out_host, int32_t* nfev_out_host, int device) {
    if (!U_host || !w_deg_host || !params_out_host) return set_error(NLML_E_INVALID, "null pointer argument");
    if (n_rows < 2 || n_cols < 1) return set_error(NLML_E_INVALID, "need at least 2 bins and 1 column");
    if (int rc = check_device(device)) return rc;
    DeviceGuard guard(device);
    std::vector<double> w(n_rows);
    for (int i = 0; i < n_rows; ++i) w[i] = w_deg_host[i] * (3.141592653589793238462643383279502884 / 180.0);   // np.radians
    struct Buf {
        void* p = nullptr;
        ~Buf() { cudaFree(p); }
    } dU, dw, dinit, dout, dfun, dnfev;
    NLML_CUDA(cudaMalloc(&dU.p, sizeof(double) * n_rows * n_cols));
    NLML_CUDA(cudaMalloc(&dw.p, sizeof(double) * n_rows));
    NLML_CUDA(cudaMalloc(&dinit.p, sizeof(double) * 4 * n_cols));
    NLML_CUDA(cudaMalloc(&dout.p, sizeof(double) * 4 * n_cols));
    NLML_CUDA(cudaMalloc(&dfun.p, sizeof(double) * n_cols));
    NLML_CUDA(cudaMalloc(&dnfev.p, sizeof(int) * n_cols));
    NLML_CUDA(cudaMemcpy(dU.p, U_host, sizeof(double) * n_rows * n_cols, cudaMemcpyHostToDevice));
    NLML_CUDA(cudaMemcpy(dw.p, w.data(), sizeof(double) * n_rows, cudaMemcpyHostToDevice));
    cosine_fit_kernel<<<(n_cols + 31) / 32, 32>>>((const double*)dU.p, n_rows, n_cols, (const double*)dw.p, (double*)dinit.p, (double*)dout.p,
                                                   (double*)dfun.p, (int*)dnfev.p);
    NLML_CUDA(cudaGetLastError());
    NLML_CUDA(cudaMemcpy(params_out_host, dout.p, sizeof(double) * 4 * n_cols, cudaMemcpyDeviceToHost));
    if (init_out_host) NLML_CUDA(cudaMemcpy(init_out_host, dinit.p, sizeof(double) * 4 * n_cols, cudaMemcpyDeviceToHost));
    if (fun_out_host) NLML_CUDA(cudaMemcpy(fun_out_host, dfun.p, sizeof(double) * n_cols, cudaMemcpyDeviceToHost));
    if (nfev_out_host) NLML_CUDA(cudaMemcpy(nfev_out_host, dnfev.p, sizeof(int) * n_cols, cudaMemcpyDeviceToHost));
    return 0;
}

// W = core x_5 U_feat (/root/reference/TD_main.py:231-238: tl.tensordot(core, U_feat^T, axes=(4, 0))): W2[r][f] = sum_m core2[r][m] U[f][m]
extern "C" int nlml_core_times_features_f32(const float* core_host, const float* U_feat_host, int64_t R, int M, int F, float* W_out_host,
                                            int device) {
    if (!core_host || !U_feat_host || !W_out_host) return set_error(NLML_E_INVALID, "null pointer argument");
    if (R < 1 || M < 1 || F < 1) return set_error(NLML_E_INVALID, "sizes must be positive");
    if (int rc = check_device(device)) return rc;
    DeviceGuard guard(device);
    struct Buf {
        void* p = nullptr;
        ~Buf() { cudaFree(p); }
    } dc, du, dq;
    const int64_t Rp = ceil_div(R, 128) * 128;
    NLML_CUDA(cudaMalloc(&dc.p, sizeof(float) * R * M));
    NLML_CUDA(cudaMalloc(&du.p, sizeof(float) * (size_t)F * M));
    NLML_CUDA(cudaMalloc(&dq.p, sizeof(float) * Rp * F));
    NLML_CUDA(cudaMemcpy(dc.p, core_host, sizeof(float) * R * M, cudaMemcpyHostToDevice));
    NLML_CUDA(cudaMemcpy(du.p, U_feat_host, sizeof(float) * (size_t)F * M, cudaMemcpyHostToDevice));
    // the projection kernel computes rows(core) . rows(U_feat) in its CTA-blocked layout [R/128][F][128]
    const int vec_ok = (M % 4 == 0);
    tgen::tucker_project_kernel<<<dim3((unsigned)(Rp / 128), (unsigned)ceil_div(F, 64)), 256>>>((const float*)dc.p, R, M, (const float*)du.p, F, M, vec_ok,
                                                                                               (float*)dq.p, 0);
    NLML_CUDA(cudaGetLastError());
    std::vector<float> blocked((size_t)Rp * F);
    NLML_CUDA(cudaMemcpy(blocked.data(), dq.p, sizeof(float) * Rp * F, cudaMemcpyDeviceToHost));
    for (int64_t r = 0; r < R; ++r)
        for (int f = 0; f < F; ++f) W_out_host[r * F + f] = blocked[((r / 128) * F + f) * 128 + r % 128];
    return 0;
}

extern "C" int64_t nlml_tucker_launch_count(const nlml_tucker_plan* pl) { return pl ? pl->launches : 0; }

// test hook: D[128][N] = A[128][K] * B[N][K]^T through the 3xTF32 tcgen05 building block of tucker_tc.cuh
extern "C" int nlml_debug_tf32_gemm(const float* A_dev, const float* B_dev, int K, int N, float* D_dev) {
    return nlml_debug_tf32_gemm_mode(A_dev, B_dev, K, N, D_dev, 0);
}
extern "C" int nlml_debug_tf32_gemm_mode(const float* A_dev, const float* B_dev, int K, int N, float* D_dev, int mode) {
    if (!A_dev || !B_dev || !D_dev || mode < 0 || mode > 3) return set_error(NLML_E_INVALID, "null pointer argument or bad mode");
    if (mode >= 2) {   // FP16 hi/lo building blocks (K multiple of 16, N <= 256)
        if (K < 16 || K % 16 || K > 64 || N < 16 || N % 16 || N > 256) return set_error(NLML_E_INVALID, "K must be 16..64 (multiple of 16), N 16..256 (multiple of 16)");
        const size_t smem16 = 2 * ttc::op16_bytes(128, K) + 2 * ttc::op16_bytes(N, K) + 64;
        NLML_CUDA(cudaFuncSetAttribute(ttc::tc16_check_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem16));
        ttc::tc16_check_kernel<<<1, 128, smem16>>>(A_dev, B_dev, D_dev, K, N, mode);
        NLML_CUDA(cudaGetLastError());
        NLML_CUDA(cudaDeviceSynchronize());
        return 0;
    }
    if (K < 8 || K % 8 || K > 64 || N < 16 || N % 16 || N > 256) return set_error(NLML_E_INVALID, "K must be 8..64 (multiple of 8), N 16..256 (multiple of 16)");
    ttc::TcCheckArgs a{A_dev, B_dev, D_dev, K, N, mode};
    const size_t smem = 2 * ttc::op_bytes(128, K) + 2 * ttc::op_bytes(N, K) + 64;
    NLML_CUDA(cudaFuncSetAttribute(ttc::tc_check_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ttc::tc_check_kernel<<<1, 128, smem>>>(a);
    NLML_CUDA(cudaGetLastError());
    NLML_CUDA(cudaDeviceSynchronize());
    return 0;
}

extern "C" int nlml_measure_tf32_tflops(int device, double* tflops_out) {
    if (!tflops_out) return set_error(NLML_E_INVALID, "null pointer argument");
    if (int rc = check_device(device)) return rc;
    DeviceGuard guard(device);
    cudaDeviceProp prop;
    NLML_CUDA(cudaGetDeviceProperties(&prop, device));
    const int blocks = prop.multiProcessorCount, iters = 2048;
    const size_t smem = ttc::op_bytes(128, 64) + ttc::op_bytes(256, 64) + 64;
    NLML_CUDA(cudaFuncSetAttribute(tf32_peak_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaEvent_t e0, e1;
    NLML_CUDA(cudaEventCreate(&e0));
    NLML_CUDA(cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 4; ++rep) {
        NLML_CUDA(cudaEventRecord(e0));
        tf32_peak_kernel<<<blocks, 128, smem>>>(iters);
        NLML_CUDA(cudaEventRecord(e1));
        NLML_CUDA(cudaEventSynchronize(e1));
        NLML_CUDA(cudaGetLastError());
        float ms = 0.f;
        NLML_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        const double flops = 2.0 * 128 * 256 * 8 * 8.0 * (double)iters * blocks;
        if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *tflops_out = best;
    return 0;
}

static int measure_ffma(int device, int three_reg, double* tflops_out);
extern "C" int nlml_measure_fp32_tflops(int device, double* tflops_out) { return measure_ffma(device, 0, tflops_out); }
extern "C" int nlml_measure_fp32_tflops_3reg(int device, double* tflops_out) { return measure_ffma(device, 1, tflops_out); }

static int measure_ffma(int device, int three_reg, double* tflops_out) {
    if (!tflops_out) return set_error(NLML_E_INVALID, "null pointer argument");
    if (int rc = check_device(device)) return rc;
    DeviceGuard guard(device);
    cudaDeviceProp prop;
    NLML_CUDA(cudaGetDeviceProperties(&prop, device));
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    float* out = nullptr;
    float* in = nullptr;
    NLML_CUDA(cudaMalloc(&out, sizeof(float) * blocks * threads));
    NLML_CUDA(cudaMalloc(&in, sizeof(float) * 256));
    {
        float h[256];
        for (int i = 0; i < 256; ++i) h[i] = 0.9990f + 1e-6f * i;
        NLML_CUDA(cudaMemcpy(in, h, sizeof(h), cudaMemcpyHostToDevice));
    }
    cudaEvent_t e0, e1;
    NLML_CUDA(cudaEventCreate(&e0));
    NLML_CUDA(cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        NLML_CUDA(cudaEventRecord(e0));
        if (three_reg) ffma_3reg_kernel<<<blocks, threads>>>(out, in, iters);
        else ffma_peak_kernel<<<blocks, threads>>>(out, iters);
        NLML_CUDA(cudaEventRecord(e1));
        NLML_CUDA(cudaEventSynchronize(e1));
        float ms = 0.f;
        NLML_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        const double flops = 2.0 * 8 * 16 * (double)iters * blocks * threads;
        if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(out);
    cudaFree(in);
    *tflops_out = best;
    return 0;
}
