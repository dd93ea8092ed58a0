// predict16.cuh - 16-warp variant of the fused fp64 posterior-predict + acquisition kernel.
//
// Same fusion, tile (128 candidates x 128 rows of L^-1), k-tile (32), 3-stage cp.async pipeline and
// fixed-order reductions as predict_acq_kernel<DMMA> (predict_kernels.cuh), but 512 threads per CTA:
//   * phase B: warp tile 32(m) x 32(n) -> 32 fp64 accumulators (64 registers) per thread instead of 128,
//     the kernel fits in 128 registers/thread, and every SM sub-partition holds FOUR resident warps whose
//     LDS -> DMMA dependencies interleave (the 8-warp kernel has two: ncu showed ~6 % issue gaps inside the
//     DMMA loop, stalled_wait 4.8 / math_pipe_throttle 3.2 per issue);
//   * phase A (K* build, DFMA + sqrt/exp latency chains) runs with 16 warps, four row-quarters per candidate
//     column, so its latency-bound part shrinks;
//   * L2 policy hints: L^-1 (67 MB triangle at N=4096, re-read by every CTA for every tile) is loaded
//     evict_last, the CTA-private K* scratch (written once, swept cyclically: LRU-hostile) evict_first, so the
//     0.6 GB scratch stream stops evicting the factor from the 126 MB L2.
// Selected with B200BO_PREDICT_WARPS=16 (A/B measurements decide the default, see DESIGN.md).
#pragma once
#include "predict_kernels.cuh"

namespace b200bo {

constexpr int P16_NT = 512;
constexpr int P16_SPLIT = P16_NT / PBN;  // row quarters of every staged chunk in phase A

__device__ __forceinline__ unsigned long long l2_policy_evict_last() {
    unsigned long long p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;\n" : "=l"(p));
    return p;
}
__device__ __forceinline__ unsigned long long l2_policy_evict_first() {
    unsigned long long p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;\n" : "=l"(p));
    return p;
}
__device__ __forceinline__ void cp_async16_cg_hint(void* smem_dst, const void* gmem_src, unsigned long long pol) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem_src), "l"(pol));
}
__device__ __forceinline__ void st_global_hint(double* p, double v, unsigned long long pol) {
    asm volatile("st.global.L2::cache_hint.f64 [%0], %1, %2;\n" ::"l"(p), "d"(v), "l"(pol) : "memory");
}

// Modes of predict_acq16_kernel.  FULL: the fused kernel.  SCREEN: phase A in full (mu needs every K* row) but K*
// stored for the first kScreenBlocks row blocks only, phase B over those blocks, a lower-bound key per candidate
// (select.cuh prune_lower_bound) and per-CTA lists of the k smallest bounds.  GATHER: FULL over the candidates of a
// gather buffer (coordinates as loaded + global index, count on the device).
enum { P16_FULL = 0, P16_SCREEN = 1, P16_GATHER = 2 };
constexpr int kScreenBlocks = 2;

// ---- phase A: K*^T tile (np x 128) into the CTA's scratch + K* alpha_ -----------------------------
template <bool DREG, int COV, int MODE>
__device__ __forceinline__ void predict16_phase_a_impl(const PredictParams& P, const GpDev& G, long long c0,
                                                       long long m, double* __restrict__ Ks, double* smem,
                                                       double (*mu_s)[PBN], unsigned long long pol_first) {
    const int tid = threadIdx.x;
    const int d = P.d, np = G.np;
    double* xc_s = smem;                              // [d][PBN]
    double* xs_s = smem + (size_t)d * PBN;            // [2][PA_CHUNK][d]
    double* al_s = xs_s + (size_t)2 * PA_CHUNK * d;   // [2][PA_CHUNK]
    for (int idx = tid; idx < PBN * d; idx += P16_NT) {
        const int c = idx / d, j = idx - c * d;
        const long long gi = c0 + c;
        double v = 0.0;
        if (gi < m) {
            v = MODE == P16_GATHER ? P.gather_x[gi * d + j] : candidate_coord(P, gi, j);
            if (G.xform && G.xform[j] == B200BO_XFORM_ROUND) v = rint(v);
            v = v / G.ls[j];
        }
        xc_s[j * PBN + c] = v;
    }
    const int chunk_pieces = PA_CHUNK * d / 2;
    auto load_chunk = [&](int buf, int ch) {
        const double* src = G.Xs + (size_t)ch * PA_CHUNK * d;
        double* dst = xs_s + (size_t)buf * PA_CHUNK * d;
        for (int q = tid; q < chunk_pieces; q += P16_NT) cp_async16_cg(dst + 2 * q, src + 2 * q);
        if (tid < PA_CHUNK / 2)
            cp_async16_cg(al_s + buf * PA_CHUNK + 2 * tid, G.alphav + (size_t)ch * PA_CHUNK + 2 * tid);
    };
    const int nch = np / PA_CHUNK;
    load_chunk(0, 0);
    cp_async_commit();
    __syncthreads();  // xc_s visible
    const int c = tid & (PBN - 1), part = tid >> 7;  // part in [0, P16_SPLIT)
    double xc[kPredictMaxDimRegs];
    if (DREG) {
#pragma unroll
        for (int j = 0; j < kPredictMaxDimRegs; ++j) xc[j] = (j < d) ? xc_s[j * PBN + c] : 0.0;
    }
    double mu_acc = 0.0;
    constexpr int R = 8;
    constexpr int ROWS = PA_CHUNK / P16_SPLIT;  // 16 rows of every chunk per thread
    for (int ch = 0; ch < nch; ++ch) {
        if (ch + 1 < nch) load_chunk((ch + 1) & 1, ch + 1);
        cp_async_commit();
        cp_async_wait<1>();
        __syncthreads();
        const double* xs = xs_s + (size_t)(ch & 1) * PA_CHUNK * d;
        const double* al = al_s + (ch & 1) * PA_CHUNK;
        for (int r0 = part * ROWS; r0 < (part + 1) * ROWS; r0 += R) {
            double r2[R];
#pragma unroll
            for (int q = 0; q < R; ++q) r2[q] = 0.0;
            if (DREG && (d & 1) == 0) {
#pragma unroll
                for (int j = 0; j < kPredictMaxDimRegs; j += 2) {
                    if (j < d) {
#pragma unroll
                        for (int q = 0; q < R; ++q) {
                            const double2 xv = *reinterpret_cast<const double2*>(xs + (r0 + q) * d + j);
                            const double d0 = xc[j] - xv.x, d1 = xc[j + 1] - xv.y;
                            r2[q] = fma(d0, d0, r2[q]);
                            r2[q] = fma(d1, d1, r2[q]);
                        }
                    }
                }
            } else if (DREG) {
#pragma unroll
                for (int j = 0; j < kPredictMaxDimRegs; ++j) {
                    if (j < d) {
#pragma unroll
                        for (int q = 0; q < R; ++q) {
                            const double df = xc[j] - xs[(r0 + q) * d + j];
                            r2[q] = fma(df, df, r2[q]);
                        }
                    }
                }
            } else {
                for (int j = 0; j < d; ++j) {
                    const double xv = xc_s[j * PBN + c];
#pragma unroll
                    for (int q = 0; q < R; ++q) {
                        const double df = xv - xs[(r0 + q) * d + j];
                        r2[q] = fma(df, df, r2[q]);
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < R; ++q) {
                const int n = ch * PA_CHUNK + r0 + q;
                double kv = G.constv * cov_eval<COV>(r2[q]);
                if (n >= G.n) kv = 0.0;
                if (MODE != P16_SCREEN || n < kScreenBlocks * PBM) st_global_hint(Ks + (size_t)n * PBN + c, kv, pol_first);
                mu_acc = fma(al[r0 + q], kv, mu_acc);
            }
        }
        __syncthreads();  // chunk buffer free for the prefetch of chunk ch+2
    }
    cp_async_wait<0>();
    mu_s[part][c] = mu_acc;
    __threadfence_block();
    __syncthreads();
}

template <bool DREG, int MODE>
__device__ __forceinline__ void predict16_phase_a(const PredictParams& P, const GpDev& G, long long c0, long long m,
                                                  double* __restrict__ Ks, double* smem, double (*mu_s)[PBN],
                                                  unsigned long long pol_first) {
    switch (cov_code(G.family, G.nu)) {
        case 0: predict16_phase_a_impl<DREG, 0, MODE>(P, G, c0, m, Ks, smem, mu_s, pol_first); break;
        case 1: predict16_phase_a_impl<DREG, 1, MODE>(P, G, c0, m, Ks, smem, mu_s, pol_first); break;
        case 2: predict16_phase_a_impl<DREG, 2, MODE>(P, G, c0, m, Ks, smem, mu_s, pol_first); break;
        default: predict16_phase_a_impl<DREG, 3, MODE>(P, G, c0, m, Ks, smem, mu_s, pol_first); break;
    }
}

// stage loader: BK k-rows x 128 doubles of LinvT (evict_last) and of K* (evict_first), 512 threads
__device__ __forceinline__ void predict16_load_stage(double* as, double* bs, const double* Ag, const double* Bg,
                                                     int np, unsigned long long pol_last,
                                                     unsigned long long pol_first) {
    constexpr int STR = PSTR_DMMA, BK = PBK_DMMA;
    const int tid = threadIdx.x;
#pragma unroll
    for (int t = 0; t < BK * 64 / P16_NT; ++t) {
        const int q = tid + t * P16_NT;
        const int kk = q >> 6, m2 = (q & 63) * 2;
        cp_async16_cg_hint(as + kk * STR + m2, Ag + (size_t)kk * np + m2, pol_last);
        cp_async16_cg_hint(bs + kk * STR + m2, Bg + kk * PBN + m2, pol_first);
    }
}

// ---- phase B: mma.sync m8n8k4 f64; 16 warps, warp tile 32(m) x 32(n); red[4][PBN] ----------------
// over the first nb row blocks of L^-1 (all np / PBM of them but in the screen)
__device__ __forceinline__ void predict16_phase_b(const GpDev& G, const double* __restrict__ Ks, double* smem, int nb,
                                                  unsigned long long pol_last, unsigned long long pol_first) {
    constexpr int STR = PSTR_DMMA, BK = PBK_DMMA;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // the four warps of an SM sub-partition (equal warp & 3) own the four different row slabs, so skipping the
    // structurally-zero k-tiles of the diagonal block leaves every sub-partition with the same amount of work
    const int wn = warp >> 2;
    const int wm = (warp + wn) & 3;
    const int g = lane >> 2, t4 = lane & 3;
    const int np = G.np;
    double* As = smem;
    double* Bs = smem + PSTAGES * BK * STR;
    double csq[4][2];
#pragma unroll
    for (int j = 0; j < 4; ++j) csq[j][0] = csq[j][1] = 0.0;
    for (int ib = 0; ib < nb; ++ib) {
        double acc[4][4][2];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
        const int nks = (ib + 1) * (PBM / BK);
        const double* Abase = G.linvT + (size_t)ib * PBM;
#pragma unroll
        for (int s = 0; s < PSTAGES - 1; ++s) {
            if (s < nks)
                predict16_load_stage(As + s * BK * STR, Bs + s * BK * STR, Abase + (size_t)(s * BK) * np,
                                     Ks + (size_t)(s * BK) * PBN, np, pol_last, pol_first);
            cp_async_commit();
        }
        for (int ks = 0; ks < nks; ++ks) {
            cp_async_wait<PSTAGES - 2>();
            __syncthreads();
            const int nxt = ks + PSTAGES - 1;
            const bool live = ks * BK < ib * PBM + (wm + 1) * 32;
            const double* as = As + (ks % PSTAGES) * BK * STR + wm * 32 + g;
            const double* bs = Bs + (ks % PSTAGES) * BK * STR + wn * 32 + g;
#pragma unroll
            for (int k4 = 0; k4 < BK / 4; ++k4) {
                if (k4 == 1) {
                    if (nxt < nks)
                        predict16_load_stage(As + (nxt % PSTAGES) * BK * STR, Bs + (nxt % PSTAGES) * BK * STR,
                                             Abase + (size_t)(nxt * BK) * np, Ks + (size_t)(nxt * BK) * PBN, np,
                                             pol_last, pol_first);
                    cp_async_commit();
                }
                if (live) {
                    double a[4], b[4];
                    const int krow = (k4 * 4 + t4) * STR;
#pragma unroll
                    for (int i = 0; i < 4; ++i) a[i] = as[krow + i * 8];
#pragma unroll
                    for (int j = 0; j < 4; ++j) b[j] = bs[krow + j * 8];
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int j = 0; j < 4; ++j) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
                }
            }
        }
        cp_async_wait<0>();
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            double s0 = 0.0, s1 = 0.0;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                s0 = fma(acc[i][j][0], acc[i][j][0], s0);
                s1 = fma(acc[i][j][1], acc[i][j][1], s1);
            }
            csq[j][0] += s0;
            csq[j][1] += s1;
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            double v = csq[j][e];
            v += __shfl_xor_sync(0xffffffffu, v, 4);
            v += __shfl_xor_sync(0xffffffffu, v, 8);
            v += __shfl_xor_sync(0xffffffffu, v, 16);
            csq[j][e] = v;
        }
    double* red = smem;  // [4][PBN]: row slab wm, every column produced by exactly one warp
    if (g == 0) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            red[wm * PBN + wn * 32 + j * 8 + t4 * 2] = csq[j][0];
            red[wm * PBN + wn * 32 + j * 8 + t4 * 2 + 1] = csq[j][1];
        }
    }
    __syncthreads();
}

template <bool DREG, int MODE>
__global__ void __launch_bounds__(P16_NT, 1) predict_acq16_kernel(const PredictParams P) {
    extern __shared__ __align__(16) double smem[];
    __shared__ double mu_s[P16_SPLIT][PBN];
    __shared__ double base_s[PBN];
    __shared__ double prod_s[PBN];
    __shared__ SelShared sel_s;

    const int tid = threadIdx.x;
    double* Ks = P.scratch + (long long)blockIdx.x * P.scratch_stride;
    const long long m = MODE == P16_GATHER ? (long long)*P.gather_count : P.m;
    const long long ntiles = (m + PBN - 1) / PBN;
    const unsigned long long pol_last = l2_policy_evict_last(), pol_first = l2_policy_evict_first();
    if (P.sel_cta) {
        if (tid < PBN) runsel_begin(sel_s, P.sel_cta + blockIdx.x, P.sel_resume, tid);
        __syncthreads();
    }
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long c0 = tile * PBN;
        for (int g = 0; g < P.n_gps; ++g) {
            const GpDev& G = P.gp[g];
            predict16_phase_a<DREG, MODE>(P, G, c0, m, Ks, smem, mu_s, pol_first);
            predict16_phase_b(G, Ks, smem, MODE == P16_SCREEN ? kScreenBlocks : G.np / PBM, pol_last, pol_first);
            const double* red = smem;
            if (tid < PBN) {
                const int c = tid;
                const bool valid = c0 + c < m;
                const double colsq = ((red[c] + red[PBN + c]) + red[2 * PBN + c]) + red[3 * PBN + c];
                const double mu_n = ((mu_s[0][c] + mu_s[1][c]) + mu_s[2][c]) + mu_s[3][c];
                if (MODE == P16_SCREEN) {  // the steps of candidate_epilogue up to sd, with the partial colsq
                    const double mean = G.y_std * mu_n + G.y_mean;
                    double var = G.prior - colsq;
                    if (var < 0.0) var = 0.0;  // not fmax: a NaN must stay NaN
                    const double lb = prune_lower_bound(P.acq_kind, mean, sqrt(var * (G.y_std * G.y_std)), P.y_max,
                                                        P.xi, P.kappa);
                    if (valid) P.screen_key[c0 + c] = prune_key(lb);
                    runsel_update<1>(sel_s, P.sel_k, tid, lb, c0 + c + P.index_base, valid);
                } else {
                    double val = 0.0;
                    candidate_epilogue(P, G, g, mu_n, colsq, c0 + c, base_s[c], prod_s[c], &val);
                    if (P.sel_cta && g == P.n_gps - 1) {
                        const long long gi = MODE == P16_GATHER ? (valid ? P.gather_idx[c0 + c] : SEL_NOIDX)
                                                                : c0 + c + P.index_base;
                        runsel_update<1>(sel_s, P.sel_k, tid, val, gi, valid);
                    }
                }
            }
            __syncthreads();
        }
    }
    if (P.sel_cta && tid < PBN) runsel_store(sel_s, P.sel_cta + blockIdx.x, tid);
}

// ---- pruned selection: gather buffers -------------------------------------------------------------
struct GatherBuf {
    double* x;                  // [cap][d] coordinates as phase A loads them (before transform and scaling)
    long long* idx;             // [cap] global selection index
    unsigned long long* count;  // appended so far
};

// append local candidate i of launch P (its device matrix or its Philox rows)
__device__ __forceinline__ void gather_append(const PredictParams& P, long long i, const GatherBuf& B) {
    const unsigned long long pos = atomicAdd(B.count, 1ull);
    B.idx[pos] = i + P.index_base;
    for (int j = 0; j < P.d; ++j) B.x[pos * P.d + j] = candidate_coord_raw(P, i, j);
}

// pilot: the candidates of the screen's per-CTA lists (k smallest lower bounds each); one block per list
__global__ void prune_pilot_kernel(const PredictParams P, const SelList* __restrict__ lists, int k, GatherBuf B) {
    const long long gi = threadIdx.x < k ? lists[blockIdx.x].idx[threadIdx.x] : SEL_NOIDX;
    if (gi != SEL_NOIDX) gather_append(P, gi - P.index_base, B);
}

// survivors: every candidate whose lower-bound key is <= tau (non-strict: ties with the k-th record and its
// lower-index rule must stay), and every candidate without a usable bound (key 0)
__global__ void prune_compact_kernel(const PredictParams P, const unsigned long long* __restrict__ tau, GatherBuf B) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < P.m && P.screen_key[i] <= *tau) gather_append(P, i, B);
}

}  // namespace b200bo
