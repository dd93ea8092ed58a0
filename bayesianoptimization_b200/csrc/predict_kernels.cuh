// predict_kernels.cuh - the fused posterior-predict + acquisition kernel (fp64) and the
// (value,index) selection kernel.
//
// Replaces, for a batch of M candidates, the whole chain
//   K* = kernel_(X*, X)            SK/gaussian_process/_gpr.py:446, kernels.py:1720-1729
//   mu = s_y * K* alpha_ + y_mean  :447-450
//   V  = L^-1 K*^T                 :460-462   (the N^2 M term)
//   var = diag - sum_i V_i^2, clamp, sd = sqrt(var * s_y^2)   :480-500
//   -base_acq(mu, sd) [* prod_j p_j]   R/bayes_opt/acquisition.py:199-217, :485/:660/:847,
//                                      R/bayes_opt/constraint.py:200-221
// in ONE launch.  V is formed as the triangular GEMM  V = Linv * K*^T  against the cached
// explicit inverse of the Cholesky factor (computed once at fit time), so the per-candidate
// work has no dependency chain.
//
// Decomposition: a persistent grid (one CTA per SM); each CTA owns tiles of BN = 128
// candidates.  Per tile and per GP:
//   phase A  build K*^T (np x 128) once into a CTA-private HBM/L2 scratch + accumulate K* alpha_
//   phase B  for each 128-row block of Linv: acc(128x128) = sum_{k<=rows} LinvT[k][rows]^T K*[k][:],
//            8x8 register tiles, 3-stage cp.async pipeline; then colsq += sum_rows acc^2
//   phase C  mu, sd, acquisition / constraint probability per candidate
// All reductions are fixed-order (no floating-point atomics): results are bit-reproducible and
// independent of the grid size.
#pragma once
#include "common.cuh"
#include "select.cuh"
#include "tc_common.cuh"

namespace b200bo {

struct GpDev {
    const double* Xs;      // [np][d]   transform(X)/length_scale, zero padded
    const double* linvT;   // [np][np]  (L^-1)^T row-major: linvT[k][i] = Linv[i][k]
    const double* alphav;  // [np]      alpha_, zero padded
    const double* ls;      // [d]       length scales (replicated when isotropic)
    const int* xform;      // [d] or nullptr
    const uint8_t* linv_tc;  // fp32 mode: L^-1 as tf32 (hi,lo) UMMA operand images, or nullptr
    int n, np, family, nu;
    double constv, y_mean, y_std, lb, ub;
    double prior;  // prior variance kernel_.diag(x*) = constv + WhiteKernel noise_level
};

struct PredictParams {
    GpDev gp[B200BO_MAX_GPS];
    int n_gps, d, acq_kind, pad0;
    double kappa, xi, y_max;
    const double* Xc;  // [m][d], or nullptr: candidates generated in-kernel (Philox, select.cuh)
    const double* pbounds;  // Philox mode: [2][d] = lo_j, (hi_j - lo_j)
    unsigned long long seed;  // Philox key
    long long index_base;  // global index of this launch's candidate 0 (Philox row / selection index)
    SelList* sel_cta;  // [gridDim.x] per-CTA running selection, or nullptr (no fused selection)
    int sel_k, sel_resume;  // resume: continue the lists of the previous launch (chunked batches)
    long long m;
    double* acq_out;   // [m] or nullptr
    double* mu_out;    // [m] or nullptr (target GP)
    double* sd_out;    // [m] or nullptr (target GP)
    double* scratch;   // gridDim.x * scratch_stride doubles
    long long scratch_stride;
    unsigned long long* clamp_count;  // nullable; [0] negative variances clamped to 0, [1] non-finite candidate coordinates
    // pruned selection (predict16.cuh): screen output / gather-mode source
    unsigned long long* screen_key;  // screen: [m] lower-bound selection key per candidate, 0 = must be evaluated
    const double* gather_x;          // gather: [count][d] candidate coordinates as loaded
    const long long* gather_idx;     // gather: [count] global selection index
    const unsigned long long* gather_count;
};

// coordinate j of candidate gi (local index) as the reference's x_tries[gi, j]
// A non-finite coordinate is counted in clamp_count[1]: the host entry points turn it into the ValueError
// ("Input X contains NaN or infinity") sklearn's validate_data raises - checked where the data is read anyway instead
// of a separate pass over the batch on the host (10 ms per 2^20 x 16 batch).
__device__ __forceinline__ double candidate_coord_raw(const PredictParams& P, long long gi, int j) {
    if (P.Xc) return P.Xc[gi * P.d + j];
    return philox_coord(P.seed, gi + P.index_base, j, P.pbounds[j], P.pbounds[P.d + j]);
}
__device__ __forceinline__ double candidate_coord(const PredictParams& P, long long gi, int j) {
    const double v = candidate_coord_raw(P, gi, j);
    if (P.Xc && !isfinite(v) && P.clamp_count) atomicAdd(P.clamp_count + 1, 1ull);
    return v;
}

constexpr int PBM = 128, PBN = 128, PBK = 16, PSTAGES = 3, PNT = 256;
// smem row stride (doubles) of the A/B k-tiles.  DFMA variant: dense rows (conflict-free 16-byte
// fragment loads).  DMMA variant: +4 doubles: an LDS.64 is served per half-warp (4 k-rows x 4
// columns of an m8n8k4 fragment); a row stride of 264 words = 8 (mod 32) puts the four k-rows of
// each half-warp on disjoint bank octets -> 2 wavefronts per request, the minimum for 256 bytes.
constexpr int PSTR_DFMA = 128, PSTR_DMMA = 132;
// phase A needs (128 + 2*64) * d doubles (d <= 64 -> 128 KiB); phase B (DFMA) 96 KiB
constexpr int kPredictSmemBytesDfma = 133120;  // + 1 KiB staged alpha_
constexpr int PBK_DMMA = 32;  // k-tile of the DMMA variant (one CTA barrier per 32 k)
constexpr int kPredictSmemBytesDmma = PSTAGES * PBK_DMMA * 2 * PSTR_DMMA * 8;  // 202752
constexpr int kPredictMaxDimRegs = 16;  // candidates held in registers when d <= 16

enum { PREDICT_IMPL_DFMA = 0, PREDICT_IMPL_DMMA = 1, PREDICT_IMPL_TF32 = 2 };

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// ---- per-candidate epilogue shared by the tiled and the small-batch kernels ---------------------
// mu_n: K* alpha_ (normalised units); colsq: sum_i V_i^2.  g = 0: target GP -> base acquisition;
// g >= 1: constraint GP -> probability factor.  The last GP writes -base * prod.
__device__ __forceinline__ void candidate_epilogue(const PredictParams& P, const GpDev& G, int g,
                                                   double mu_n, double colsq, long long gi,
                                                   double& base_neg, double& prod, double* final_val = nullptr) {
    const double mean = G.y_std * mu_n + G.y_mean;
    double var = G.prior - colsq;
    if (var < 0.0) {
        var = 0.0;
        if (P.clamp_count && gi < P.m) atomicAdd(P.clamp_count, 1ull);
    }
    const double sd = sqrt(var * (G.y_std * G.y_std));
    if (g == 0) {
        double base = 0.0;
        if (P.acq_kind == B200BO_ACQ_UCB) {
            base = mean + P.kappa * sd;
        } else if (P.acq_kind == B200BO_ACQ_EI) {
            const double a = mean - P.y_max - P.xi;
            const double z = a / sd;
            base = a * ndtr(z) + sd * norm_pdf(z);
        } else if (P.acq_kind == B200BO_ACQ_POI) {
            const double z = (mean - P.y_max - P.xi) / sd;
            base = ndtr(z);
        }
        base_neg = -1.0 * base;
        prod = 1.0;
        if (gi < P.m) {
            if (P.mu_out) P.mu_out[gi] = mean;
            if (P.sd_out) P.sd_out[gi] = sd;
        }
    } else {
        const double p_lo = (G.lb == -CUDART_INF) ? 0.0 : norm_cdf_loc_scale(G.lb, mean, sd);
        const double p_hi = (G.ub == CUDART_INF) ? 1.0 : norm_cdf_loc_scale(G.ub, mean, sd);
        // constraint.py:208 (J=1: result = p_hi - p_lo) / :219 (result *= ...)
        prod = (g == 1) ? (p_hi - p_lo) : prod * (p_hi - p_lo);
    }
    if (g == P.n_gps - 1) {
        const double val = (P.n_gps > 1) ? base_neg * prod : base_neg;
        if (final_val) *final_val = val;
        if (P.acq_out && gi < P.m) P.acq_out[gi] = val;
    }
}

// ---- phase A: K*^T tile (np x 128) into the CTA's scratch + K* alpha_ ---------------------------
// Thread = one candidate column (two threads per column split the rows).  Training rows stream
// through shared memory in chunks of 64 (double-buffered cp.async), so every row read is a
// warp-wide broadcast LDS; DREG keeps the candidate's coordinates in registers (d <= 16).
// COV is a template parameter so that the covariance is branch-free straight-line code.
constexpr int PA_CHUNK = 64;  // training rows per staged chunk

// TC = false: K* written as fp64 [np][128] (operand of the fp64 GEMM variants).
// TC = true : K* written as tf32 (hi, lo) pairs in the UMMA operand-image layout of tc_common.cuh
//             ([np/32][hi|lo][16 KiB], candidate = operand row, training index = K).
template <bool DREG, int COV, bool TC>
__device__ __forceinline__ void predict_phase_a_impl(const PredictParams& P, const GpDev& G, long long c0,
                                                     double* __restrict__ Ks, double* smem,
                                                     double (*mu_s)[PBN]) {
    const int tid = threadIdx.x;
    const int d = P.d, np = G.np;
    double* xc_s = smem;                       // [d][PBN]
    double* xs_s = smem + (size_t)d * PBN;     // [2][PA_CHUNK][d]
    double* al_s = xs_s + (size_t)2 * PA_CHUNK * d;  // [2][PA_CHUNK] alpha_ of the staged rows
    for (int idx = tid; idx < PBN * d; idx += PNT) {
        const int c = idx / d, j = idx - c * d;
        const long long gi = c0 + c;
        double v = 0.0;
        if (gi < P.m) {
            v = candidate_coord(P, gi, j);
            if (G.xform && G.xform[j] == B200BO_XFORM_ROUND) v = rint(v);
            v = v / G.ls[j];
        }
        xc_s[j * PBN + c] = v;
    }
    const int chunk_pieces = PA_CHUNK * d / 2;  // 16-byte pieces per chunk (PA_CHUNK*d is even)
    auto load_chunk = [&](int buf, int ch) {
        const double* src = G.Xs + (size_t)ch * PA_CHUNK * d;
        double* dst = xs_s + (size_t)buf * PA_CHUNK * d;
        for (int q = tid; q < chunk_pieces; q += PNT) cp_async16_cg(dst + 2 * q, src + 2 * q);
        if (tid < PA_CHUNK / 2)
            cp_async16_cg(al_s + buf * PA_CHUNK + 2 * tid, G.alphav + (size_t)ch * PA_CHUNK + 2 * tid);
    };
    const int nch = np / PA_CHUNK;
    load_chunk(0, 0);
    cp_async_commit();
    __syncthreads();  // xc_s visible
    const int c = tid & (PBN - 1), half = tid >> 7;
    double xc[kPredictMaxDimRegs];
    if (DREG) {
#pragma unroll
        for (int j = 0; j < kPredictMaxDimRegs; ++j) xc[j] = (j < d) ? xc_s[j * PBN + c] : 0.0;
    }
    double mu_acc = 0.0;
    constexpr int R = 8;
    for (int ch = 0; ch < nch; ++ch) {
        if (ch + 1 < nch) load_chunk((ch + 1) & 1, ch + 1);
        cp_async_commit();
        cp_async_wait<1>();
        __syncthreads();
        const double* xs = xs_s + (size_t)(ch & 1) * PA_CHUNK * d;
        const double* al = al_s + (ch & 1) * PA_CHUNK;
        for (int r0 = half * (PA_CHUNK / 2); r0 < (half + 1) * (PA_CHUNK / 2); r0 += R) {
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
            float hi[R], lo[R];
#pragma unroll
            for (int q = 0; q < R; ++q) {
                const int n = ch * PA_CHUNK + r0 + q;
                double kv = G.constv * cov_eval<COV>(r2[q]);
                if (n >= G.n) kv = 0.0;
                if (TC) {
                    hi[q] = tc::to_tf32((float)kv);
                    lo[q] = tc::to_tf32((float)(kv - (double)hi[q]));
                } else {
                    Ks[(size_t)n * PBN + c] = kv;
                }
                mu_acc = fma(al[r0 + q], kv, mu_acc);
            }
            if (TC) {
                const int n0 = ch * PA_CHUNK + r0;  // multiple of 8: two groups of 4 consecutive k
                uint8_t* img = reinterpret_cast<uint8_t*>(Ks) + (size_t)(n0 >> 5) * (2 * tc::kTcImgBytes);
#pragma unroll
                for (int h4 = 0; h4 < 2; ++h4) {
                    const int off = tc::tc_img_offset(c, (n0 & 31) + 4 * h4);
                    *reinterpret_cast<float4*>(img + off) =
                        make_float4(hi[4 * h4], hi[4 * h4 + 1], hi[4 * h4 + 2], hi[4 * h4 + 3]);
                    *reinterpret_cast<float4*>(img + tc::kTcImgBytes + off) =
                        make_float4(lo[4 * h4], lo[4 * h4 + 1], lo[4 * h4 + 2], lo[4 * h4 + 3]);
                }
            }
        }
        __syncthreads();  // chunk buffer free for the prefetch of chunk ch+2
    }
    cp_async_wait<0>();
    mu_s[half][c] = mu_acc;
    if (TC) {
        tc::fence_proxy_async_global();  // scratch images will be read by bulk async copies
        tc::fence_proxy_async_smem();    // and the stage buffers overwritten by them
    }
    __threadfence_block();
    __syncthreads();
}

template <bool DREG, bool TC = false>
__device__ __forceinline__ void predict_phase_a(const PredictParams& P, const GpDev& G, long long c0,
                                                double* __restrict__ Ks, double* smem,
                                                double (*mu_s)[PBN]) {
    switch (cov_code(G.family, G.nu)) {
        case 0: predict_phase_a_impl<DREG, 0, TC>(P, G, c0, Ks, smem, mu_s); break;
        case 1: predict_phase_a_impl<DREG, 1, TC>(P, G, c0, Ks, smem, mu_s); break;
        case 2: predict_phase_a_impl<DREG, 2, TC>(P, G, c0, Ks, smem, mu_s); break;
        default: predict_phase_a_impl<DREG, 3, TC>(P, G, c0, Ks, smem, mu_s); break;
    }
}

// stage loader shared by both GEMM variants: BK k-rows x 128 doubles of LinvT and of K*
template <int STR, int BK>
__device__ __forceinline__ void predict_load_stage(double* as, double* bs, const double* Ag,
                                                   const double* Bg, int np) {
    const int tid = threadIdx.x;
#pragma unroll
    for (int t = 0; t < BK / 4; ++t) {
        const int q = tid + t * PNT;
        const int kk = q >> 6, m2 = (q & 63) * 2;
        cp_async16_cg(as + kk * STR + m2, Ag + (size_t)kk * np + m2);
        cp_async16_cg(bs + kk * STR + m2, Bg + kk * PBN + m2);
    }
}

// ---- phase B (DFMA): 8x8 register tiles; returns per-column sums of V^2 in red[16][PBN] -------
__device__ __forceinline__ void predict_phase_b_dfma(const GpDev& G, const double* __restrict__ Ks,
                                                     double* smem) {
    constexpr int STR = PSTR_DFMA, BK = PBK;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int np = G.np;
    double* As = smem;
    double* Bs = smem + PSTAGES * BK * STR;
    double csq[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) csq[j] = 0.0;
    const int nb = np / PBM;
    for (int ib = 0; ib < nb; ++ib) {
        double acc[8][8];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[i][j] = 0.0;
        const int nks = (ib + 1) * (PBM / BK);
        const double* Abase = G.linvT + (size_t)ib * PBM;
#pragma unroll
        for (int s = 0; s < PSTAGES - 1; ++s) {
            if (s < nks)
                predict_load_stage<STR, BK>(As + s * BK * STR, Bs + s * BK * STR,
                                            Abase + (size_t)(s * BK) * np, Ks + (size_t)(s * BK) * PBN, np);
            cp_async_commit();
        }
        for (int ks = 0; ks < nks; ++ks) {
            cp_async_wait<PSTAGES - 2>();
            __syncthreads();
            const int nxt = ks + PSTAGES - 1;
            if (nxt < nks)
                predict_load_stage<STR, BK>(As + (nxt % PSTAGES) * BK * STR, Bs + (nxt % PSTAGES) * BK * STR,
                                            Abase + (size_t)(nxt * BK) * np, Ks + (size_t)(nxt * BK) * PBN, np);
            cp_async_commit();
            const double* as = As + (ks % PSTAGES) * BK * STR;
            const double* bs = Bs + (ks % PSTAGES) * BK * STR;
#pragma unroll
            for (int kk = 0; kk < PBK; ++kk) {
                double a[8], b[8];
#pragma unroll
                for (int p = 0; p < 4; ++p) {
                    const double2 t = *reinterpret_cast<const double2*>(as + kk * STR + p * 32 + ty * 2);
                    a[2 * p] = t.x;
                    a[2 * p + 1] = t.y;
                }
#pragma unroll
                for (int p = 0; p < 4; ++p) {
                    const double2 t = *reinterpret_cast<const double2*>(bs + kk * STR + p * 32 + tx * 2);
                    b[2 * p] = t.x;
                    b[2 * p + 1] = t.y;
                }
#pragma unroll
                for (int i = 0; i < 8; ++i)
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
            }
        }
        cp_async_wait<0>();
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            double s = 0.0;
#pragma unroll
            for (int i = 0; i < 8; ++i) s = fma(acc[i][j], acc[i][j], s);
            csq[j] += s;
        }
    }
    double* red = smem;  // [16][PBN]
#pragma unroll
    for (int p = 0; p < 4; ++p) {
        red[ty * PBN + p * 32 + tx * 2] = csq[2 * p];
        red[ty * PBN + p * 32 + tx * 2 + 1] = csq[2 * p + 1];
    }
    __syncthreads();
}

// ---- phase B (DMMA): mma.sync m8n8k4 f64; warp tile 32(m) x 64(n); red[4][PBN] -----------------
__device__ __forceinline__ void predict_phase_b_dmma(const GpDev& G, const double* __restrict__ Ks,
                                                     double* smem) {
    constexpr int STR = PSTR_DMMA, BK = PBK_DMMA;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // warps w and w+4 share an SM sub-partition: give them row slabs s and 3-s so that skipping
    // the structurally-zero part of the diagonal block (k beyond the slab's last row) leaves every
    // sub-partition with the same amount of work
    const int wn = warp >> 2;
    const int wm = wn ? 3 - (warp & 3) : (warp & 3);
    const int g = lane >> 2, t4 = lane & 3;
    const int np = G.np;
    double* As = smem;
    double* Bs = smem + PSTAGES * BK * STR;
    double csq[8][2];
#pragma unroll
    for (int j = 0; j < 8; ++j) csq[j][0] = csq[j][1] = 0.0;
    const int nb = np / PBM;
    for (int ib = 0; ib < nb; ++ib) {
        double acc[4][8][2];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
        const int nks = (ib + 1) * (PBM / BK);
        const double* Abase = G.linvT + (size_t)ib * PBM;
#pragma unroll
        for (int s = 0; s < PSTAGES - 1; ++s) {
            if (s < nks)
                predict_load_stage<STR, BK>(As + s * BK * STR, Bs + s * BK * STR,
                                            Abase + (size_t)(s * BK) * np, Ks + (size_t)(s * BK) * PBN, np);
            cp_async_commit();
        }
        for (int ks = 0; ks < nks; ++ks) {
            cp_async_wait<PSTAGES - 2>();
            __syncthreads();
            const int nxt = ks + PSTAGES - 1;
            // diagonal block of L^-1 (k in [ib*128, ib*128+128)): rows wm*32.. have zeros for
            // k > row, so the k-tiles beyond this warp's slab contribute nothing
            const bool live = ks * BK < ib * PBM + (wm + 1) * 32;
            const double* as = As + (ks % PSTAGES) * BK * STR + wm * 32 + g;
            const double* bs = Bs + (ks % PSTAGES) * BK * STR + wn * 64 + g;
#pragma unroll
            for (int k4 = 0; k4 < BK / 4; ++k4) {
                if (k4 == 1) {
                    // prefetch issued behind the first batch of MMAs so the tensor pipe is already
                    // busy while the LDGSTS addresses are generated
                    if (nxt < nks)
                        predict_load_stage<STR, BK>(As + (nxt % PSTAGES) * BK * STR, Bs + (nxt % PSTAGES) * BK * STR,
                                                    Abase + (size_t)(nxt * BK) * np, Ks + (size_t)(nxt * BK) * PBN, np);
                    cp_async_commit();
                }
                if (live) {
                    double a[4], b[8];
                    const int krow = (k4 * 4 + t4) * STR;
#pragma unroll
                    for (int i = 0; i < 4; ++i) a[i] = as[krow + i * 8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) b[j] = bs[krow + j * 8];
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int j = 0; j < 8; ++j) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
                }
            }
        }
        cp_async_wait<0>();
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 8; ++j) {
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
    // rows of one m8 fragment live in lanes with equal (lane & 3): butterfly over lane bits 2..4
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            double v = csq[j][e];
            v += __shfl_xor_sync(0xffffffffu, v, 4);
            v += __shfl_xor_sync(0xffffffffu, v, 8);
            v += __shfl_xor_sync(0xffffffffu, v, 16);
            csq[j][e] = v;
        }
    double* red = smem;  // [4][PBN]
    if (g == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            red[wm * PBN + wn * 64 + j * 8 + t4 * 2] = csq[j][0];
            red[wm * PBN + wn * 64 + j * 8 + t4 * 2 + 1] = csq[j][1];
        }
    }
    __syncthreads();
}

template <int IMPL, bool DREG>
__global__ void __launch_bounds__(PNT, 1) predict_acq_kernel(const PredictParams P) {
    extern __shared__ __align__(16) double smem[];
    __shared__ double mu_s[2][PBN];
    __shared__ double base_s[PBN];
    __shared__ double prod_s[PBN];
    __shared__ SelShared sel_s;

    const int tid = threadIdx.x;
    double* Ks = P.scratch + (long long)blockIdx.x * P.scratch_stride;
    const long long ntiles = (P.m + PBN - 1) / PBN;
    constexpr int NRED = (IMPL == PREDICT_IMPL_DMMA) ? 4 : 16;
    if (P.sel_cta) {
        if (tid < PBN) runsel_begin(sel_s, P.sel_cta + blockIdx.x, P.sel_resume, tid);
        __syncthreads();
    }

    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long c0 = tile * PBN;
        for (int g = 0; g < P.n_gps; ++g) {
            const GpDev& G = P.gp[g];
            predict_phase_a<DREG>(P, G, c0, Ks, smem, mu_s);
            if (IMPL == PREDICT_IMPL_DMMA)
                predict_phase_b_dmma(G, Ks, smem);
            else
                predict_phase_b_dfma(G, Ks, smem);
            const double* red = smem;

            // ---------------- phase C: per-candidate epilogue --------------------------------
            if (tid < PBN) {
                const int c = tid;
                double colsq = 0.0;
#pragma unroll
                for (int r = 0; r < NRED; ++r) colsq += red[r * PBN + c];
                double val = 0.0;
                candidate_epilogue(P, G, g, mu_s[0][c] + mu_s[1][c], colsq, c0 + c, base_s[c], prod_s[c], &val);
                if (P.sel_cta && g == P.n_gps - 1)
                    runsel_update<1>(sel_s, P.sel_k, tid, val, c0 + c + P.index_base, c0 + c < P.m);
            }
            __syncthreads();
        }
    }
    if (P.sel_cta && tid < PBN) runsel_store(sel_s, P.sel_cta + blockIdx.x, tid);
}

// =======================================================================================
// fp32 mode: the same fused kernel with the N^2 term on the 5th-generation tensor cores.
//   V = L^-1 K*^T as 3xTF32 (a_hi*b_hi + a_hi*b_lo + a_lo*b_hi), fp32 accumulators in TMEM.
//   K* itself, K* alpha_ (the mean) and the whole epilogue stay fp64: only the triangular product
//   and the sum of squares run at reduced precision (north_star tolerance for this mode: 1e-3).
// Warp roles during the GEMM phase (one CTA per SM, 256 threads, TMEM 2 x 128 columns):
//   warp 0 / lane 0  producer: 1-D bulk async copies (TMA engine) of pre-tiled operand images
//                    [A_hi|A_lo] (L^-1, tiled once at fit time) and [B_hi|B_lo] (written by phase A)
//   warp 1 / lane 0  tcgen05.mma issuer: 4 k-steps x 3 products per 32-k stage, tcgen05.commit
//                    releases the stage / publishes the accumulator
//   warps 4..7       epilogue: tcgen05.ld of their TMEM quadrant, per-thread sum of squares
// The operand images use the SWIZZLE_NONE K-major core-matrix layout, so a stage is a verbatim
// 64 KiB byte copy - no tensor map, no swizzle bookkeeping.
// =======================================================================================
constexpr int TC_STAGES = 3;
constexpr int TC_STAGE_BYTES = 4 * tc::kTcImgBytes;                // A_hi, A_lo, B_hi, B_lo
constexpr int kPredictSmemBytesTc = TC_STAGES * TC_STAGE_BYTES;    // 196608
constexpr int TC_TMEM_COLS = 256;                                  // two 128-column accumulators

template <bool DREG>
__global__ void __launch_bounds__(PNT, 1) predict_acq_tc_kernel(const PredictParams P) {
    extern __shared__ __align__(16) double smem[];
    __shared__ double mu_s[2][PBN];
    __shared__ double base_s[PBN];
    __shared__ double prod_s[PBN];
    __shared__ double red_s[4][PBN];
    __shared__ uint64_t full_bar[TC_STAGES], empty_bar[TC_STAGES], accfull_bar[2], accempty_bar[2];
    __shared__ uint32_t tmem_base_s;
    __shared__ SelShared sel_s;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint8_t* stage_mem = reinterpret_cast<uint8_t*>(smem);
    double* Ks = P.scratch + (long long)blockIdx.x * P.scratch_stride;  // holds the B images (bytes)
    const long long ntiles = (P.m + PBN - 1) / PBN;
    if (P.sel_cta) {
        if (tid < PBN) runsel_begin(sel_s, P.sel_cta + blockIdx.x, P.sel_resume, tid);
        __syncthreads();
    }

    if (tid == 0) {
        for (int s = 0; s < TC_STAGES; ++s) {
            tc::mbar_init(&full_bar[s], 1);
            tc::mbar_init(&empty_bar[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            tc::mbar_init(&accfull_bar[b], 1);
            tc::mbar_init(&accempty_bar[b], 4);
        }
        tc::mbar_fence_init();
    }
    if (warp == 1) tc::tmem_alloc(&tmem_base_s, TC_TMEM_COLS);
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();
    const uint32_t tmem_base = tmem_base_s;
    const uint32_t idesc = tc::umma_idesc_tf32(128, 128);

    uint32_t stage_it = 0;  // stages filled / consumed so far (producer and MMA thread count alike)
    uint32_t acc_it = 0;    // accumulator buffers produced / drained so far

    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long c0 = tile * PBN;
        for (int g = 0; g < P.n_gps; ++g) {
            const GpDev& G = P.gp[g];
            predict_phase_a<DREG, true>(P, G, c0, Ks, smem, mu_s);
            const int nb = G.np / PBM;
            const int nkt_row = G.np / tc::kTcK;  // images per row block in the A array
            const uint8_t* Bimg = reinterpret_cast<const uint8_t*>(Ks);

            if (warp == 0) {
                if (lane == 0) {
                    uint32_t it = stage_it;
                    for (int ib = 0; ib < nb; ++ib) {
                        const int nkt = (ib + 1) * (PBM / tc::kTcK);
                        const uint8_t* Aimg = G.linv_tc + (size_t)ib * nkt_row * (2 * tc::kTcImgBytes);
                        for (int kt = 0; kt < nkt; ++kt, ++it) {
                            const int s = it % TC_STAGES;
                            tc::mbar_wait(&empty_bar[s], ((it / TC_STAGES) & 1) ^ 1);
                            tc::mbar_arrive_expect_tx(&full_bar[s], TC_STAGE_BYTES);
                            uint8_t* dst = stage_mem + (size_t)s * TC_STAGE_BYTES;
                            tc::bulk_g2s(dst, Aimg + (size_t)kt * (2 * tc::kTcImgBytes), 2 * tc::kTcImgBytes,
                                         &full_bar[s]);
                            tc::bulk_g2s(dst + 2 * tc::kTcImgBytes, Bimg + (size_t)kt * (2 * tc::kTcImgBytes),
                                         2 * tc::kTcImgBytes, &full_bar[s]);
                        }
                    }
                }
            } else if (warp == 1) {
                if (lane == 0) {
                    uint32_t it = stage_it, ai = acc_it;
                    for (int ib = 0; ib < nb; ++ib, ++ai) {
                        const int nkt = (ib + 1) * (PBM / tc::kTcK);
                        const uint32_t buf = ai & 1;
                        tc::mbar_wait(&accempty_bar[buf], ((ai >> 1) & 1) ^ 1);
                        tc::tc_fence_after_sync();
                        const uint32_t d_tmem = tmem_base + buf * 128;
                        for (int kt = 0; kt < nkt; ++kt, ++it) {
                            const int s = it % TC_STAGES;
                            tc::mbar_wait(&full_bar[s], (it / TC_STAGES) & 1);
                            tc::tc_fence_after_sync();
                            const uint32_t base = tc::smem_u32(stage_mem + (size_t)s * TC_STAGE_BYTES);
#pragma unroll
                            for (int j = 0; j < tc::kTcK / 8; ++j) {
                                const uint32_t koff = j * 2 * tc::kTcLBO;
                                const uint64_t a_hi = tc::umma_desc_kmajor_noswz(base + koff, tc::kTcLBO, tc::kTcSBO);
                                const uint64_t a_lo = tc::umma_desc_kmajor_noswz(base + tc::kTcImgBytes + koff,
                                                                                 tc::kTcLBO, tc::kTcSBO);
                                const uint64_t b_hi = tc::umma_desc_kmajor_noswz(base + 2 * tc::kTcImgBytes + koff,
                                                                                 tc::kTcLBO, tc::kTcSBO);
                                const uint64_t b_lo = tc::umma_desc_kmajor_noswz(base + 3 * tc::kTcImgBytes + koff,
                                                                                 tc::kTcLBO, tc::kTcSBO);
                                tc::umma_tf32(d_tmem, a_hi, b_hi, idesc, (kt | j) ? 1u : 0u);
                                tc::umma_tf32(d_tmem, a_hi, b_lo, idesc, 1u);
                                tc::umma_tf32(d_tmem, a_lo, b_hi, idesc, 1u);
                            }
                            tc::umma_commit(&empty_bar[s]);
                        }
                        tc::umma_commit(&accfull_bar[buf]);
                    }
                }
            }
            float csq[PBN];
            if (warp >= 4) {
                const int q = warp & 3;
#pragma unroll
                for (int j = 0; j < PBN; ++j) csq[j] = 0.f;
                uint32_t ai = acc_it;
                for (int ib = 0; ib < nb; ++ib, ++ai) {
                    const uint32_t buf = ai & 1;
                    tc::mbar_wait(&accfull_bar[buf], (ai >> 1) & 1);
                    tc::tc_fence_after_sync();
                    const uint32_t taddr = tmem_base + buf * 128 + ((uint32_t)(q * 32) << 16);
#pragma unroll
                    for (int cc = 0; cc < PBN; cc += 32) {
                        uint32_t r[32];
                        tc::tmem_ld_32x32(taddr + cc, r);
                        tc::tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const float v = __uint_as_float(r[j]);
                            csq[cc + j] = fmaf(v, v, csq[cc + j]);
                        }
                    }
                    tc::tc_fence_before_sync();
                    __syncwarp();
                    if (lane == 0) tc::mbar_arrive(&accempty_bar[buf]);
                }
            }
            // every role advanced by the same amounts
            {
                uint32_t stages = 0;
                for (int ib = 0; ib < nb; ++ib) stages += (ib + 1) * (PBM / tc::kTcK);
                stage_it += stages;
                acc_it += nb;
            }
            tc::tc_fence_before_sync();
            __syncthreads();
            tc::tc_fence_after_sync();
            if (warp >= 4) {
                const int q = warp & 3;
                // sum over the 32 rows (lanes) of this quadrant; fp64 from here on
#pragma unroll
                for (int j = 0; j < PBN; ++j) {
                    double v = (double)csq[j];
                    v += __shfl_xor_sync(0xffffffffu, v, 16);
                    v += __shfl_xor_sync(0xffffffffu, v, 8);
                    v += __shfl_xor_sync(0xffffffffu, v, 4);
                    v += __shfl_xor_sync(0xffffffffu, v, 2);
                    v += __shfl_xor_sync(0xffffffffu, v, 1);
                    if (lane == 0) red_s[q][j] = v;
                }
            }
            __syncthreads();
            if (tid < PBN) {
                const int c = tid;
                const double colsq = ((red_s[0][c] + red_s[1][c]) + red_s[2][c]) + red_s[3][c];
                double val = 0.0;
                candidate_epilogue(P, G, g, mu_s[0][c] + mu_s[1][c], colsq, c0 + c, base_s[c], prod_s[c], &val);
                if (P.sel_cta && g == P.n_gps - 1)
                    runsel_update<1>(sel_s, P.sel_k, tid, val, c0 + c + P.index_base, c0 + c < P.m);
            }
            tc::fence_proxy_async_smem();
            __syncthreads();
        }
    }
    if (P.sel_cta && tid < PBN) runsel_store(sel_s, P.sel_cta + blockIdx.x, tid);
    tc::tc_fence_before_sync();
    __syncthreads();
    if (warp == 1) tc::tmem_dealloc(tmem_base, TC_TMEM_COLS);
}

// ---------------------------------------------------------------------------------------
// fp32 mode, overlapped version (d <= 16): the K* build of the NEXT job runs on four dedicated
// builder warps while the tensor cores work on the current one, so the fp64 front end disappears
// behind the GEMM.  512 threads = 4 warp groups:
//   warps 0-3   producer (warp 0, one lane), tcgen05.mma issuer (warp 1, one lane), 2 spare
//   warps 4-7   epilogue: tcgen05.ld of their TMEM quadrant, warp transpose-reduce of v^2 over the
//               32 rows, cross-warp sum, per-candidate acquisition epilogue
//   warps 8-15  builders: two threads per candidate; K* in fp64 -> tf32 (hi,lo) operand images in a
//               double-buffered global scratch, K* alpha_ in fp64
// A job is one (candidate tile, GP).  mbarriers: full/empty (smem stages), accfull/accempty (TMEM
// buffers), b_ready[2] (builders -> producer/epilogue), job_done[2] (epilogue -> builders).
// ---------------------------------------------------------------------------------------
constexpr int TC2_NT = 512;       // 16 warps: 4 (producer, MMA, 2 spare) + 4 epilogue + 8 builders
constexpr int TC2_NB = 256;       // builder threads: two per candidate column (row halves of every chunk)
constexpr int kPredictSmemBytesTc2 = TC_STAGES * TC_STAGE_BYTES + 2 * PA_CHUNK * kPredictMaxDimRegs * 8;  // 212992

template <int COV>
__device__ __forceinline__ void tc2_build_job(const PredictParams& P, const GpDev& G, long long c0, int btid,
                                              uint8_t* __restrict__ Bimg, double* xs_s, double* mu_out) {
    const int d = P.d, np = G.np;
    const int c = btid & (PBN - 1), half = btid >> 7;
    double xc[kPredictMaxDimRegs];
    {
        const long long gi = c0 + c;
#pragma unroll
        for (int j = 0; j < kPredictMaxDimRegs; ++j) {
            double v = 0.0;
            if (j < d && gi < P.m) {
                v = candidate_coord(P, gi, j);
                if (G.xform && G.xform[j] == B200BO_XFORM_ROUND) v = rint(v);
                v = v / G.ls[j];
            }
            xc[j] = v;
        }
    }
    const int chunk_pieces = PA_CHUNK * d / 2;
    auto load_chunk = [&](int buf, int ch) {
        const double* src = G.Xs + (size_t)ch * PA_CHUNK * d;
        double* dst = xs_s + (size_t)buf * PA_CHUNK * kPredictMaxDimRegs;
        for (int q = btid; q < chunk_pieces; q += TC2_NB) cp_async16_cg(dst + 2 * q, src + 2 * q);
    };
    const int nch = np / PA_CHUNK;
    load_chunk(0, 0);
    cp_async_commit();
    double mu_acc = 0.0;
    constexpr int R = 8;
    for (int ch = 0; ch < nch; ++ch) {
        if (ch + 1 < nch) load_chunk((ch + 1) & 1, ch + 1);
        cp_async_commit();
        cp_async_wait<1>();
        tc::named_bar_sync(2, TC2_NB);
        const double* xs = xs_s + (size_t)(ch & 1) * PA_CHUNK * kPredictMaxDimRegs;
        for (int r0 = half * (PA_CHUNK / 2); r0 < (half + 1) * (PA_CHUNK / 2); r0 += R) {
            double r2[R];
#pragma unroll
            for (int q = 0; q < R; ++q) r2[q] = 0.0;
            if ((d & 1) == 0) {
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
            } else {
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
            }
            float hi[R], lo[R];
#pragma unroll
            for (int q = 0; q < R; ++q) {
                const int n = ch * PA_CHUNK + r0 + q;
                double kv = G.constv * cov_eval<COV>(r2[q]);
                if (n >= G.n) kv = 0.0;
                hi[q] = tc::to_tf32((float)kv);
                lo[q] = tc::to_tf32((float)(kv - (double)hi[q]));
                mu_acc = fma(__ldg(G.alphav + n), kv, mu_acc);
            }
            const int n0 = ch * PA_CHUNK + r0;
            uint8_t* img = Bimg + (size_t)(n0 >> 5) * (2 * tc::kTcImgBytes);
#pragma unroll
            for (int h4 = 0; h4 < 2; ++h4) {
                const int off = tc::tc_img_offset(c, (n0 & 31) + 4 * h4);
                *reinterpret_cast<float4*>(img + off) =
                    make_float4(hi[4 * h4], hi[4 * h4 + 1], hi[4 * h4 + 2], hi[4 * h4 + 3]);
                *reinterpret_cast<float4*>(img + tc::kTcImgBytes + off) =
                    make_float4(lo[4 * h4], lo[4 * h4 + 1], lo[4 * h4 + 2], lo[4 * h4 + 3]);
            }
        }
        tc::named_bar_sync(2, TC2_NB);
    }
    cp_async_wait<0>();
    *mu_out = mu_acc;
}

// Row blocks are processed in PAIRS against each K* stage (two TMEM accumulators per buffer), which
// halves the HBM traffic of the K* images (their 0.6 GB working set cannot live in L2).  A stage
// holds HALF a k-tile (16 k) of every operand image: [A(ib0) hi|lo][A(ib1) hi|lo][B hi|lo], 6 x 8 KiB;
// four stages keep three loads in flight behind the MMAs (the 2-stage/32-k version was latency bound).
constexpr int TC2_STAGES = 4;
constexpr int TC2_HALF = tc::kTcImgBytes / 2;         // 8192: k 0..15 or 16..31 of an image
constexpr int TC2_STAGE_BYTES = 6 * TC2_HALF;         // 49152
constexpr int TC2_TMEM_COLS = 512;                    // 2 buffers x 2 row blocks x 128 columns
static_assert(TC2_STAGES * TC2_STAGE_BYTES + 2 * PA_CHUNK * kPredictMaxDimRegs * 8 == kPredictSmemBytesTc2, "smem");

__global__ void __launch_bounds__(TC2_NT, 1) predict_acq_tc2_kernel(const PredictParams P) {
    extern __shared__ __align__(16) double smem[];
    __shared__ double mu_s[2][2][PBN];  // [job parity][row half][candidate]
    __shared__ float red_s[4][PBN];
    __shared__ uint64_t full_bar[TC2_STAGES], empty_bar[TC2_STAGES], accfull_bar[2], accempty_bar[2];
    __shared__ uint64_t bready_bar[2], jobdone_bar[2];
    __shared__ uint32_t tmem_base_s;
    __shared__ SelShared sel_s;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint8_t* stage_mem = reinterpret_cast<uint8_t*>(smem);
    double* xs_s = reinterpret_cast<double*>(stage_mem + TC2_STAGES * TC2_STAGE_BYTES);
    uint8_t* scratch = reinterpret_cast<uint8_t*>(P.scratch + (long long)blockIdx.x * P.scratch_stride);
    const size_t buf_bytes = (size_t)P.scratch_stride * 4;  // two buffers of scratch_stride*4 bytes each
    const long long ntiles = (P.m + PBN - 1) / PBN;
    const long long my_tiles = (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x;
    const long long njobs = my_tiles * P.n_gps;
    constexpr int KT_PER_BLOCK = PBM / tc::kTcK;  // 4 k-tiles per 128 rows
    constexpr uint32_t IMG2 = 2 * tc::kTcImgBytes;

    if (tid == 0) {
        for (int s = 0; s < TC2_STAGES; ++s) {
            tc::mbar_init(&full_bar[s], 1);
            tc::mbar_init(&empty_bar[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            tc::mbar_init(&accfull_bar[b], 1);
            tc::mbar_init(&accempty_bar[b], 4);
            tc::mbar_init(&bready_bar[b], TC2_NB / 32);
            tc::mbar_init(&jobdone_bar[b], 4);
        }
        tc::mbar_fence_init();
    }
    if (warp == 1) tc::tmem_alloc(&tmem_base_s, TC2_TMEM_COLS);
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();
    const uint32_t tmem_base = tmem_base_s;

    // measurement hooks (B200BO_TC_DEBUG): bit 0 = builders only, bit 1 = GEMM only (results invalid)
    const bool dbg_no_gemm = (P.pad0 & 1) != 0, dbg_no_build = (P.pad0 & 2) != 0;
    if (warp == 0) {
        // ------------------------------ producer -------------------------------------------
        if (lane == 0 && !dbg_no_gemm) {
            uint32_t it = 0;
            for (long long j = 0; j < njobs; ++j) {
                const GpDev& G = P.gp[j % P.n_gps];
                const int nb = G.np / PBM, nkt_row = G.np / tc::kTcK;
                const uint8_t* Bimg = scratch + (size_t)(j & 1) * buf_bytes;
                tc::mbar_wait(&bready_bar[j & 1], (uint32_t)((j >> 1) & 1));
                for (int ib0 = 0; ib0 < nb; ib0 += 2) {
                    const bool two = ib0 + 1 < nb;
                    const int nkt0 = (ib0 + 1) * KT_PER_BLOCK, nkt = two ? nkt0 + KT_PER_BLOCK : nkt0;
                    const uint8_t* A0 = G.linv_tc + (size_t)ib0 * nkt_row * IMG2;
                    const uint8_t* A1 = A0 + (size_t)nkt_row * IMG2;
                    for (int ht = 0; ht < 2 * nkt; ++ht, ++it) {
                        const int kt = ht >> 1;
                        const size_t hoff = (size_t)(ht & 1) * TC2_HALF;  // which 16-k half of the images
                        const int s = it % TC2_STAGES;
                        tc::mbar_wait(&empty_bar[s], ((it / TC2_STAGES) & 1) ^ 1);
                        const bool a0 = kt < nkt0;
                        tc::mbar_arrive_expect_tx(&full_bar[s], (1u + (a0 ? 1u : 0u) + (two ? 1u : 0u)) * 2u * TC2_HALF);
                        uint8_t* dst = stage_mem + (size_t)s * TC2_STAGE_BYTES;
                        const uint8_t* a0p = A0 + (size_t)kt * IMG2 + hoff;
                        const uint8_t* a1p = A1 + (size_t)kt * IMG2 + hoff;
                        const uint8_t* bp = Bimg + (size_t)kt * IMG2 + hoff;
                        if (a0) {
                            tc::bulk_g2s(dst, a0p, TC2_HALF, &full_bar[s]);
                            tc::bulk_g2s(dst + TC2_HALF, a0p + tc::kTcImgBytes, TC2_HALF, &full_bar[s]);
                        }
                        if (two) {
                            tc::bulk_g2s(dst + 2 * TC2_HALF, a1p, TC2_HALF, &full_bar[s]);
                            tc::bulk_g2s(dst + 3 * TC2_HALF, a1p + tc::kTcImgBytes, TC2_HALF, &full_bar[s]);
                        }
                        tc::bulk_g2s(dst + 4 * TC2_HALF, bp, TC2_HALF, &full_bar[s]);
                        tc::bulk_g2s(dst + 5 * TC2_HALF, bp + tc::kTcImgBytes, TC2_HALF, &full_bar[s]);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------ tcgen05.mma issuer ---------------------------------
        if (lane == 0 && !dbg_no_gemm) {
            const uint32_t idesc = tc::umma_idesc_tf32(128, 128);
            uint32_t it = 0, ai = 0;
            for (long long j = 0; j < njobs; ++j) {
                const GpDev& G = P.gp[j % P.n_gps];
                const int nb = G.np / PBM;
                for (int ib0 = 0; ib0 < nb; ib0 += 2, ++ai) {
                    const bool two = ib0 + 1 < nb;
                    const int nkt0 = (ib0 + 1) * KT_PER_BLOCK, nkt = two ? nkt0 + KT_PER_BLOCK : nkt0;
                    const uint32_t buf = ai & 1;
                    tc::mbar_wait(&accempty_bar[buf], ((ai >> 1) & 1) ^ 1);
                    tc::tc_fence_after_sync();
                    const uint32_t d0 = tmem_base + buf * 256, d1 = d0 + 128;
                    for (int ht = 0; ht < 2 * nkt; ++ht, ++it) {
                        const int kt = ht >> 1;
                        const int s = it % TC2_STAGES;
                        tc::mbar_wait(&full_bar[s], (it / TC2_STAGES) & 1);
                        tc::tc_fence_after_sync();
                        const uint32_t base = tc::smem_u32(stage_mem + (size_t)s * TC2_STAGE_BYTES);
                        const bool a0 = kt < nkt0;
#pragma unroll
                        for (int k8 = 0; k8 < 2; ++k8) {
                            const uint32_t koff = k8 * 2 * tc::kTcLBO;
                            const uint64_t b_hi = tc::umma_desc_kmajor_noswz(base + 4 * TC2_HALF + koff, tc::kTcLBO, tc::kTcSBO);
                            const uint64_t b_lo = tc::umma_desc_kmajor_noswz(base + 5 * TC2_HALF + koff, tc::kTcLBO, tc::kTcSBO);
                            if (a0) {
                                const uint64_t a_hi = tc::umma_desc_kmajor_noswz(base + koff, tc::kTcLBO, tc::kTcSBO);
                                const uint64_t a_lo = tc::umma_desc_kmajor_noswz(base + TC2_HALF + koff, tc::kTcLBO, tc::kTcSBO);
                                tc::umma_tf32(d0, a_hi, b_hi, idesc, (ht | k8) ? 1u : 0u);
                                tc::umma_tf32(d0, a_hi, b_lo, idesc, 1u);
                                tc::umma_tf32(d0, a_lo, b_hi, idesc, 1u);
                            }
                            if (two) {
                                const uint64_t a_hi = tc::umma_desc_kmajor_noswz(base + 2 * TC2_HALF + koff, tc::kTcLBO, tc::kTcSBO);
                                const uint64_t a_lo = tc::umma_desc_kmajor_noswz(base + 3 * TC2_HALF + koff, tc::kTcLBO, tc::kTcSBO);
                                tc::umma_tf32(d1, a_hi, b_hi, idesc, (ht | k8) ? 1u : 0u);
                                tc::umma_tf32(d1, a_hi, b_lo, idesc, 1u);
                                tc::umma_tf32(d1, a_lo, b_hi, idesc, 1u);
                            }
                        }
                        tc::umma_commit(&empty_bar[s]);
                    }
                    tc::umma_commit(&accfull_bar[buf]);
                }
            }
        }
    } else if (warp >= 4 && warp < 8) {
        // ------------------------------ epilogue --------------------------------------------
        const int q = warp & 3, etid = tid - 128;
        uint32_t ai = 0;
        double base_neg = 0.0, prod = 1.0;
        if (P.sel_cta) {
            runsel_begin(sel_s, P.sel_cta + blockIdx.x, P.sel_resume, etid);
            tc::named_bar_sync(1, 128);
        }
        for (long long j = 0; j < njobs; ++j) {
            const int g = (int)(j % P.n_gps);
            const GpDev& G = P.gp[g];
            const long long tile = blockIdx.x + (j / P.n_gps) * gridDim.x;
            const int nb = G.np / PBM;
            float csum[4] = {0.f, 0.f, 0.f, 0.f};  // columns lane, lane+32, lane+64, lane+96
            for (int ib0 = 0; ib0 < nb && !dbg_no_gemm; ib0 += 2, ++ai) {
                const bool two = ib0 + 1 < nb;
                const uint32_t buf = ai & 1;
                tc::mbar_wait(&accfull_bar[buf], (ai >> 1) & 1);
                tc::tc_fence_after_sync();
                const uint32_t taddr = tmem_base + buf * 256 + ((uint32_t)(q * 32) << 16);
                const int nchunk = two ? 8 : 4;
                for (int cc = 0; cc < nchunk; ++cc) {
                    uint32_t r[32];
                    tc::tmem_ld_32x32(taddr + cc * 32, r);
                    tc::tmem_ld_wait();
                    float v[32];
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        const float x = __uint_as_float(r[i]);
                        v[i] = x * x;
                    }
                    // warp transpose-reduce: afterwards lane L holds the sum over the 32 rows of column L
#pragma unroll
                    for (int s = 16; s >= 1; s >>= 1) {
#pragma unroll
                        for (int i = 0; i < s; ++i) {
                            const bool up = (lane & s) != 0;
                            const float send = up ? v[i] : v[i + s];
                            const float recv = __shfl_xor_sync(0xffffffffu, send, s);
                            v[i] = (up ? v[i + s] : v[i]) + recv;
                        }
                    }
                    const int c4 = cc & 3;
                    csum[0] += (c4 == 0) ? v[0] : 0.f;
                    csum[1] += (c4 == 1) ? v[0] : 0.f;
                    csum[2] += (c4 == 2) ? v[0] : 0.f;
                    csum[3] += (c4 == 3) ? v[0] : 0.f;
                }
                tc::tc_fence_before_sync();
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(&accempty_bar[buf]);
            }
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) red_s[q][cc * 32 + lane] = csum[cc];
            tc::named_bar_sync(1, 128);
            const double colsq =
                (((double)red_s[0][etid] + (double)red_s[1][etid]) + (double)red_s[2][etid]) + (double)red_s[3][etid];
            tc::mbar_wait(&bready_bar[j & 1], (uint32_t)((j >> 1) & 1));  // acquire the builders' mean
            double val = 0.0;
            candidate_epilogue(P, G, g, mu_s[j & 1][0][etid] + mu_s[j & 1][1][etid], colsq, tile * PBN + etid,
                               base_neg, prod, &val);
            if (P.sel_cta && g == P.n_gps - 1)
                runsel_update<1>(sel_s, P.sel_k, etid, val, tile * PBN + etid + P.index_base, tile * PBN + etid < P.m);
            tc::named_bar_sync(1, 128);
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&jobdone_bar[j & 1]);
        }
        if (P.sel_cta) runsel_store(sel_s, P.sel_cta + blockIdx.x, etid);
    } else if (warp >= 8) {
        // ------------------------------ builders ---------------------------------------------
        const int btid = tid - 256;
        for (long long j = 0; j < njobs; ++j) {
            const int g = (int)(j % P.n_gps);
            const GpDev& G = P.gp[g];
            const long long tile = blockIdx.x + (j / P.n_gps) * gridDim.x;
            tc::mbar_wait(&jobdone_bar[j & 1], (uint32_t)(((j >> 1) & 1) ^ 1));  // buffer j&1 free again
            uint8_t* Bimg = scratch + (size_t)(j & 1) * buf_bytes;
            double mu = 0.0;
            if (!dbg_no_build) switch (cov_code(G.family, G.nu)) {
                case 0: tc2_build_job<0>(P, G, tile * PBN, btid, Bimg, xs_s, &mu); break;
                case 1: tc2_build_job<1>(P, G, tile * PBN, btid, Bimg, xs_s, &mu); break;
                case 2: tc2_build_job<2>(P, G, tile * PBN, btid, Bimg, xs_s, &mu); break;
                default: tc2_build_job<3>(P, G, tile * PBN, btid, Bimg, xs_s, &mu); break;
            }
            mu_s[j & 1][btid >> 7][btid & (PBN - 1)] = mu;
            tc::fence_proxy_async_global();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&bready_bar[j & 1]);
        }
    }
    tc::tc_fence_before_sync();
    __syncthreads();
    if (warp == 1) tc::tmem_dealloc(tmem_base, TC2_TMEM_COLS);
}

// L^-1 (fp64, row-major) -> tf32 (hi, lo) operand images [ib][kt][hi|lo][16 KiB] (lower k-tiles only)
__global__ void __launch_bounds__(256) pretile_linv_tc_kernel(const double* __restrict__ W, int np,
                                                              uint8_t* __restrict__ out) {
    const int kt = blockIdx.x, ib = blockIdx.y;
    if (kt >= (ib + 1) * (PBM / tc::kTcK)) return;
    uint8_t* img = out + ((size_t)ib * (np / tc::kTcK) + kt) * (2 * tc::kTcImgBytes);
    for (int idx = threadIdx.x; idx < PBM * tc::kTcK; idx += 256) {
        const int r = idx / tc::kTcK, k = idx % tc::kTcK;
        const double w = W[(size_t)(ib * PBM + r) * np + kt * tc::kTcK + k];
        const float hi = tc::to_tf32((float)w);
        const float lo = tc::to_tf32((float)(w - (double)hi));
        const int off = tc::tc_img_offset(r, k);
        *reinterpret_cast<float*>(img + off) = hi;
        *reinterpret_cast<float*>(img + tc::kTcImgBytes + off) = lo;
    }
}

// =======================================================================================
// Small-batch path (m <= a few hundred candidates: the single-row / finite-difference-stencil
// calls L-BFGS-B makes, R/bayes_opt/acquisition.py:366).  The tiled kernel would run one
// 128-wide tile on one SM; here the triangular product V = Linv K*^T for up to 32 candidates is
// spread over the whole GPU as fixed-size work units (64 rows x <=512 k), with fixed-order
// partial sums (deterministic).  Three launches per pass of 32 candidates and per GP:
//   small_kstar_kernel  K*[k][c] (+ per-block partials of K* alpha_)
//   small_trsv_kernel   partial V for each (row-block, k-chunk) unit
//   small_finish_kernel sum units, square, reduce rows, epilogue (all GPs)
// =======================================================================================
constexpr int SMC = 32;      // candidates per pass
constexpr int SROWS = 64;    // rows per unit
constexpr int SKCH = 512;    // k per unit
constexpr int SKT = 32;      // k sub-tile staged in smem
constexpr int SWSTR = SKT + 2;

struct SmallGp {
    const double* W;        // [np][np] Linv row-major
    double* ksm;            // [np][SMC]
    double* partial;        // [nunits][SROWS][SMC]
    double* mu_part;        // [np/128][SMC]
    double* colsq_rb;       // [np/SROWS][SMC] per pass: sum over the rows of a row block of V^2
    const int2* unit_tab;   // [nunits] (row-block, k-chunk)
    const int2* rb_tab;     // [np/SROWS] (first unit, number of units)
};

// One launch group covers up to SMAXP passes (blockIdx.y / blockIdx.x of the finish kernel = pass): the
// passes of a batch run concurrently (an L-BFGS-B round of all seeds + their stencils is ~170 rows = 6
// passes: 3 launches instead of 18, and six times as many CTAs in flight).
constexpr int SMAXP = 8;

struct SmallParams {
    PredictParams P;
    SmallGp sg[B200BO_MAX_GPS];
    long long c0;  // first candidate of pass 0 of this launch group
    long long m_end;  // one past the last candidate of the batch
    int nunits[B200BO_MAX_GPS];  // work units per pass (stride of `partial` between passes)
};

__device__ __forceinline__ long long small_pass_c0(const SmallParams& S, int pass) { return S.c0 + (long long)pass * SMC; }
__device__ __forceinline__ int small_pass_mc(const SmallParams& S, int pass) {
    const long long left = S.m_end - small_pass_c0(S, pass);
    return (int)(left < SMC ? (left < 0 ? 0 : left) : SMC);
}

// K*[k][c] for one block of 128 training rows and one pass of 32 candidates (blockIdx.y = pass): thread =
// (candidate c, group of 16 rows); the training row is a warp-wide broadcast load, K* rows are written as
// coalesced 256-byte segments; per-candidate partial of K* alpha_ over the block in a fixed order.
__global__ void __launch_bounds__(256)
small_kstar_kernel(const SmallParams S, int g) {
    const GpDev& G = S.P.gp[g];
    const SmallGp& Q = S.sg[g];
    __shared__ double xc_s[SMC][B200BO_MAX_DIM + 1];
    __shared__ double wsum[8][SMC];
    const int tid = threadIdx.x, d = S.P.d;
    const int pass = blockIdx.y, mc = small_pass_mc(S, pass);
    const long long pc0 = small_pass_c0(S, pass);
    double* ksm = Q.ksm + (size_t)pass * G.np * SMC;
    double* mu_part = Q.mu_part + (size_t)pass * (G.np / 128) * SMC;
    for (int idx = tid; idx < SMC * d; idx += 256) {
        const int c = idx / d, j = idx - c * d;
        double v = 0.0;
        if (c < mc) {
            v = candidate_coord(S.P, pc0 + c, j);
            if (G.xform && G.xform[j] == B200BO_XFORM_ROUND) v = rint(v);
            v = v / G.ls[j];
        }
        xc_s[c][j] = v;
    }
    __syncthreads();
    const int c = tid & 31, rg = tid >> 5;
    double mu_acc = 0.0;
    for (int q = 0; q < 16; ++q) {
        const int n = blockIdx.x * 128 + rg * 16 + q;
        double kv = 0.0;
        if (c < mc && n < G.n) {
            const double* xr = G.Xs + (size_t)n * d;
            double r2 = 0.0;
            for (int j = 0; j < d; ++j) {
                const double df = xc_s[c][j] - xr[j];
                r2 = fma(df, df, r2);
            }
            kv = G.constv * cov_from_r2(r2, G.family, G.nu);
        }
        ksm[(size_t)n * SMC + c] = kv;
        mu_acc = fma(G.alphav[n], kv, mu_acc);
    }
    wsum[rg][c] = mu_acc;
    __syncthreads();
    if (tid < SMC) {
        double t = 0.0;
#pragma unroll
        for (int r = 0; r < 8; ++r) t += wsum[r][tid];
        mu_part[(size_t)blockIdx.x * SMC + tid] = t;
    }
}

// Partial V for one work unit (64 rows x <= 512 k) and a GROUP of up to STPG passes (blockIdx.y = group): the W tile
// is staged once per k sub-tile and used for every pass of the group.  (One CTA per pass re-read L^-1 six times per
// round; all eight passes in one CTA needed 178 registers and 83 KB -> one CTA per SM, half the throughput.  Groups
// of four: ~100 registers, 49 KB -> two to three resident CTAs per SM.)
constexpr int STPG = 4;
constexpr int kSmallTrsvSmemBytes = (SROWS * SWSTR + STPG * SKT * SMC) * 8;  // 50176
__global__ void __launch_bounds__(256, 2)
small_trsv_kernel(const SmallParams S, int g, int npass) {
    const GpDev& G = S.P.gp[g];
    const SmallGp& Q = S.sg[g];
    extern __shared__ __align__(16) double strsv_smem[];
    double* Wt = strsv_smem;                  // [SROWS][SWSTR]
    double* Kt = strsv_smem + SROWS * SWSTR;  // [STPG][SKT][SMC]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int p0 = blockIdx.y * STPG, pn = min(STPG, npass - p0);
    const int2 u = Q.unit_tab[blockIdx.x];
    const int r0 = u.x * SROWS;
    const int kbeg = u.y * SKCH;
    const int kend = min(kbeg + SKCH, r0 + SROWS);
    const int np = G.np;
    double acc[STPG][8];
#pragma unroll
    for (int p = 0; p < STPG; ++p)
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[p][q] = 0.0;
    for (int k0 = kbeg; k0 < kend; k0 += SKT) {
        for (int idx = tid; idx < SROWS * SKT; idx += 256) {
            const int r = idx / SKT, kk = idx % SKT;
            Wt[r * SWSTR + kk] = Q.W[(size_t)(r0 + r) * np + k0 + kk];
        }
        for (int p = 0; p < pn; ++p) {
            const double* ksm = Q.ksm + (size_t)(p0 + p) * np * SMC + (size_t)k0 * SMC;
            for (int idx = tid; idx < SKT * SMC; idx += 256) Kt[p * SKT * SMC + idx] = ksm[idx];
        }
        __syncthreads();
#pragma unroll 2
        for (int kk = 0; kk < SKT; kk += 2) {
            double2 w[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) w[q] = *reinterpret_cast<const double2*>(&Wt[(warp * 8 + q) * SWSTR + kk]);
#pragma unroll
            for (int p = 0; p < STPG; ++p) {
                if (p < pn) {
                    const double k0v = Kt[p * SKT * SMC + kk * SMC + lane], k1v = Kt[p * SKT * SMC + (kk + 1) * SMC + lane];
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        acc[p][q] = fma(w[q].x, k0v, acc[p][q]);
                        acc[p][q] = fma(w[q].y, k1v, acc[p][q]);
                    }
                }
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int p = 0; p < STPG; ++p) {
        if (p < pn) {
            double* out = Q.partial + ((size_t)(p0 + p) * S.nunits[g] + blockIdx.x) * SROWS * SMC;
#pragma unroll
            for (int q = 0; q < 8; ++q) out[(warp * 8 + q) * SMC + lane] = acc[p][q];
        }
    }
}

// Per (row block of 64 rows, pass): sum the k-chunk partials of every row in a fixed order, square, and reduce the
// 64 rows -> colsq_rb[pass][row block][candidate].  grid (np / 64, npass).
__global__ void __launch_bounds__(256)
small_reduce_kernel(const SmallParams S, int g) {
    const GpDev& G = S.P.gp[g];
    const SmallGp& Q = S.sg[g];
    __shared__ double red[8][SMC];
    const int tid = threadIdx.x, c = tid & 31, rg = tid >> 5;
    const int pass = blockIdx.y;
    const int2 rb = Q.rb_tab[blockIdx.x];
    const double* partial = Q.partial + (size_t)pass * S.nunits[g] * SROWS * SMC;
    double s = 0.0;
    for (int q = 0; q < 8; ++q) {
        const int r = rg * 8 + q;
        double v = 0.0;
        for (int j = 0; j < rb.y; ++j) v += partial[((size_t)(rb.x + j) * SROWS + r) * SMC + c];
        s = fma(v, v, s);
    }
    red[rg][c] = s;
    __syncthreads();
    if (tid < SMC) {
        double t = 0.0;
#pragma unroll
        for (int r = 0; r < 8; ++r) t += red[r][tid];
        Q.colsq_rb[((size_t)pass * (G.np / SROWS) + blockIdx.x) * SMC + tid] = t;
    }
}

// Per pass (blockIdx.x): sum the row-block and K* alpha_ partials in index order, then the per-candidate epilogue
// of every GP.  256 threads = 32 candidates x 8 slices of the partial lists (fixed-order two-level sum).
__global__ void __launch_bounds__(256)
small_finish_kernel(const SmallParams S) {
    __shared__ double red[8][SMC];
    __shared__ double colsq_s[B200BO_MAX_GPS][SMC];
    __shared__ double mu_s[B200BO_MAX_GPS][SMC];
    const int tid = threadIdx.x, c = tid & 31, sl = tid >> 5;
    const int pass = blockIdx.x, mc = small_pass_mc(S, pass);
    const long long pc0 = small_pass_c0(S, pass);
    for (int g = 0; g < S.P.n_gps; ++g) {
        const GpDev& G = S.P.gp[g];
        const SmallGp& Q = S.sg[g];
        const int nrb = G.np / SROWS, nb = G.np / 128;
        const double* crb = Q.colsq_rb + (size_t)pass * nrb * SMC;
        const double* mu_part = Q.mu_part + (size_t)pass * nb * SMC;
        // slice sl sums a contiguous range of the lists; the 8 slice sums are then added in order
        double s = 0.0;
        for (int b = sl * ((nrb + 7) / 8); b < min(nrb, (sl + 1) * ((nrb + 7) / 8)); ++b) s += crb[(size_t)b * SMC + c];
        red[sl][c] = s;
        __syncthreads();
        if (sl == 0) {
            double t = 0.0;
#pragma unroll
            for (int r = 0; r < 8; ++r) t += red[r][c];
            colsq_s[g][c] = t;
        }
        __syncthreads();
        s = 0.0;
        for (int b = sl * ((nb + 7) / 8); b < min(nb, (sl + 1) * ((nb + 7) / 8)); ++b) s += mu_part[(size_t)b * SMC + c];
        red[sl][c] = s;
        __syncthreads();
        if (sl == 0) {
            double t = 0.0;
#pragma unroll
            for (int r = 0; r < 8; ++r) t += red[r][c];
            mu_s[g][c] = t;
        }
        __syncthreads();
    }
    if (sl == 0 && c < mc) {
        double base_neg = 0.0, prod = 1.0;
        for (int g = 0; g < S.P.n_gps; ++g)
            candidate_epilogue(S.P, S.P.gp[g], g, mu_s[g][c], colsq_s[g][c], pc0 + c, base_neg, prod);
    }
}

// ---------------------------------------------------------------------------------------
// Selection: record 0 = np.argmin(vals) (first NaN wins, ties -> lowest index);
// records 1..k = the k smallest by (value, index) with NaN last (np.argsort order for
// distinct values).  Single CTA of 1024 threads; k+1 fixed-order passes over vals (L2).
// (R/bayes_opt/acquisition.py:313-317)
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024)
select_kernel(const double* __restrict__ vals, long long m, int k, SelRecord* __restrict__ out,
              long long index_base) {
    __shared__ unsigned long long skey[1024];
    __shared__ long long sidx[1024];
    __shared__ unsigned long long prev_key;
    __shared__ long long prev_idx;
    const int tid = threadIdx.x;
    for (int round = 0; round <= k; ++round) {
        const bool argmin_round = (round == 0);
        const bool bounded = (round >= 2);
        const unsigned long long pk = bounded ? prev_key : 0ull;
        const long long pi = bounded ? prev_idx : -1;
        unsigned long long bk = 0xFFFFFFFFFFFFFFFFull;
        long long bi = -1;
        for (long long i = tid; i < m; i += 1024) {
            const double v = vals[i];
            const unsigned long long key = argmin_round ? key_nan_first(v) : key_nan_last(v);
            if (bounded && (key < pk || (key == pk && i <= pi))) continue;
            if (bi < 0 || key < bk) {  // i increases, so ties keep the lowest index
                bk = key;
                bi = i;
            }
        }
        skey[tid] = bk;
        sidx[tid] = bi;
        __syncthreads();
        for (int s = 512; s > 0; s >>= 1) {
            if (tid < s) {
                const unsigned long long ok = skey[tid + s];
                const long long oi = sidx[tid + s];
                const long long mi = sidx[tid];
                const bool take = (oi >= 0) && (mi < 0 || ok < skey[tid] || (ok == skey[tid] && oi < mi));
                if (take) {
                    skey[tid] = ok;
                    sidx[tid] = oi;
                }
            }
            __syncthreads();
        }
        if (tid == 0) {
            const long long w = sidx[0];
            out[round].index = (w >= 0) ? w + index_base : -1;
            out[round].value = (w >= 0) ? vals[w] : CUDART_NAN;
            prev_key = skey[0];
            prev_idx = (w >= 0) ? w : (long long)0x7FFFFFFFFFFFFFFFll;
        }
        __syncthreads();
    }
}

}  // namespace b200bo
