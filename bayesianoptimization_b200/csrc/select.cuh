// select.cuh - (value, index) selection fused into the predict/acquisition kernels, and the
// device-side candidate source of the throughput mode (Philox4x32-10).
//
// Replaces the selection step of AcquisitionFunction._random_sample_minimize
// (R/bayes_opt/acquisition.py:312-317:  ys.argmin(), np.argsort(ys)[:n_x_seeds]) WITHOUT materialising
// ys[M]: every CTA of the persistent kernel keeps the k smallest (key, index) pairs it has produced so far
// in shared memory (sorted), folds each tile's 128 fresh values into that list, and writes the list once
// at the end; one tiny kernel k-way-merges the per-CTA lists.  (key, index) is a strict total order, so
// the result is independent of the grid size, the tile->CTA assignment and the insertion order:
// bit-reproducible, identical for any number of GPUs.
//   record 0     np.argmin semantics: first NaN wins, else the smallest value, ties -> lowest index
//   records 1..k np.argsort order: ascending value, ties -> lowest index, NaN last
#pragma once
#include "common.cuh"

namespace b200bo {

constexpr int SEL_MAXK = B200BO_MAX_TOPK;
constexpr long long SEL_NOIDX = 0x7FFFFFFFFFFFFFFFll;

struct SelRecord {
    double value;
    long long index;
};

// sorted ascending by (key, idx); unused slots hold (~0, SEL_NOIDX)
struct SelList {
    unsigned long long key[SEL_MAXK];
    long long idx[SEL_MAXK];
    long long nan_idx;  // lowest global index with a NaN value, or SEL_NOIDX
    long long pad;
};

// shared-memory working state of one CTA
struct SelShared {
    SelList list;
    unsigned long long skey[128];
    long long sidx[128];
    int nstage;
    int pad;
};

__device__ __forceinline__ double key_to_value(unsigned long long key) {
    if (key == 0xFFFFFFFFFFFFFFFFull) return CUDART_NAN;
    const unsigned long long u = (key & 0x8000000000000000ull) ? (key & 0x7FFFFFFFFFFFFFFFull) : ~key;
    return __longlong_as_double((long long)u);
}

__device__ __forceinline__ void named_bar_sync_sel(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;\n" ::"r"(id), "r"(nthreads) : "memory");
}

// called by thread t == 0 of the group before the first update
__device__ __forceinline__ void runsel_init(SelShared& S, int t) {
    for (int i = t; i < SEL_MAXK; i += 128) {
        S.list.key[i] = 0xFFFFFFFFFFFFFFFFull;
        S.list.idx[i] = SEL_NOIDX;
    }
    if (t == 0) {
        S.list.nan_idx = SEL_NOIDX;
        S.nstage = 0;
    }
}

// start of a launch: fresh lists, or (chunked batches) the lists the previous launch stored
__device__ __forceinline__ void runsel_begin(SelShared& S, const SelList* prev, int resume, int t) {
    if (!resume) {
        runsel_init(S, t);
        return;
    }
    for (int i = t; i < SEL_MAXK; i += 128) {
        S.list.key[i] = prev->key[i];
        S.list.idx[i] = prev->idx[i];
    }
    if (t == 0) {
        S.list.nan_idx = prev->nan_idx;
        S.nstage = 0;
    }
}

// Fold one tile's values into the CTA's list.  Called by exactly 128 threads (t = 0..127) that own
// the named barrier BAR; v/gi = this thread's value and GLOBAL candidate index, valid = in range.
template <int BAR>
__device__ __forceinline__ void runsel_update(SelShared& S, int k, int t, double v, long long gi, bool valid) {
    const unsigned long long key = key_nan_last(v);
    if (valid && isnan(v)) atomicMin(reinterpret_cast<long long*>(&S.list.nan_idx), gi);
    const unsigned long long kk = S.list.key[k - 1];
    const long long ki = S.list.idx[k - 1];
    if (valid && (key < kk || (key == kk && gi < ki))) {
        const int pos = atomicAdd(&S.nstage, 1);
        S.skey[pos] = key;
        S.sidx[pos] = gi;
    }
    named_bar_sync_sel(BAR, 128);
    if (t == 0) {
        // only thread 0 reads the counter in this interval (it also resets it below): no other thread's speculative
        // load of it may race with that write
        const int ns = *reinterpret_cast<volatile int*>(&S.nstage);
        for (int s = 0; s < ns; ++s) {
            const unsigned long long nk = S.skey[s];
            const long long ni = S.sidx[s];
            int p = k - 1;
            if (!(nk < S.list.key[p] || (nk == S.list.key[p] && ni < S.list.idx[p]))) continue;
            while (p > 0 && (nk < S.list.key[p - 1] || (nk == S.list.key[p - 1] && ni < S.list.idx[p - 1]))) {
                S.list.key[p] = S.list.key[p - 1];
                S.list.idx[p] = S.list.idx[p - 1];
                --p;
            }
            S.list.key[p] = nk;
            S.list.idx[p] = ni;
        }
        if (ns > 0) S.nstage = 0;
    }
    named_bar_sync_sel(BAR, 128);
}

__device__ __forceinline__ void runsel_store(const SelShared& S, SelList* out, int t) {
    for (int i = t; i < SEL_MAXK; i += 128) {
        out->key[i] = S.list.key[i];
        out->idx[i] = S.list.idx[i];
    }
    if (t == 0) out->nan_idx = S.list.nan_idx;
}

// k-way merge of the per-CTA sorted lists -> (k+1) records.  One CTA of 256 threads.
__global__ void __launch_bounds__(256)
merge_sel_kernel(const SelList* __restrict__ lists, int nlists, int k, SelRecord* __restrict__ out) {
    __shared__ int head[1024];
    __shared__ unsigned long long rkey[256];
    __shared__ long long ridx[256];
    __shared__ int rlist[256];
    __shared__ long long nan_s[256];
    const int tid = threadIdx.x;
    long long nan_idx = SEL_NOIDX;
    for (int l = tid; l < nlists; l += 256) {
        head[l] = 0;
        const long long ni = lists[l].nan_idx;
        nan_idx = ni < nan_idx ? ni : nan_idx;
    }
    nan_s[tid] = nan_idx;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (tid < s && nan_s[tid + s] < nan_s[tid]) nan_s[tid] = nan_s[tid + s];
        __syncthreads();
    }
    for (int round = 0; round < k; ++round) {
        unsigned long long bk = 0xFFFFFFFFFFFFFFFFull;
        long long bi = SEL_NOIDX;
        int bl = -1;
        for (int l = tid; l < nlists; l += 256) {
            const int h = head[l];
            if (h >= k) continue;
            const unsigned long long ck = lists[l].key[h];
            const long long ci = lists[l].idx[h];
            if (ci == SEL_NOIDX) continue;
            if (bl < 0 || ck < bk || (ck == bk && ci < bi)) {
                bk = ck;
                bi = ci;
                bl = l;
            }
        }
        rkey[tid] = bk;
        ridx[tid] = bi;
        rlist[tid] = bl;
        __syncthreads();
        for (int s = 128; s > 0; s >>= 1) {
            if (tid < s) {
                const int ol = rlist[tid + s];
                if (ol >= 0 && (rlist[tid] < 0 || rkey[tid + s] < rkey[tid] ||
                                (rkey[tid + s] == rkey[tid] && ridx[tid + s] < ridx[tid]))) {
                    rkey[tid] = rkey[tid + s];
                    ridx[tid] = ridx[tid + s];
                    rlist[tid] = ol;
                }
            }
            __syncthreads();
        }
        if (tid == 0) {
            if (rlist[0] >= 0) {
                out[1 + round].value = key_to_value(rkey[0]);
                out[1 + round].index = ridx[0];
                head[rlist[0]] += 1;
            } else {
                out[1 + round].value = CUDART_NAN;
                out[1 + round].index = -1;
            }
        }
        __syncthreads();
    }
    if (tid == 0) {
        if (nan_s[0] != SEL_NOIDX) {
            out[0].value = CUDART_NAN;
            out[0].index = nan_s[0];
        } else {
            out[0] = out[1];
        }
    }
}

// ---------------------------------------------------------------------------------------
// Pruned selection (predict16.cuh, b200bo.cu eval_core).  sigma^2 = prior - sum_i V_i^2 and every term is >= 0,
// so the partial sum over the first row blocks of L^-1 (same per-thread / shuffle / red[] reduction tree as the
// full sum) bounds sigma from above in floating point too: adding a non-negative number under round-to-nearest
// never decreases a sum, and the clamp, the scaling by y_std^2 and sqrt are monotone.  mu is exact after phase A,
// and EI, UCB (kappa >= 0) and PoI (for a < 0) increase with sigma, so the acquisition at sd_up bounds the
// selected value val = -acq from below.  A candidate whose lower bound lies above tau, the k-th smallest exact
// key of candidates of the same call, cannot enter the records.
// ---------------------------------------------------------------------------------------
// Computed EI / PoI are not monotone at the ulp level (near z << 0 the two EI terms cancel and the rounding
// of z is amplified ~z^2 times): the bound is lowered by this relative margin of the summed magnitudes.
constexpr double kPruneRelMargin = 9.313225746154785e-10;  // 2^-30
constexpr double kDblMin = 2.2250738585072014e-308;

// lower bound on val = -acq for a candidate with exact mean and sd <= sd_up; NaN = no usable bound (non-finite
// intermediates, a == 0 where sd may clamp to 0 and 0/0 gives NaN, PoI with a >= 0): evaluate it in full
__device__ __forceinline__ double prune_lower_bound(int kind, double mean, double sd_up, double y_max, double xi,
                                                    double kappa) {
    if (kind == B200BO_ACQ_UCB) {
        const double v = -(mean + kappa * sd_up);  // exact bound: every operation is monotone in sd (kappa >= 0)
        return isfinite(v) ? v : CUDART_NAN;
    }
    const double a = mean - y_max - xi;
    if (!isfinite(a) || a == 0.0 || !isfinite(sd_up)) return CUDART_NAN;
    const double z = a / sd_up;
    const double cdf = ndtr(z);
    if (kind == B200BO_ACQ_POI) return a < 0.0 ? -(cdf + (kPruneRelMargin * cdf + kDblMin)) : CUDART_NAN;
    const double pdf = norm_pdf(z);
    const double up = a * cdf + sd_up * pdf;  // the EI expression of candidate_epilogue
    const double v = -(up + (kPruneRelMargin * (fabs(a) * cdf + sd_up * pdf) + kDblMin));
    return isfinite(v) ? v : CUDART_NAN;
}

// screen key: 0 (below every value key) forces a full evaluation
__device__ __forceinline__ unsigned long long prune_key(double lb) { return isnan(lb) ? 0ull : key_nan_last(lb); }

// tau = key of the k-th pilot record (records as merge_sel_kernel writes them; an empty record gives the
// all-ones key: nothing is pruned)
__global__ void prune_tau_kernel(const SelRecord* __restrict__ rec, int k, unsigned long long* tau) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    *tau = rec[k].index < 0 ? 0xFFFFFFFFFFFFFFFFull : key_nan_last(rec[k].value);
}

// Merge of per-device record sets (multi-GPU exchange, SURVEY.md 8e): rec[g][0] = device g's argmin record
// (NaN first), rec[g][1..k] = its top-k (ascending, index < 0 = empty).  Same ordering rules as above.
__global__ void merge_records_kernel(const SelRecord* __restrict__ rec, int ndev, int k, SelRecord* __restrict__ out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const int stride = k + 1;
    unsigned long long bk = 0;
    long long bi = -1;
    double bv = CUDART_NAN;
    for (int g = 0; g < ndev; ++g) {
        const SelRecord r = rec[g * stride];
        if (r.index < 0) continue;
        const unsigned long long key = key_nan_first(r.value);
        if (bi < 0 || key < bk || (key == bk && r.index < bi)) {
            bk = key;
            bi = r.index;
            bv = r.value;
        }
    }
    out[0].value = bv;
    out[0].index = bi;
    int head[64];
    for (int g = 0; g < ndev && g < 64; ++g) head[g] = 1;
    for (int round = 0; round < k; ++round) {
        int bg = -1;
        unsigned long long ck = 0;
        long long ci = 0;
        double cv = 0.0;
        for (int g = 0; g < ndev && g < 64; ++g) {
            if (head[g] > k) continue;
            const SelRecord r = rec[g * stride + head[g]];
            if (r.index < 0) continue;
            const unsigned long long key = key_nan_last(r.value);
            if (bg < 0 || key < ck || (key == ck && r.index < ci)) {
                bg = g;
                ck = key;
                ci = r.index;
                cv = r.value;
            }
        }
        if (bg >= 0) {
            out[1 + round].value = cv;
            out[1 + round].index = ci;
            head[bg] += 1;
        } else {
            out[1 + round].value = CUDART_NAN;
            out[1 + round].index = -1;
        }
    }
}

// ---------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11) - counter-based, so a candidate's coordinates depend only on
// (seed, global row index, column): identical whatever tile, CTA or GPU evaluates the row.
//   counter = (row_lo, row_hi, col/2, 0), key = (seed_lo, seed_hi)
//   u64 word (col even: o0 | o1 << 32 ; col odd: o2 | o3 << 32) -> u = (word >> 11) * 2^-53
//   x = lo + (hi - lo) * u        (two roundings, no fma: oracle/gp_oracle.py philox_uniform matches bitwise)
// ---------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ void philox4x32_10(unsigned c0, unsigned c1, unsigned c2, unsigned c3,
                                                       unsigned k0, unsigned k1, unsigned out[4]) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned long long p0 = (unsigned long long)0xD2511F53u * c0;
        const unsigned long long p1 = (unsigned long long)0xCD9E8D57u * c2;
        const unsigned n0 = (unsigned)(p1 >> 32) ^ c1 ^ k0;
        const unsigned n1 = (unsigned)p1;
        const unsigned n2 = (unsigned)(p0 >> 32) ^ c3 ^ k1;
        const unsigned n3 = (unsigned)p0;
        c0 = n0;
        c1 = n1;
        c2 = n2;
        c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0;
    out[1] = c1;
    out[2] = c2;
    out[3] = c3;
}

__device__ __forceinline__ double philox_coord(unsigned long long seed, long long row, int col, double lo,
                                               double span) {
    unsigned o[4];
    philox4x32_10((unsigned)row, (unsigned)((unsigned long long)row >> 32), (unsigned)(col >> 1), 0u,
                  (unsigned)seed, (unsigned)(seed >> 32), o);
    const unsigned long long w = (col & 1) ? ((unsigned long long)o[2] | ((unsigned long long)o[3] << 32))
                                           : ((unsigned long long)o[0] | ((unsigned long long)o[1] << 32));
    const double u = (double)(w >> 11) * 1.1102230246251565e-16;  // 2^-53
    return __dadd_rn(lo, __dmul_rn(span, u));
}

// rows of the Philox candidate matrix for a list of global indices (the winners' coordinates)
__global__ void philox_rows_kernel(unsigned long long seed, const double* __restrict__ bounds, int d,
                                   const SelRecord* __restrict__ rec, int nrec, double* __restrict__ out) {
    const int r = blockIdx.x;
    if (r >= nrec) return;
    const long long row = rec[r].index;
    for (int j = threadIdx.x; j < d; j += blockDim.x)
        out[(size_t)r * d + j] = (row >= 0) ? philox_coord(seed, row, j, bounds[j], bounds[d + j]) : CUDART_NAN;
}

}  // namespace b200bo
