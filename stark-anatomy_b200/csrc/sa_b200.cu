// sa_b200.cu -- kernels and C ABI (include/sa_b200.h) of the B200 NTT + FRI engine.
// Compile: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -shared -Xcompiler -fPIC
//
// Reference behaviour reproduced (bit-exact): code/ntt.py:3-30,61,133,172, code/fri.py:85,
// code/merkle.py:6-27, code/algebra.py:53-57,75-94.
#include <cuda_runtime.h>
#include <pthread.h>
#include <sched.h>

#include <algorithm>
#include <atomic>
#include <cctype>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/sa_b200.h"
#include "field.cuh"
#include "fri_merkle.cuh"
#include "hash.cuh"
#include "ntt_plan.cuh"
#include "ntt_tile.cuh"

using namespace sa;


// ------------------------------------------------------------------ plumbing --
static thread_local std::string g_last_error;
static std::atomic<uint64_t> g_launches{0};

#define SA_CUDA(expr)                                                                          \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            g_last_error = std::string(#expr) + ": " + cudaGetErrorString(_e);                 \
            return SA_ECUDA;                                                                   \
        }                                                                                      \
    } while (0)
#define SA_LAUNCH_CHECK()                                                                      \
    do {                                                                                       \
        g_launches.fetch_add(1, std::memory_order_relaxed);                                    \
        cudaError_t _e = cudaGetLastError();                                                   \
        if (_e != cudaSuccess) {                                                               \
            g_last_error = std::string("kernel launch: ") + cudaGetErrorString(_e);            \
            return SA_ECUDA;                                                                   \
        }                                                                                      \
    } while (0)

static inline fe fe_from_limbs(const uint64_t x[2]) {
    return fe_make((uint32_t)x[0], (uint32_t)(x[0] >> 32), (uint32_t)x[1], (uint32_t)(x[1] >> 32));
}
static inline bool host_is_pow2(size_t n) { return n && !(n & (n - 1)); }
static inline int host_log2(size_t n) {
    int l = 0;
    while ((size_t(1) << l) < n) l++;
    return l;
}

// ------------------------------------------------------------------- kernels --
template <int LOGL, int ELOG, int C>
struct TileLaunch {
    using P = TilePlan<LOGL, ELOG, C>;
    // aim for 1024 resident threads per SM with 8-element blocks (<= 64 registers) and 512 with
    // 16-element blocks (<= 128 registers)
    static constexpr int TARGET = (P::EL <= 3 && LOGL > 3) ? 1024 : 512;
    static constexpr int MINB = TARGET / P::THREADS > 0 ? TARGET / P::THREADS : 1;
};

template <int LOGL, int ELOG, int C, int FLAGS>
__global__ void __launch_bounds__(TilePlan<LOGL, ELOG, C>::THREADS, TileLaunch<LOGL, ELOG, C>::MINB)
    ntt_tile_kernel(const __grid_constant__ TileArgs a, long long total_tiles, int tiles_per_batch) {
    using P = TilePlan<LOGL, ELOG, C>;
    using S = TileStages<LOGL, ELOG, C, FLAGS>;
    extern __shared__ uint4 sa_smem_u4[];
    fe *smem = reinterpret_cast<fe *>(sa_smem_u4);
    const int tic = threadIdx.x / P::TPT, t = threadIdx.x % P::TPT;
    const long long tile = (long long)blockIdx.x * P::TPC + tic;
    const bool valid = tile < total_tiles;
    const long long b = valid ? tile / tiles_per_batch : 0;
    const int col0 = valid ? (int)(tile % tiles_per_batch) * C : 0;
    fe *sm = smem + (size_t)tic * P::L * C;
    fe *tw = nullptr;
    uint64_t *bar = nullptr;
    // programmatic dependent launch: the next launch on this stream (pass 2 after pass 1, the next transform
    // of a chain) may become resident while this grid still runs; it parks at griddepcontrol.wait below
    asm volatile("griddepcontrol.launch_dependents;");
    if constexpr (P::NLOOP > 0) {
        // stage the twiddle table of this tile length into shared memory (bulk-async copy + mbarrier);
        // the table is a cached constant of the plan, not an output of the preceding launch
        tw = smem + P::TILE_BYTES / sizeof(fe);
        bar = reinterpret_cast<uint64_t *>(tw + P::L);
        if (threadIdx.x == 0) tile_stage_twiddles(tw, a.tw, (uint32_t)P::TW_BYTES, bar);
        __syncthreads();  // the barrier is initialised before anybody polls it
    }
    // everything the preceding launch wrote (the intermediate of the four-step split, or this call's input)
    // is complete and visible after this point; a no-op for a launch without the PDL attribute
    asm volatile("griddepcontrol.wait;" ::: "memory");
#pragma unroll 1
    for (int st = 0; st < P::NLOOP; st++) {
        S::full(st, t, sm, a, b, col0, valid, tw, bar);
        __syncthreads();
    }
    S::last(t, sm, a, b, col0, valid);
}

// out[slot(e)] = base^e * lead (Montgomery form) for e < count; 16 consecutive powers per thread.
// swz != 0 stores in the bank-spreading order of tile_tw_slot (stage-twiddle tables, count % 64 == 0
// or count < 8 so the permutation stays inside the table).
__global__ void k_pow_table(fe *out, fe base_m, fe lead_m, long long count, int swz) {
    const long long e0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 16;
    if (e0 >= count) return;
    fe acc = fe_montmul(fe_mont_pow_u64(base_m, (uint64_t)e0), lead_m);
    for (int i = 0; i < 16 && e0 + i < count; i++) {
        const long long e = e0 + i;
        tile_st(out + (swz ? (long long)tile_tw_slot((int)e) : e), acc);
        acc = fe_montmul(acc, base_m);
    }
}
// out[k * n2 + j] = w^(k*j) * scale (Montgomery form): row k is the power table of w^k
__global__ void k_twb_table(fe *out, fe w_m, fe scale_m, int n1, int n2) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long per_row = (n2 + 15) / 16;
    const long long k = idx / per_row;
    const long long j0 = (idx % per_row) * 16;
    if (k >= n1) return;
    const fe wk = fe_mont_pow_u64(w_m, (uint64_t)k);
    fe acc = fe_montmul(fe_mont_pow_u64(wk, (uint64_t)j0), scale_m);
    for (int i = 0; i < 16 && j0 + i < n2; i++) {
        tile_st(out + k * n2 + j0 + i, acc);
        acc = fe_montmul(acc, wk);
    }
}

__global__ void k_pointwise_mul(fe *out, const fe *a, const fe *b, long long n) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        tile_st(out + i, fe_montmul(fe_to_mont(tile_ld(a + i)), tile_ld(b + i)));
}
// out = a / b with Montgomery's batch-inversion trick over 8 strided elements per thread
__global__ void k_pointwise_div(fe *out, const fe *a, const fe *b, long long n, int *zero_flag) {
    constexpr int G = 8;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (long long base = i0; base < n; base += stride * G) {
        fe bm[G], pre[G];
        fe acc = fe_mont_one();
#pragma unroll
        for (int g = 0; g < G; g++) {
            const long long i = base + g * stride;
            fe v = (i < n) ? tile_ld(b + i) : fe_one();
            if (fe_is_zero(v)) {
                *zero_flag = 1;
                v = fe_one();
            }
            bm[g] = fe_to_mont(v);
            pre[g] = acc;
            acc = fe_montmul(acc, bm[g]);
        }
        fe inv = fe_mont_inv(acc);
#pragma unroll
        for (int g = G - 1; g >= 0; g--) {
            const long long i = base + g * stride;
            const fe binv = fe_montmul(inv, pre[g]);  // Montgomery form of 1/b[i]
            inv = fe_montmul(inv, bm[g]);
            if (i < n) tile_st(out + i, fe_montmul(tile_ld(a + i), binv));
        }
    }
}
// out[i] = in[i] * factor^i; thread handles i, i + T, i + 2T, ... with running factor^T
__global__ void k_scale(fe *out, const fe *in, long long n, fe factor_m, fe factor_T_m) {
    const long long T = (long long)gridDim.x * blockDim.x;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe f = fe_mont_pow_u64(factor_m, (uint64_t)i);
    for (; i < n; i += T) {
        tile_st(out + i, fe_montmul(tile_ld(in + i), f));
        f = fe_montmul(f, factor_T_m);
    }
}
// Horner, one thread per point (coefficients are read through the read-only path, broadcast)
__global__ void k_poly_eval(fe *out, const fe *coeffs, long long ncoef, const fe *points, long long npts) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= npts) return;
    const fe x_m = fe_to_mont(tile_ld(points + j));
    fe acc = fe_zero();
    for (long long i = ncoef - 1; i >= 0; i--) acc = fe_add(fe_montmul(acc, x_m), tile_ldg(coeffs + i));
    tile_st(out + j, acc);
}
// prod (X - d_i): one CTA, coefficients in shared memory, one sweep per domain point
constexpr int ZF_THREADS = 1024, ZF_MAXK = 4096, ZF_PER = (ZF_MAXK + 1 + ZF_THREADS - 1) / ZF_THREADS;
__global__ void __launch_bounds__(ZF_THREADS) k_zerofier(fe *out, const fe *domain, int k) {
    extern __shared__ uint4 sa_smem_u4[];
    fe *c = reinterpret_cast<fe *>(sa_smem_u4);
    fe *dm = c + (k + 1);
    const int tid = threadIdx.x;
    for (int j = tid; j <= k; j += ZF_THREADS) c[j] = (j == 0) ? fe_one() : fe_zero();
    for (int j = tid; j < k; j += ZF_THREADS) dm[j] = fe_to_mont(tile_ld(domain + j));
    __syncthreads();
    for (int i = 0; i < k; i++) {
        const fe d = dm[i];
        fe val[ZF_PER];
#pragma unroll
        for (int s = 0; s < ZF_PER; s++) {
            const int j = tid + s * ZF_THREADS;
            if (j <= i + 1) {  // new[j] = old[j-1] - d * old[j]
                const fe lower = j ? c[j - 1] : fe_zero();
                const fe cur = (j <= i) ? c[j] : fe_zero();
                val[s] = fe_sub(lower, fe_montmul(cur, d));
            }
        }
        __syncthreads();
#pragma unroll
        for (int s = 0; s < ZF_PER; s++) {
            const int j = tid + s * ZF_THREADS;
            if (j <= i + 1) c[j] = val[s];
        }
        __syncthreads();
    }
    for (int j = tid; j <= k; j += ZF_THREADS) tile_st(out + j, c[j]);
}
// Lagrange interpolation pieces.  q_i = z / (X - d_i) by synthetic division (descending m):
//   q_i[m-1] = z[m] + d_i * q_i[m];  D_i = q_i(d_i) = z'(d_i);  weight w_i = v_i / D_i
__global__ void k_interp_weights(fe *w_m, const fe *domain, const fe *values, const fe *z, int k, int *zero_flag) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= k) return;
    const fe d = fe_to_mont(tile_ld(domain + i));
    fe carry = fe_zero(), denom = fe_zero();
    for (int m = k; m > 0; m--) {
        carry = fe_add(tile_ldg(z + m), fe_montmul(carry, d));
        denom = fe_add(fe_montmul(denom, d), carry);
    }
    if (fe_is_zero(denom)) {
        *zero_flag = 1;
        denom = fe_one();
    }
    tile_st(w_m + i, fe_montmul(fe_to_mont(tile_ld(values + i)), fe_mont_inv(fe_to_mont(denom))));
}
// QT[m][i] = w_i * q_i[m]  (coalesced over i)
__global__ void k_interp_rows(fe *QT, const fe *domain, const fe *w_m, const fe *z, int k) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= k) return;
    const fe d = fe_to_mont(tile_ld(domain + i)), w = tile_ld(w_m + i);
    fe carry = fe_zero();
    for (int m = k; m > 0; m--) {
        carry = fe_add(tile_ldg(z + m), fe_montmul(carry, d));
        tile_st(QT + (size_t)(m - 1) * k + i, fe_montmul(carry, w));
    }
}
// out[m] = sum_i QT[m][i]; one CTA per coefficient
__global__ void __launch_bounds__(256) k_interp_colsum(fe *out, const fe *QT, int k) {
    __shared__ uint4 red_u4[256];
    fe *red = reinterpret_cast<fe *>(red_u4);
    const int m = blockIdx.x, tid = threadIdx.x;
    fe acc = fe_zero();
    for (int i = tid; i < k; i += 256) acc = fe_add(acc, tile_ld(QT + (size_t)m * k + i));
    red[tid] = acc;
    __syncthreads();
    for (int w = 128; w >= 1; w >>= 1) {
        if (tid < w) red[tid] = fe_add(red[tid], red[tid + w]);
        __syncthreads();
    }
    if (tid == 0) tile_st(out + m, red[0]);
}
// ---- multi-GPU assembly by push: one read of a finished block, one fully coalesced 16-byte store per lane
// and destination (a warp writes 512 contiguous bytes to every peer: NVLink sees whole packets, unlike the 64-byte
// segments the transform's own last pass produces)
struct PushArgs {
    uint4 *dst[TILE_MAX_PEERS];
    int ndst;
};
__global__ void __launch_bounds__(256) k_push(const __grid_constant__ PushArgs a, const uint4 *src, size_t n16) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + 3 * stride < n16; i += 4 * stride) {  // four loads in flight per thread
        uint4 v[4];
#pragma unroll
        for (int u = 0; u < 4; u++) v[u] = __ldcs(src + i + u * stride);
#pragma unroll
        for (int u = 0; u < 4; u++)
#pragma unroll
            for (int p = 0; p < TILE_MAX_PEERS; p++)
                if (p < a.ndst) a.dst[p][i + u * stride] = v[u];
    }
    for (; i < n16; i += stride) {
        const uint4 v = __ldcs(src + i);
#pragma unroll
        for (int p = 0; p < TILE_MAX_PEERS; p++)
            if (p < a.ndst) a.dst[p][i] = v;
    }
}

// variant: ONE multimem.st per 16 bytes through a multicast address (NVLS): the store leaves this GPU once and the
// NVSwitch replicates it into every rank's buffer bound to the multicast object (sa_push_mcast)
__global__ void __launch_bounds__(256) k_push_mcast(fe *mc, const fe *src, size_t n16) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + 3 * stride < n16; i += 4 * stride) {
        fe v[4];
#pragma unroll
        for (int u = 0; u < 4; u++) v[u] = tile_ld(src + i + u * stride);
#pragma unroll
        for (int u = 0; u < 4; u++) tile_st_multicast(mc + i + u * stride, v[u]);
    }
    for (; i < n16; i += stride) tile_st_multicast(mc + i, tile_ld(src + i));
}

// ---- subproduct tree over a domain of k points (fast_zerofier / fast_interpolate, ntt.py:66-130) ----
// The k points sit in the first k of K = 2^ceil(log2 k) leaf slots.  Level j has K >> j nodes of
// m = 2^j coefficients each, stored back to back.  A node whose leaf range lies completely inside the
// domain is FULL: its zerofier is monic of degree exactly m and only the low m coefficients are stored
// (the leading 1 is implied).  Any other node is stored EXPLICITLY (degree < m, all coefficients); a node
// without points is the constant 1.  With child vectors vL, vR a parent is
//     cyclic_product_2m(vL, vR) + x^m * ([L full] vR + [R full] vL)
// (the cyclic product of size 2m never wraps: both factors have degree < m), FULL iff both children are.
__device__ __forceinline__ bool tree_full(long long node, int mlog, long long k) { return ((node + 1) << mlog) <= k; }
__global__ void k_tree_leaves(fe *v0, const fe *domain, long long k, long long K) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < K) tile_st(v0 + i, i < k ? fe_neg(tile_ld(domain + i)) : fe_one());
}
// dst node (2m slots) = [src node (m coefficients), m zeros]
__global__ void k_tree_pad(fe *dst, const fe *src, long long K, int mlog) {
    const long long stride = (long long)gridDim.x * blockDim.x, m = 1ll << mlog;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < 2 * K; idx += stride) {
        const long long node = idx >> (mlog + 1), t = idx & (2 * m - 1);
        tile_st(dst + idx, t < m ? tile_ld(src + node * m + t) : fe_zero());
    }
}
// transformed children (blocks of 2m) -> transformed parents: out[p][t] = in[2p][t] * in[2p+1][t]
__global__ void k_tree_pairmul(fe *out, const fe *in, long long K, int mlog) {
    const long long stride = (long long)gridDim.x * blockDim.x, two_m = 2ll << mlog;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < K; idx += stride) {
        const long long p = idx >> (mlog + 1), t = idx & (two_m - 1);
        const fe a = tile_ld(in + (2 * p) * two_m + t), b = tile_ld(in + (2 * p + 1) * two_m + t);
        tile_st(out + idx, fe_montmul(fe_to_mont(a), b));
    }
}
// interpolation up-sweep: out[p][t] = P[2p][t] * V[2p+1][t] + P[2p+1][t] * V[2p][t]
__global__ void k_tree_cross(fe *out, const fe *Pt, const fe *Vt, long long K, int mlog) {
    const long long stride = (long long)gridDim.x * blockDim.x, two_m = 2ll << mlog;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < K; idx += stride) {
        const long long p = idx >> (mlog + 1), t = idx & (two_m - 1);
        const long long l = (2 * p) * two_m + t, r = (2 * p + 1) * two_m + t;
        const fe a = fe_montmul(fe_to_mont(tile_ld(Pt + l)), tile_ld(Vt + r));
        const fe b = fe_montmul(fe_to_mont(tile_ld(Pt + r)), tile_ld(Vt + l));
        tile_st(out + idx, fe_add(a, b));
    }
}
// parent[p][m + t] += [L full] right[t] + [R full] left[t]; (left, right) = the child vectors of `add`
// (the zerofier tree adds the children's own vectors, the interpolation sweep the OTHER tree's: P_L * M_R
// picks up x^m * P_L when M_R is full, so `swap` exchanges the roles)
__global__ void k_tree_fix(fe *parent, const fe *add, long long K, int mlog, long long k, int swap) {
    const long long stride = (long long)gridDim.x * blockDim.x, m = 1ll << mlog;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < K / 2; idx += stride) {
        const long long p = idx >> mlog, t = idx & (m - 1);
        const bool lfull = tree_full(2 * p, mlog, k), rfull = tree_full(2 * p + 1, mlog, k);
        if (!lfull && !rfull) continue;
        const fe left = tile_ld(add + (2 * p) * m + t), right = tile_ld(add + (2 * p + 1) * m + t);
        fe acc = tile_ld(parent + p * 2 * m + m + t);
        if (swap) {
            if (rfull) acc = fe_add(acc, left);
            if (lfull) acc = fe_add(acc, right);
        } else {
            if (lfull) acc = fe_add(acc, right);
            if (rfull) acc = fe_add(acc, left);
        }
        tile_st(parent + p * 2 * m + m + t, acc);
    }
}
// out[i] = (i + 1) * z[i + 1], i < k  (formal derivative of a polynomial with k + 1 coefficients)
__global__ void k_derivative(fe *out, const fe *z, long long k) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < k) tile_st(out + i, fe_montmul(fe_to_mont(fe_from_u64((uint64_t)(i + 1))), tile_ld(z + i + 1)));
}
// leaves of the interpolation sweep: q_i = v_i / M'(d_i) for i < k, 0 for the empty slots
__global__ void k_tree_qleaves(fe *P0, const fe *q, long long k, long long K) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < K) tile_st(P0 + i, i < k ? tile_ld(q + i) : fe_zero());
}
// zerofier coefficients from the tree's root vector: k == K -> implied leading 1
__global__ void k_tree_root(fe *out, const fe *root, long long k, long long K) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= k) tile_st(out + i, (i == K) ? fe_one() : tile_ld(root + i));
}

// ---- multi-point evaluation over the same tree (fast_evaluate, ntt.py:82-100, and M'(d_i) of fast_interpolate) ----
// The reference walks DOWN a remainder tree (f mod left zerofier, f mod right zerofier, ...).  Here the walk down is
// the TRANSPOSE of the interpolation up-sweep (Bostan-Lecerf-Schost): the up-sweep q -> P = sum q_i M / (X - d_i) is
// linear, rev(P) / rev(M) = sum q_i / (1 - d_i x) has the power sums sum_i q_i d_i^j as coefficients, i.e.
// (transposed Vandermonde) = (multiply by alpha = 1 / rev(M) mod x^n) o (reverse) o (up-sweep), so
//   f(d_i) = (up-sweep)^T [ (rev(f) * alpha mod x^n) shifted ],
// and the transposed up-sweep turns every product P_L * M_R into a CORRELATION with M_R: with the node transforms
// kept from the build, c_L = IDFT(DFT(c_node)[t] * DFT(M_R)[-t])[0..m) (+ c_node[m..2m) for the implied leading 1 of
// a full M_R), c_R likewise with M_L.  No division anywhere: one power-series inverse (Newton) at the top, then per
// level one batched forward transform, one pointwise kernel, one batched inverse transform, one fix-up.
// W (two blocks of 4s): [0] = rev_k(z) mod x^2s, zero padded; [1] = alpha mod x^s, zero padded.  z has k + 1 coefficients.
__global__ void k_series_pad(fe *W, const fe *z, long long k, const fe *alpha, long long s) {
    const long long stride = (long long)gridDim.x * blockDim.x, n4 = 4 * s;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < 2 * n4; idx += stride) {
        const long long t = idx & (n4 - 1);
        fe v = fe_zero();
        if (idx < n4) {
            if (t < 2 * s && t <= k) v = tile_ld(z + (k - t));
        } else if (t < s) {
            v = tile_ld(alpha + t);
        }
        tile_st(W + idx, v);
    }
}
// Newton step in the transform domain: W[0][t] = a * (2 - r * a), r = W[0][t], a = W[1][t]  (degree < 4s: no wrap)
__global__ void k_series_step(fe *W, long long n4) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    const fe two = fe_make(2, 0, 0, 0);
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n4; t += stride) {
        const fe r = tile_ld(W + t), a_m = fe_to_mont(tile_ld(W + n4 + t));
        const fe ra = fe_montmul(a_m, r);  // canonical r * a
        tile_st(W + t, fe_montmul(a_m, fe_sub(two, ra)));
    }
}
// W (two blocks of n2): [0] = rev_{n-1}(f) (f has nf <= n coefficients), [1] = alpha mod x^n, both zero padded
__global__ void k_eval_top_pad(fe *W, const fe *f, long long nf, const fe *alpha, long long n, long long n2) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < 2 * n2; idx += stride) {
        const long long t = idx & (n2 - 1);
        fe v = fe_zero();
        if (idx < n2) {
            if (t < n && n - 1 - t < nf) v = tile_ld(f + (n - 1 - t));
        } else if (t < n) {
            v = tile_ld(alpha + t);
        }
        tile_st(W + idx, v);
    }
}
// root vector of the walk down: c[i] = s[n - k + i] for i < k (s = rev(f) * alpha), 0 for the empty slots
__global__ void k_eval_root(fe *c, const fe *s, long long n, long long k, long long K) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < K) tile_st(c + i, i < k ? tile_ld(s + (n - k + i)) : fe_zero());
}
// O[child][t] = chat[parent][t] * VT[sibling][(2m - t) mod 2m]   (child blocks of 2m; VT = level-mlog transforms)
__global__ void k_tree_down(fe *O, const fe *chat, const fe *VT, long long K, int mlog) {
    const long long stride = (long long)gridDim.x * blockDim.x, two_m = 2ll << mlog;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < 2 * K; idx += stride) {
        const long long child = idx >> (mlog + 1), t = idx & (two_m - 1);
        const fe a = tile_ld(chat + (child >> 1) * two_m + t);
        const fe b = tile_ld(VT + (child ^ 1) * two_m + ((two_m - t) & (two_m - 1)));
        tile_st(O + idx, fe_montmul(fe_to_mont(a), b));
    }
}
// next[child][j] = O[child][j] + [sibling full] * cur[parent][m + j],  j < m
__global__ void k_tree_down_fix(fe *next, const fe *O, const fe *cur, long long K, int mlog, long long k) {
    const long long stride = (long long)gridDim.x * blockDim.x, m = 1ll << mlog;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < K; idx += stride) {
        const long long child = idx >> mlog, j = idx & (m - 1);
        fe v = tile_ld(O + child * 2 * m + j);
        if (tree_full(child ^ 1, mlog, k)) v = fe_add(v, tile_ld(cur + (child >> 1) * 2 * m + m + j));
        tile_st(next + idx, v);
    }
}

__global__ void k_fri_fold(fe *next, const fe *cw, long long half, const fe *xinv, fe s_m, fe inv2_m) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < half; i += stride) {
        const fe t_m = fe_montmul(tile_ldg(xinv + i), s_m);
        tile_st(next + i, fri_fold_one(tile_ld(cw + i), tile_ld(cw + half + i), t_m, inv2_m));
    }
}

// One CTA reduces `chunk` bottom nodes to one node, writing every level to the heap-ordered tree.
// Phase 1: every thread reduces its 2^ipt_log bottom nodes privately (no barrier); phase 2: the
// per-thread digests are reduced through shared memory.  mode 2 is the fused FRI round:
// fold -> leaf digest -> subtree, one pass over the codeword.
// the host waits for the root of every FRI round before it can draw the next challenge: the last CTA
// of a tree writes it straight into mapped host memory, followed (system-scope fence) by a sequence
// number the host spins on - no copy engine, no stream synchronisation on the critical path
__device__ __forceinline__ void merkle_publish_root(const MerkleArgs &a, const uint64_t *root) {
    volatile uint64_t *out = a.root_out;
#pragma unroll
    for (int i = 0; i < 8; i++) out[i] = root[i];
    __threadfence_system();
    out[8] = a.root_seq;
}
// the work of one CTA (`blk` of `nblocks`) on one level-range of one tree; sm = MK_THREADS * 8 words of
// shared memory, s_last = one shared word
__device__ __forceinline__ void merkle_chunk_body(const MerkleArgs &a, const long long blk, const unsigned nblocks,
                                                  uint64_t *sm, int &s_last) {
    const int tid = threadIdx.x;
    const int active = a.chunk >> a.ipt_log;  // threads with a private subtree
    uint64_t d[8];
    if (tid < active) merkle_private(d, a, blk, tid);
    if (a.red_log == 0) {  // the next launch picks the subtree roots up from the tree
        if (a.root_out && tid == 0) merkle_publish_root(a, d);  // (a tree of one leaf)
        return;
    }
    if (tid < active) {
#pragma unroll
        for (int i = 0; i < 8; i++) sm[tid * 8 + i] = d[i];
    }
    __syncthreads();
    // index of thread 0's subtree root; the level above it starts at base >> 1, and so on
    long long base = (a.width + blk * a.chunk) >> a.ipt_log;
    int wl = active / 2, levels = a.red_log, coop_max = a.coop_max;
    for (int pass = 0;; pass++) {
        for (int lvl = 0; lvl < levels; wl >>= 1, lvl++) {
            base >>= 1;
            if (wl > coop_max || wl > MK_THREADS / 4) {  // plenty of nodes: one thread per node
                const bool mine = tid < wl;
                if (mine) merkle_node_digest(d, sm + (2 * tid) * 8, sm + (2 * tid + 1) * 8);
                __syncthreads();
                if (mine) {
                    uint64_t *node = a.tree + (base + tid) * 8;
#pragma unroll
                    for (int i = 0; i < 8; i++) {
                        sm[tid * 8 + i] = d[i];
                        node[i] = d[i];
                    }
                }
            } else {  // few nodes, the level is a dependency chain: four lanes per node (hash.cuh)
                const int q = tid >> 2, j = tid & 3;
                const bool warp_on = (tid >> 5) < ((4 * wl + 31) >> 5);  // whole warps only (shuffles)
                uint64_t lo = 0, hi = 0;
                if (warp_on) blake2b_coop4_node(lo, hi, sm + (2 * (q < wl ? q : 0)) * 8, j);
                __syncthreads();
                if (warp_on && q < wl) {
                    uint64_t *node = a.tree + (base + q) * 8;
                    sm[q * 8 + j] = lo;
                    sm[q * 8 + 4 + j] = hi;
                    node[j] = lo;
                    node[4 + j] = hi;
                }
            }
            __syncthreads();
        }
        if (pass == 1 || a.ticket == nullptr) break;
        // Every CTA has reduced its chunk to one digest (heap node nblocks + blk).  The CTA that
        // arrives last reduces those nblocks digests as well instead of leaving them to one more
        // launch (each thread fences its own stores, the barrier orders them before the ticket).
        __threadfence();
        __syncthreads();
        if (tid == 0) s_last = atomicAdd(a.ticket, 1u) == nblocks - 1;
        __syncthreads();
        if (!s_last) return;
        const int g = (int)nblocks;
        if (tid == 0) *a.ticket = 0;  // as the next launch on this stream expects it
        __threadfence();
        if (tid < g) {
            const uint64_t *node = a.tree + (size_t)(g + tid) * 8;
#pragma unroll
            for (int i = 0; i < 8; i++) sm[tid * 8 + i] = __ldcg(node + i);  // written by other SMs: not via L1
        }
        __syncthreads();
        base = g;
        wl = g / 2;
        levels = 31 - __clz(g);
        coop_max = MK_THREADS / 4;  // this part is a dependency chain whatever the shape below was
    }
    if (a.root_out && tid == 0) merkle_publish_root(a, sm);
}

// At least 2 resident CTAs per SM, so at most 128 registers: without the bound the kernel drifted to 148
// registers in round 2 (one CTA per SM, 2^20-leaf tree 341 -> 383 us)
__global__ void __launch_bounds__(MK_THREADS, 2) k_merkle_chunk(const __grid_constant__ MerkleArgs a) {
    __shared__ uint64_t sm[MK_THREADS * 8];
    __shared__ int s_last;  // after sm: ptxas then places sm at offset 0, which its 128-bit accesses need
    merkle_chunk_body(a, blockIdx.x, gridDim.x, sm, s_last);
}

__global__ void k_merkle_paths(uint64_t *out, const uint64_t *tree, long long n, int depth,
                               const uint64_t *indices, long long k) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = k * depth * 8;
    if (t >= total) return;
    const int w = (int)(t & 7);
    const long long ql = t >> 3;
    const int level = (int)(ql % depth);
    const long long q = ql / depth;
    const long long node = ((n + (long long)indices[q]) >> level) ^ 1;
    out[t] = tree[node * 8 + w];
}
__global__ void k_gather(fe *out, const fe *values, const uint64_t *indices, long long k) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < k) tile_st(out + t, tile_ld(values + indices[t]));
}

// --- self test: PTX carry-chain field ops vs the portable C++ ones -------------------------
__device__ __forceinline__ uint64_t sa_splitmix(uint64_t &s) {
    uint64_t z = (s += 0x9E3779B97F4A7C15ULL);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}
__device__ __forceinline__ fe sa_rand_fe(uint64_t &s, int kind) {
    const uint64_t a = sa_splitmix(s), b = sa_splitmix(s);
    fe r = fe_make((uint32_t)a, (uint32_t)(a >> 32), (uint32_t)b, (uint32_t)(b >> 32));
    switch (kind & 15) {  // edge cases
        case 0: r = fe_zero(); break;
        case 1: r = fe_one(); break;
        case 2: r = fe_make(0, 0, 0, P3); break;                                  // p - 1
        case 3: r = fe_make(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, P3 - 1); break;  // p - 2
        case 4: r.v[3] = P3; r.v[2] = 0; r.v[1] = 0; r.v[0] = 0; break;
        case 5: r.v[0] = 0; break;
        case 6: r.v[0] = 0; r.v[1] = 0; r.v[2] = 0; break;
        default: break;
    }
    // canonicalise: force below p
    if (r.v[3] > P3 || (r.v[3] == P3 && (r.v[2] | r.v[1] | r.v[0]) != 0)) r.v[3] -= P3;
    return r;
}
__global__ void k_selftest_field(unsigned long long *mismatches, long long count, uint64_t seed) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    uint64_t s = seed + 0x1234567ULL * (uint64_t)i;
    const fe a = sa_rand_fe(s, (int)(i % 37)), b = sa_rand_fe(s, (int)((i / 37) % 41));
    int bad = 0;
    bad += !fe_eq(fe_add(a, b), fe_add_portable(a, b));
    bad += !fe_eq(fe_sub(a, b), fe_sub_portable(a, b));
    bad += !fe_eq(fe_montmul(a, b), fe_montmul_portable(a, b));
    if (bad) atomicAdd(mismatches, (unsigned long long)bad);
}

template <int OP, int ILP>
__global__ void k_microbench(fe *sink, int iters) {
    fe x[ILP], y[ILP];
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
#pragma unroll
    for (int i = 0; i < ILP; i++) {
        x[i] = fe_make(t + i, t * 3 + 1, i + 7, 0x12345678u + i);
        y[i] = fe_make(t * 5 + i, t + 11, i + 3, 0x0ABCDEF0u + i);
    }
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < ILP; i++) {
            if (OP == 0) x[i] = fe_montmul(x[i], y[i]);
            if (OP == 1) x[i] = fe_add(x[i], y[i]);
            if (OP == 2) x[i] = fe_sub(x[i], y[i]);
            if (OP == 3) {
                const fe tt = fe_montmul(y[i], x[(i + 1) % ILP]);
                const fe e = x[i];
                x[i] = fe_add(e, tt);
                y[i] = fe_sub(e, tt);
            }
        }
    }
    fe acc = x[0];
#pragma unroll
    for (int i = 1; i < ILP; i++) acc = fe_add(acc, fe_add(x[i], y[i]));
    if (acc.v[0] == 0xDEADBEEFu && acc.v[1] == 0x1u) tile_st(sink + t, acc);
}

// blake2b-only roof of the Merkle kernels: every thread hashes a chain of node messages (128 bytes = one
// compression each, merkle.py:11) that never leave its registers
template <int ILP>
__global__ void __launch_bounds__(MK_THREADS) k_microbench_b2(uint64_t *sink, int iters) {
    uint64_t d[ILP][8];
    const uint64_t t = blockIdx.x * blockDim.x + threadIdx.x;
#pragma unroll
    for (int i = 0; i < ILP; i++)
#pragma unroll
        for (int k = 0; k < 8; k++) d[i][k] = t * 0x9E3779B97F4A7C15ull + 131 * i + k;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < ILP; i++) merkle_node_digest(d[i], d[i], d[(i + 1) % ILP]);
    }
    uint64_t acc = 0;
#pragma unroll
    for (int i = 0; i < ILP; i++)
#pragma unroll
        for (int k = 0; k < 8; k++) acc ^= d[i][k];
    if (acc == 0x1234567ull) sink[t] = acc;
}

// ------------------------------------------------------------- workspaces --
// Grow-only scratch buffers, one per (device, stream): the four-step NTT needs an n*batch
// intermediate and allocating it per call (even stream-ordered) costs more than the kernels.
static std::mutex g_ws_mu;
static std::map<std::tuple<int, cudaStream_t, int>, std::pair<void *, size_t>> g_ws;
static int get_workspace(void **out, size_t bytes, cudaStream_t st, int tag = 0) {
    int dev = 0;
    SA_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_ws_mu);
    auto &slot = g_ws[std::make_tuple(dev, st, tag)];
    if (slot.second < bytes) {
        if (slot.first) {
            SA_CUDA(cudaStreamSynchronize(st));  // earlier work on this stream may still use it
            SA_CUDA(cudaFree(slot.first));
            slot.first = nullptr;
            slot.second = 0;
        }
        SA_CUDA(cudaMalloc(&slot.first, bytes));
        slot.second = bytes;
    }
    *out = slot.first;
    return SA_OK;
}
// stream-ordered pool allocations (small flags, host-entry staging) keep their memory cached
static void keep_pool_memory() {
    static std::once_flag once;
    std::call_once(once, [] {
        int dev = 0;
        cudaMemPool_t pool;
        if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
            uint64_t keep = UINT64_MAX;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    });
}

// ---------------------------------------------------------------- NTT plans --
// Twiddle tables are cached per (device, log n, root, direction); FRI x^-1 tables per (device, omega, n).
// Both live in one LRU bounded by bytes (sa_cache_limit): fast_multiply's order shrinking
// (ntt.py:47-49) and a prover that walks through many domains generate new roots all the time, and
// a 2^20 plan holds a 16 MiB inter-pass matrix.  Entries are handed out as shared_ptr: an evicted
// table is freed when its last user lets go, and cudaFree waits for kernels still reading it.
struct DeviceTables {
    std::vector<void *> ptrs;
    size_t bytes = 0;
    int device = 0;
    int alloc(void **out, size_t nbytes) {
        SA_CUDA(cudaMalloc(out, nbytes));
        ptrs.push_back(*out);
        bytes += nbytes;
        return SA_OK;
    }
    ~DeviceTables() {
        if (ptrs.empty()) return;
        int cur = 0;
        const bool sw = cudaGetDevice(&cur) == cudaSuccess && cur != device && cudaSetDevice(device) == cudaSuccess;
        for (void *p : ptrs) cudaFree(p);
        if (sw) cudaSetDevice(cur);
        cudaGetLastError();
    }
};
struct NttPlan : DeviceTables {
    int log_n = 0, l1 = 0, l2 = 0, l3 = 0;
    fe *tw1 = nullptr, *tw2 = nullptr, *tw3 = nullptr, *twb = nullptr, *twb2 = nullptr;
    fe cst1[8], cst2[8], cst3[8];
    fe scale_m;     // n^-1 (Montgomery) for single-tile inverse transforms
    int has_scale = 0;
};
struct XinvTable : DeviceTables {
    fe *tab = nullptr;
};
using PlanPtr = std::shared_ptr<NttPlan>;
using XinvPtr = std::shared_ptr<XinvTable>;
// kind (0 plan, 1 xinv), device, log_n | n, root lo, root hi, inverse
using CacheKey = std::tuple<int, int, uint64_t, uint64_t, uint64_t, int>;
struct CacheEntry {
    std::shared_ptr<DeviceTables> tables;
    uint64_t tick = 0;
};
static std::mutex g_plan_mu;
static std::map<CacheKey, CacheEntry> g_cache;
static size_t g_cache_bytes = 0;
static size_t g_cache_limit = (size_t)4 << 30;  // bytes; SA_CACHE_LIMIT_MIB / sa_cache_limit()
static uint64_t g_cache_tick = 0;

static void cache_config() {
    static std::once_flag once;
    std::call_once(once, [] {
        if (const char *e = getenv("SA_CACHE_LIMIT_MIB")) {
            const long long v = atoll(e);
            if (v >= 0) g_cache_limit = (size_t)v << 20;
        }
    });
}
// g_plan_mu held.  Drops least-recently-used entries until `incoming` more bytes fit (an entry larger
// than the whole limit is still admitted alone: the call that needs it has to run).
static void cache_make_room(size_t incoming) {
    while (!g_cache.empty() && g_cache_bytes + incoming > g_cache_limit) {
        auto victim = g_cache.begin();
        for (auto it = g_cache.begin(); it != g_cache.end(); ++it)
            if (it->second.tick < victim->second.tick) victim = it;
        g_cache_bytes -= victim->second.tables->bytes;
        g_cache.erase(victim);  // frees the device memory once nobody holds the tables any more
    }
}
template <class T>
static std::shared_ptr<T> cache_find(const CacheKey &key) {
    cache_config();
    std::lock_guard<std::mutex> lock(g_plan_mu);
    auto it = g_cache.find(key);
    if (it == g_cache.end()) return nullptr;
    it->second.tick = ++g_cache_tick;
    return std::static_pointer_cast<T>(it->second.tables);
}
// publishes `made` unless another thread got there first (then that one wins and `made` is dropped)
template <class T>
static std::shared_ptr<T> cache_publish(const CacheKey &key, std::shared_ptr<T> made) {
    std::lock_guard<std::mutex> lock(g_plan_mu);
    auto it = g_cache.find(key);
    if (it != g_cache.end()) {
        it->second.tick = ++g_cache_tick;
        return std::static_pointer_cast<T>(it->second.tables);
    }
    cache_make_room(made->bytes);
    CacheEntry e;
    e.tables = made;
    e.tick = ++g_cache_tick;
    g_cache.emplace(key, e);
    g_cache_bytes += made->bytes;
    return made;
}

static int build_pow_table(DeviceTables &owner, fe **out, const fe &base_m, const fe &lead_m, long long count,
                           cudaStream_t st, int swz = 0) {
    int rc = owner.alloc((void **)out, sizeof(fe) * (size_t)count);
    if (rc != SA_OK) return rc;
    const long long threads = (count + 15) / 16;
    const int bs = 128;
    k_pow_table<<<(unsigned)((threads + bs - 1) / bs), bs, 0, st>>>(*out, base_m, lead_m, count, swz);
    SA_LAUNCH_CHECK();
    return SA_OK;
}

// validates the root like ntt.py:10-11 and returns (creating if needed) the plan.  Tables are built
// outside the cache lock; a failed build frees what it had allocated (the plan object owns them).
static int get_plan(PlanPtr *plan_out, int log_n, const fe &root, int inverse, cudaStream_t st) {
    int dev = 0;
    SA_CUDA(cudaGetDevice(&dev));
    const uint64_t rlo = (uint64_t)root.v[0] | ((uint64_t)root.v[1] << 32);
    const uint64_t rhi = (uint64_t)root.v[2] | ((uint64_t)root.v[3] << 32);
    const CacheKey key(0, dev, (uint64_t)log_n, rlo, rhi, inverse ? 1 : 0);
    if ((*plan_out = cache_find<NttPlan>(key))) return SA_OK;
    const uint64_t n = 1ull << log_n;
    const fe root_m = fe_to_mont(root);
    if (!fe_eq(fe_mont_pow_u64(root_m, n), fe_mont_one())) return SA_EROOTORDER;
    if (fe_eq(fe_mont_pow_u64(root_m, n / 2), fe_mont_one())) return SA_ENOTPRIM;
    // the transform root: root itself, or root^-1 for intt (ntt.py:29)
    const fe w_m = inverse ? fe_mont_inv(root_m) : root_m;
    const fe ninv_m = fe_mont_inv(fe_to_mont(fe_from_u64(n)));  // ntt.py:27
    PlanPtr made = std::make_shared<NttPlan>();
    NttPlan &p = *made;
    p.device = dev;
    p.log_n = log_n;
    int rc;
    const NttShape shape = ntt_shape(log_n);
    p.l1 = shape.l1;
    p.l2 = shape.l2;
    p.l3 = shape.l3;
    if (shape.l3 > 0) {
        const int n1 = 1 << p.l1, n2 = 1 << p.l2, n3 = 1 << p.l3;
        const long long m = (long long)n2 * n3;
        const fe w1_m = fe_mont_pow_u64(w_m, (uint64_t)m);     // n1-point transforms over j1
        const fe wsub_m = fe_mont_pow_u64(w_m, (uint64_t)n1);  // root of the length-m sub-transforms
        const fe w2_m = fe_mont_pow_u64(wsub_m, (uint64_t)n3);
        const fe w3_m = fe_mont_pow_u64(wsub_m, (uint64_t)n2);
        if ((rc = build_pow_table(p, &p.tw1, w1_m, fe_mont_one(), n1, st, 1)) != SA_OK) return rc;
        if ((rc = build_pow_table(p, &p.tw2, w2_m, fe_mont_one(), n2, st, 1)) != SA_OK) return rc;
        if ((rc = build_pow_table(p, &p.tw3, w3_m, fe_mont_one(), n3, st, 1)) != SA_OK) return rc;
        ntt_fill_cst(p.cst1, w1_m, n1);
        ntt_fill_cst(p.cst2, w2_m, n2);
        ntt_fill_cst(p.cst3, w3_m, n3);
        if ((rc = p.alloc((void **)&p.twb, sizeof(fe) * (size_t)n)) != SA_OK) return rc;
        if ((rc = p.alloc((void **)&p.twb2, sizeof(fe) * (size_t)m)) != SA_OK) return rc;
        const int bs = 128;
        long long threads = (long long)n1 * ((m + 15) / 16);
        k_twb_table<<<(unsigned)((threads + bs - 1) / bs), bs, 0, st>>>(p.twb, w_m, inverse ? ninv_m : fe_mont_one(),
                                                                      n1, (int)m);
        SA_LAUNCH_CHECK();
        threads = (long long)n2 * ((n3 + 15) / 16);
        k_twb_table<<<(unsigned)((threads + bs - 1) / bs), bs, 0, st>>>(p.twb2, wsub_m, fe_mont_one(), n2, n3);
        SA_LAUNCH_CHECK();
    } else if (log_n <= 10) {
        if ((rc = build_pow_table(p, &p.tw1, w_m, fe_mont_one(), (long long)n, st, 1)) != SA_OK) return rc;
        ntt_fill_cst(p.cst1, w_m, (int)n);
        p.has_scale = inverse ? 1 : 0;
        p.scale_m = inverse ? ninv_m : fe_mont_one();
    } else {
        const int n1 = 1 << p.l1, n2 = 1 << p.l2;
        const fe w1_m = fe_mont_pow_u64(w_m, (uint64_t)n2);  // root of the length-n1 column transforms
        const fe w2_m = fe_mont_pow_u64(w_m, (uint64_t)n1);  // root of the length-n2 row transforms
        if ((rc = build_pow_table(p, &p.tw1, w1_m, fe_mont_one(), n1, st, 1)) != SA_OK) return rc;
        if ((rc = build_pow_table(p, &p.tw2, w2_m, fe_mont_one(), n2, st, 1)) != SA_OK) return rc;
        ntt_fill_cst(p.cst1, w1_m, n1);
        ntt_fill_cst(p.cst2, w2_m, n2);
        if ((rc = p.alloc((void **)&p.twb, sizeof(fe) * (size_t)n)) != SA_OK) return rc;
        const long long threads = (long long)n1 * ((n2 + 15) / 16);
        const int bs = 128;
        k_twb_table<<<(unsigned)((threads + bs - 1) / bs), bs, 0, st>>>(
            p.twb, w_m, inverse ? ninv_m : fe_mont_one(), n1, n2);
        SA_LAUNCH_CHECK();
    }
    // the tables were built on `st`; other streams may pick the plan up from the cache right away,
    // so they must be complete before it is published (one-time cost per plan)
    SA_CUDA(cudaStreamSynchronize(st));
    *plan_out = cache_publish<NttPlan>(key, made);
    return SA_OK;
}

// kernels with more than 48 KB of dynamic shared memory need the opt-in once per (kernel, device)
constexpr int SA_MAX_DEVICES = 64;
template <class K>
static int optin_smem(K kernel, std::atomic<bool> *done, size_t smem) {
    int dev = 0;
    SA_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= SA_MAX_DEVICES || !done[dev].load(std::memory_order_acquire)) {
        SA_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        if (dev >= 0 && dev < SA_MAX_DEVICES) done[dev].store(true, std::memory_order_release);
    }
    return SA_OK;
}

template <int LOGL, int ELOG, int C, int FLAGS>
static int launch_tile_variant(const TileArgs &a, cudaStream_t st) {
    using P = TilePlan<LOGL, ELOG, C>;
    const int tiles_per_batch = (a.ncols + C - 1) / C;
    const long long total = (long long)tiles_per_batch * a.nbatch;
    const long long grid = (total + P::TPC - 1) / P::TPC;
    const size_t smem = P::smem_bytes();
    if (smem > 48 * 1024) {
        static std::atomic<bool> attr_done[SA_MAX_DEVICES];
        const int rc = optin_smem(ntt_tile_kernel<LOGL, ELOG, C, FLAGS>, attr_done, smem);
        if (rc != SA_OK) return rc;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(P::THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const int tpb = tiles_per_batch;
    SA_CUDA(cudaLaunchKernelEx(&cfg, ntt_tile_kernel<LOGL, ELOG, C, FLAGS>, a, total, tpb));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return SA_OK;
}
template <int LOGL, int ELOG, int C>
static int launch_tile(const TileArgs &a, cudaStream_t st) {
    const int variant = tile_variant<LOGL, ELOG, C>(a);
    if constexpr (LOGL >= 5) {
        switch (variant) {
            case TF_FULL | TF_TWB: return launch_tile_variant<LOGL, ELOG, C, TF_FULL | TF_TWB>(a, st);
            case TF_FULL: return launch_tile_variant<LOGL, ELOG, C, TF_FULL>(a, st);
            case TF_FULL | TF_PEERS: return launch_tile_variant<LOGL, ELOG, C, TF_FULL | TF_PEERS>(a, st);
        }
    }
    if (variant & TF_PEERS) return launch_tile_variant<LOGL, ELOG, C, TF_DYNAMIC | TF_PEERS>(a, st);
    return launch_tile_variant<LOGL, ELOG, C, TF_DYNAMIC>(a, st);
}

// tile shape: register block (log2 elements per thread) and columns per tile; with -DSA_TUNE
// the environment variables SA_NTT_ELOG / SA_NTT_C select a shape for tuning runs.
#ifdef SA_TUNE
static int g_tile_elog = -1, g_tile_c = -1;
static void tile_config() {
    if (g_tile_elog >= 0) return;
    const char *e = getenv("SA_NTT_ELOG"), *c = getenv("SA_NTT_C");
    g_tile_elog = e ? atoi(e) : 0;
    g_tile_c = c ? atoi(c) : 0;
}
#endif
template <int LOGL>
static int launch_tile_shape(const TileArgs &a, cudaStream_t st) {
#ifdef SA_TUNE
    tile_config();
    if (LOGL >= 9 && g_tile_elog > 0) {
        if (g_tile_elog == 3 && g_tile_c == 8) return launch_tile<LOGL, 3, 8>(a, st);
        if (g_tile_elog == 3 && g_tile_c == 4) return launch_tile<LOGL, 3, 4>(a, st);
        if (g_tile_elog == 3 && g_tile_c == 2) return launch_tile<LOGL, 3, 2>(a, st);
        if (g_tile_elog == 4 && g_tile_c == 4) return launch_tile<LOGL, 4, 4>(a, st);
        if (g_tile_elog == 4 && g_tile_c == 2) return launch_tile<LOGL, 4, 2>(a, st);
        if (g_tile_elog == 4 && g_tile_c == 8) return launch_tile<LOGL, 4, 8>(a, st);
    }
#endif
    // measured on B200 (profiles/r01_notes.md, r01e_tile_shapes_tma_twiddles.jsonl): with the stage
    // twiddles in shared memory, 16-element register blocks on 4-column tiles (2 CTAs x 256 threads
    // per SM) win for the big tiles
    if constexpr (LOGL >= 9) {
        // multi-GPU assembly (sa_ntt_multi): 8-column tiles store 128-byte instead of 64-byte segments to the
        // peers - the pass is bound by NVLink, not by the butterflies (8 GPUs, 16 x 2^20 incl. assembly: 0.468 ms
        // against 0.665 ms with 4-column tiles, profiles/r02_notes.md)
        if (a.npeer > 0 || a.mc_out != nullptr) return launch_tile<LOGL, 4, 8>(a, st);
        // (a LONE 2^20 transform is one partial wave per pass: 256 tiles on 2 x 148 slots, 108 SMs carry 8 columns
        // and 40 carry 4.  Seven-column tiles - 147 CTAs of 448 threads, one per SM, every SM the same 7 columns -
        // were built, emulated bit-exact and measured: 70 us against 60 us.  One 14-warp CTA per SM whose warps
        // all sit in the same phase loses more than the balance gains; profiles/r02q_lone_tiles.jsonl.  So was a grid
        // of exactly two CTAs per SM, 136 four-column and 160 three-column tiles in one launch (no SM above 7
        // columns): 64.6 us against 58.7 us, profiles/r02v_lone_mix.jsonl - a lone pass is bound by the latency of a
        // tile's own dependent phases, not by the busiest SM's column count.)
        return launch_tile<LOGL, 4, 4>(a, st);
    }
    return launch_tile<LOGL, 4, 8>(a, st);
}
static int launch_tile_dyn(int logl, const TileArgs &a, cudaStream_t st) {
    switch (logl) {
        case 1: return launch_tile_shape<1>(a, st);
        case 2: return launch_tile_shape<2>(a, st);
        case 3: return launch_tile_shape<3>(a, st);
        case 4: return launch_tile_shape<4>(a, st);
        case 5: return launch_tile_shape<5>(a, st);
        case 6: return launch_tile_shape<6>(a, st);
        case 7: return launch_tile_shape<7>(a, st);
        case 8: return launch_tile_shape<8>(a, st);
        case 9: return launch_tile_shape<9>(a, st);
        case 10: return launch_tile_shape<10>(a, st);
    }
    return SA_ESIZE;
}

// ------------------------------------------------------------------- C ABI --
extern "C" {

const char *sa_version(void) { return "sa_b200 0.1 sm_100a"; }
const char *sa_last_error(void) { return g_last_error.c_str(); }
uint64_t sa_launch_count(void) { return g_launches.load(); }

}  // extern "C"

// the transform proper; `peers` (npeer <= TILE_MAX_PEERS) are extra destinations of the LAST pass: the
// same element offsets as `out`, in other GPUs' memory (sa_ntt_multi)
static int ntt_run(void *out, const void *in, int log_n, const uint64_t root[2], int inverse, size_t batch,
                   cudaStream_t st, fe *const *peers, int npeer, fe *mc = nullptr) {
    if (log_n < 0 || log_n > NTT_MAX_LOG_N) return SA_ESIZE;
    if (batch == 0) return SA_OK;
    const size_t n = size_t(1) << log_n;
    if (log_n == 0) {  // ntt.py:5-6 / :23-24: a length-1 sequence is returned as is
        if (out != in) SA_CUDA(cudaMemcpyAsync(out, in, 16 * batch, cudaMemcpyDeviceToDevice, st));
        for (int i = 0; i < npeer; i++)
            SA_CUDA(cudaMemcpyAsync(peers[i], in, 16 * batch, cudaMemcpyDeviceToDevice, st));
        if (mc) return SA_ESIZE;  // (no kernel runs for length-1 transforms: not offered through a multicast address)
        return SA_OK;
    }
    PlanPtr p;  // keeps the tables alive until the launches below are enqueued (cudaFree waits for them)
    int rc = get_plan(&p, log_n, fe_from_limbs(root), inverse, st);
    if (rc != SA_OK) return rc;
    TileArgs a;
    memset(&a, 0, sizeof(a));
    auto with_peers = [&](TileArgs &t) {
        t.npeer = npeer;
        for (int i = 0; i < npeer; i++) t.peer_out[i] = peers[i];
        t.mc_out = mc;
    };
    if (log_n <= 10) {
        // every transform is one tile column; in-place is safe because a tile reads all of
        // its columns into registers before it writes any of them
        if (batch > (size_t)1 << 30) return SA_ESIZE;
        ntt_fill_single(a, (const fe *)in, (fe *)out, log_n, batch, p->tw1, p->cst1, p->has_scale, p->scale_m);
        with_peers(a);
        return launch_tile_dyn(log_n, a, st);
    }
    NttShape shape;
    shape.log_n = log_n;
    shape.l1 = p->l1;
    shape.l2 = p->l2;
    shape.l3 = p->l3;
    fe *tmp = nullptr;
    if ((rc = get_workspace((void **)&tmp, sizeof(fe) * n * batch, st)) != SA_OK) return rc;
    if (shape.l3 > 0) {
        if (batch * ((size_t)1 << (p->l1 > p->l2 ? p->l1 : p->l2)) > ((size_t)1 << 30)) return SA_ESIZE;
        // `out` doubles as the first intermediate (tiles read before they write: in == out is fine)
        ntt_fill_3pass_a(a, (const fe *)in, (fe *)out, shape, batch, p->tw1, p->twb, p->cst1);
        if ((rc = launch_tile_dyn(p->l1, a, st)) != SA_OK) return rc;
        ntt_fill_3pass_b(a, (const fe *)out, tmp, shape, batch, p->tw2, p->twb2, p->cst2);
        if ((rc = launch_tile_dyn(p->l2, a, st)) != SA_OK) return rc;
        ntt_fill_3pass_c(a, tmp, (fe *)out, shape, batch, p->tw3, p->cst3);
        with_peers(a);
        return launch_tile_dyn(p->l3, a, st);
    }
    ntt_fill_pass1(a, (const fe *)in, tmp, shape, batch, p->tw1, p->twb, p->cst1);
    rc = launch_tile_dyn(p->l1, a, st);
    if (rc == SA_OK) {
        ntt_fill_pass2(a, tmp, (fe *)out, shape, batch, p->tw2, p->cst2);
        with_peers(a);
        rc = launch_tile_dyn(p->l2, a, st);
    }
    return rc;
}

extern "C" {

int sa_ntt(void *out, const void *in, int log_n, const uint64_t root[2], int inverse, size_t batch,
           void *stream) {
    return ntt_run(out, in, log_n, root, inverse, batch, (cudaStream_t)stream, nullptr, 0);
}

// ---- buffers shared between the processes of one box (one process per GPU) ----
int sa_peer_alloc(void **ptr, size_t bytes, uint8_t handle_out[64]) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handles are 64 bytes");
    *ptr = nullptr;
    SA_CUDA(cudaMalloc(ptr, bytes ? bytes : 1));  // (IPC needs a cudaMalloc allocation of its own, not a pool block)
    SA_CUDA(cudaMemset(*ptr, 0, bytes ? bytes : 1));
    cudaIpcMemHandle_t h;
    const cudaError_t e = cudaIpcGetMemHandle(&h, *ptr);
    if (e != cudaSuccess) {
        cudaFree(*ptr);
        *ptr = nullptr;
        SA_CUDA(e);
    }
    memcpy(handle_out, &h, 64);
    return SA_OK;
}
int sa_peer_open(void **ptr, const uint8_t handle[64]) {
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    *ptr = nullptr;
    // opened with THIS device current: the mapping lands in this device's address space and peer access to
    // the owner is enabled on the way, which is what lets this device's kernels store into it
    SA_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return SA_OK;
}
int sa_peer_close(void *ptr) {
    if (ptr) SA_CUDA(cudaIpcCloseMemHandle(ptr));
    return SA_OK;
}
int sa_peer_free(void *ptr) {
    if (ptr) SA_CUDA(cudaFree(ptr));
    return SA_OK;
}
int sa_copy_async(void *dst, const void *src, size_t bytes, void *stream) {
    if (bytes) SA_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, (cudaStream_t)stream));
    return SA_OK;
}

int sa_ntt_mcast(void *mc, void *local, size_t out_offset, const void *in, int log_n, const uint64_t root[2],
                 int inverse, size_t batch, void *stream) {
    if (!mc || !local) return SA_ESIZE;
    return ntt_run((fe *)local + out_offset, in, log_n, root, inverse, batch, (cudaStream_t)stream, nullptr, 0,
                   (fe *)mc + out_offset);
}

int sa_push(void *const *dsts, int ndst, const void *src, size_t bytes, void *stream) {
    if (ndst < 0 || ndst > TILE_MAX_PEERS || (bytes & 15) || (((uintptr_t)src) & 15)) return SA_ESIZE;
    if (ndst == 0 || bytes == 0) return SA_OK;
    PushArgs a;
    memset(&a, 0, sizeof(a));
    a.ndst = ndst;
    for (int i = 0; i < ndst; i++) {
        if (((uintptr_t)dsts[i]) & 15) return SA_ESIZE;
        a.dst[i] = (uint4 *)dsts[i];
    }
    static const int ctas = [] {
        const char *e = getenv("SA_PUSH_CTAS");
        return e && atoi(e) > 0 ? atoi(e) : 148;
    }();
    const size_t n16 = bytes / 16;
    size_t grid = (n16 + 255) / 256;
    if (grid > (size_t)ctas) grid = (size_t)ctas;
    k_push<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(a, (const uint4 *)src, n16);
    SA_LAUNCH_CHECK();
    return SA_OK;
}

int sa_push_mcast(void *mc_dst, const void *src, size_t bytes, void *stream) {
    if (!mc_dst || (bytes & 15) || (((uintptr_t)src) & 15) || (((uintptr_t)mc_dst) & 15)) return SA_ESIZE;
    if (bytes == 0) return SA_OK;
    static const int ctas = [] {
        const char *e = getenv("SA_PUSH_CTAS");
        return e && atoi(e) > 0 ? atoi(e) : 148;
    }();
    const size_t n16 = bytes / 16;
    size_t grid = (n16 + 255) / 256;
    if (grid > (size_t)ctas) grid = (size_t)ctas;
    k_push_mcast<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>((fe *)mc_dst, (const fe *)src, n16);
    SA_LAUNCH_CHECK();
    return SA_OK;
}

int sa_enable_peer_access(int peer_device) {
    int dev = 0;
    SA_CUDA(cudaGetDevice(&dev));
    if (peer_device == dev) return SA_OK;
    int can = 0;
    SA_CUDA(cudaDeviceCanAccessPeer(&can, dev, peer_device));
    if (!can) {
        g_last_error = "sa_enable_peer_access: no peer access between these devices";
        return SA_ECUDA;
    }
    const cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) {
        cudaGetLastError();
        return SA_OK;
    }
    SA_CUDA(e);
    return SA_OK;
}

int sa_ntt_multi(void *const *outs, int nouts, size_t out_offset, const void *in, int log_n,
                 const uint64_t root[2], int inverse, size_t batch, void *stream) {
    if (nouts < 1 || nouts > TILE_MAX_PEERS + 1) return SA_ESIZE;
    fe *peers[TILE_MAX_PEERS];
    for (int i = 1; i < nouts; i++) peers[i - 1] = (fe *)outs[i] + out_offset;
    return ntt_run((fe *)outs[0] + out_offset, in, log_n, root, inverse, batch, (cudaStream_t)stream, peers,
                   nouts - 1);
}

// Host entry: H2D, transforms, D2H.  Batches are cut into chunks of a few transforms that rotate over
// a few internal streams so that the upload of chunk i+1, the kernels of chunk i and the download
// of chunk i-1 overlap (PCIe is full duplex); with pinned host buffers the call is bound by the
// slower copy direction instead of the sum of both.
constexpr int HOST_STREAMS_MAX = 8;
// one set of copy streams (and of the device buffers that go with them) per device; a set is used by
// one sa_ntt_host call at a time - the link is the shared resource anyway
struct CopySet {
    cudaStream_t streams[HOST_STREAMS_MAX];
    cudaEvent_t events[HOST_STREAMS_MAX + 1];
    std::mutex busy;
};
static std::map<int, CopySet *> g_copy_sets;
static std::mutex g_copy_mu;
static int g_host_streams = 4;            // SA_HOST_STREAMS
static size_t g_host_chunk = 32u << 20;   // SA_HOST_CHUNK_MIB: bytes per pipelined chunk
static int g_host_ramp = 1;               // SA_HOST_RAMP: first/last chunks start at chunk >> ramp
// (measured, profiles/r01g_e2e_pipeline_sweep.txt: 4 streams x 32 MiB with a one-step ramp 6.35 ms per
//  16 x 2^20 call, 3 x 16 MiB flat 6.48-6.58 ms; the link does 49.6 GB/s each way on monolithic copies)
static int get_copy_set(CopySet **out) {
    int dev = 0;
    SA_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_copy_mu);
    auto it = g_copy_sets.find(dev);
    if (it != g_copy_sets.end()) {
        *out = it->second;
        return SA_OK;
    }
    static bool configured = false;
    if (!configured) {
        configured = true;
        if (const char *e = getenv("SA_HOST_STREAMS")) {
            const int v = atoi(e);
            if (v >= 1 && v <= HOST_STREAMS_MAX) g_host_streams = v;
        }
        if (const char *e = getenv("SA_HOST_CHUNK_MIB")) {
            const int v = atoi(e);
            if (v >= 1 && v <= 1024) g_host_chunk = (size_t)v << 20;
        }
        if (const char *e = getenv("SA_HOST_RAMP")) {
            const int v = atoi(e);
            if (v >= 0 && v <= 6) g_host_ramp = v;
        }
    }
    CopySet *set = new CopySet();
    for (int i = 0; i < g_host_streams; i++)
        SA_CUDA(cudaStreamCreateWithFlags(&set->streams[i], cudaStreamNonBlocking));
    for (int i = 0; i <= g_host_streams; i++)
        SA_CUDA(cudaEventCreateWithFlags(&set->events[i], cudaEventDisableTiming));
    g_copy_sets[dev] = set;
    *out = set;
    return SA_OK;
}

int sa_ntt_host(void *out_host, const void *in_host, int log_n, const uint64_t root[2], int inverse,
                size_t batch, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (log_n < 0 || log_n > NTT_MAX_LOG_N) return SA_ESIZE;
    const size_t one = size_t(16) << log_n;
    const size_t bytes = one * batch;
    if (bytes == 0) return SA_OK;
    int rc;
    CopySet *cset = nullptr;
    if ((rc = get_copy_set(&cset)) != SA_OK) return rc;
    // chunk = as many transforms as fit g_host_chunk (default two 2^20 transforms); small jobs stay on `st`
    size_t per_chunk = one >= g_host_chunk ? 1 : g_host_chunk / one;
    if (per_chunk > batch) per_chunk = batch;
    const size_t nchunks = (batch + per_chunk - 1) / per_chunk;
    if (nchunks < 2) {
        void *dev = nullptr;
        if ((rc = get_workspace(&dev, bytes, st, 1)) != SA_OK) return rc;
        SA_CUDA(cudaMemcpyAsync(dev, in_host, bytes, cudaMemcpyHostToDevice, st));
        rc = sa_ntt(dev, dev, log_n, root, inverse, batch, stream);
        if (rc == SA_OK) SA_CUDA(cudaMemcpyAsync(out_host, dev, bytes, cudaMemcpyDeviceToHost, st));
        SA_CUDA(cudaStreamSynchronize(st));
        return rc;
    }
    const int ns = g_host_streams;
    std::lock_guard<std::mutex> one_call_at_a_time(cset->busy);
    cudaStream_t *g_copy_streams = cset->streams;
    cudaEvent_t *g_copy_events = cset->events;
    // chunk sizes (in transforms): ramp up from a small first chunk and down to a small last one, so
    // that the stretch where only one copy direction is busy (before the first kernel can start, after
    // the last one has finished) is short while the bulk moves in few large copies
    std::vector<size_t> counts;
    {
        std::vector<size_t> head;
        // (per_chunk <= 1 has nothing to ramp; the start is clamped so that c <<= 1 always makes progress)
        if (g_host_ramp && per_chunk > 1)
            for (size_t c = std::max<size_t>(1, per_chunk >> g_host_ramp); c < per_chunk; c <<= 1) head.push_back(c);
        size_t ramp = 0;
        for (size_t c : head) ramp += c;
        if (2 * ramp >= batch) head.clear(), ramp = 0;
        counts = head;
        for (size_t left = batch - 2 * ramp; left > 0;) {
            const size_t c = left < per_chunk ? left : per_chunk;
            counts.push_back(c);
            left -= c;
        }
        counts.insert(counts.end(), head.rbegin(), head.rend());
    }
    void *buf[HOST_STREAMS_MAX];
    for (int i = 0; i < ns; i++)
        if ((rc = get_workspace(&buf[i], per_chunk * one, g_copy_streams[i], 1)) != SA_OK) return rc;
    SA_CUDA(cudaEventRecord(g_copy_events[ns], st));
    for (int i = 0; i < ns; i++) SA_CUDA(cudaStreamWaitEvent(g_copy_streams[i], g_copy_events[ns], 0));
    rc = SA_OK;
    size_t first = 0;
    for (size_t c = 0; c < counts.size() && rc == SA_OK; c++) {
        const int si = (int)(c % ns);
        cudaStream_t cs = g_copy_streams[si];
        const size_t cnt = counts[c];
        const char *src = (const char *)in_host + first * one;
        char *dst = (char *)out_host + first * one;
        first += cnt;
        // within one stream the copies and kernels of successive chunks are ordered, so one device
        // buffer per stream is enough; different streams overlap upload, kernels and download
        SA_CUDA(cudaMemcpyAsync(buf[si], src, cnt * one, cudaMemcpyHostToDevice, cs));
#ifdef SA_TUNE
        static const bool skip_ntt = getenv("SA_HOST_SKIP_NTT") != nullptr;  // copy pipeline alone (diagnostic)
        if (!skip_ntt)
#endif
        rc = sa_ntt(buf[si], buf[si], log_n, root, inverse, cnt, (void *)cs);
        if (rc == SA_OK) SA_CUDA(cudaMemcpyAsync(dst, buf[si], cnt * one, cudaMemcpyDeviceToHost, cs));
    }
    for (int i = 0; i < ns; i++) {
        SA_CUDA(cudaEventRecord(g_copy_events[i], g_copy_streams[i]));
        SA_CUDA(cudaStreamWaitEvent(st, g_copy_events[i], 0));
    }
    SA_CUDA(cudaStreamSynchronize(st));
    return rc;
}

// ---- pinned host buffers next to the GPU ----
static bool gpu_local_cpus(cpu_set_t *set) {
    int dev = 0;
    char bdf[32] = {0};
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetPCIBusId(bdf, sizeof(bdf), dev) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    for (char *c = bdf; *c; c++) *c = (char)tolower((unsigned char)*c);
    const std::string path = std::string("/sys/bus/pci/devices/") + bdf + "/local_cpulist";
    FILE *f = fopen(path.c_str(), "r");
    if (!f) return false;
    char text[4096] = {0};
    const size_t got = fread(text, 1, sizeof(text) - 1, f);
    fclose(f);
    if (got == 0) return false;
    CPU_ZERO(set);
    int count = 0;
    for (char *tok = strtok(text, ",\n"); tok; tok = strtok(nullptr, ",\n")) {  // "0-31,64-95"
        int a = 0, b = 0;
        const int k = sscanf(tok, "%d-%d", &a, &b);
        if (k < 1) continue;
        if (k == 1) b = a;
        for (int c = a; c <= b && c < CPU_SETSIZE; c++, count++) CPU_SET(c, set);
    }
    return count > 0;
}

void *sa_host_alloc(size_t bytes) {
    if (bytes == 0) bytes = 1;
    cpu_set_t before, near, both;
    const bool have_before = pthread_getaffinity_np(pthread_self(), sizeof(before), &before) == 0;
    bool moved = false;
    if (have_before && gpu_local_cpus(&near)) {
        CPU_AND(&both, &before, &near);
        if (CPU_COUNT(&both) > 0) moved = pthread_setaffinity_np(pthread_self(), sizeof(both), &both) == 0;
    }
    void *p = nullptr;
    const cudaError_t e = cudaHostAlloc(&p, bytes, cudaHostAllocPortable);  // pages are placed now, here
    if (e == cudaSuccess) memset(p, 0, bytes);
    if (moved) pthread_setaffinity_np(pthread_self(), sizeof(before), &before);
    if (e != cudaSuccess) {
        g_last_error = std::string("sa_host_alloc: ") + cudaGetErrorString(e);
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

int sa_host_free(void *p) {
    if (p) SA_CUDA(cudaFreeHost(p));
    return SA_OK;
}

static inline unsigned grid_for(long long n, int bs, long long cap = 148 * 16) {
    long long g = (n + bs - 1) / bs;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (unsigned)g;
}

int sa_pointwise_mul(void *out, const void *a, const void *b, size_t n, void *stream) {
    if (n == 0) return SA_OK;
    k_pointwise_mul<<<grid_for((long long)n, 256), 256, 0, (cudaStream_t)stream>>>((fe *)out, (const fe *)a,
                                                                                   (const fe *)b, (long long)n);
    SA_LAUNCH_CHECK();
    return SA_OK;
}

int sa_pointwise_div(void *out, const void *a, const void *b, size_t n, void *stream) {
    if (n == 0) return SA_OK;
    cudaStream_t st = (cudaStream_t)stream;
    int *flag = nullptr;
    keep_pool_memory();
    SA_CUDA(cudaMallocAsync((void **)&flag, sizeof(int), st));
    SA_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), st));
    k_pointwise_div<<<grid_for(((long long)n + 7) / 8, 128), 128, 0, st>>>((fe *)out, (const fe *)a,
                                                                          (const fe *)b, (long long)n, flag);
    SA_LAUNCH_CHECK();
    int h = 0;
    SA_CUDA(cudaMemcpyAsync(&h, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
    SA_CUDA(cudaStreamSynchronize(st));
    cudaFreeAsync(flag, st);
    return h ? SA_EDIVZERO : SA_OK;
}

int sa_scale(void *out, const void *in, size_t n, const uint64_t factor[2], void *stream) {
    if (n == 0) return SA_OK;
    const int bs = 256;
    const unsigned grid = grid_for((long long)n, bs, 148 * 4);
    const fe f_m = fe_to_mont(fe_from_limbs(factor));
    const fe fT_m = fe_mont_pow_u64(f_m, (uint64_t)grid * bs);
    k_scale<<<grid, bs, 0, (cudaStream_t)stream>>>((fe *)out, (const fe *)in, (long long)n, f_m, fT_m);
    SA_LAUNCH_CHECK();
    return SA_OK;
}

static int poly_eval_horner(void *out, const void *coeffs, size_t ncoef, const void *points, size_t npoints,
                            void *stream) {
    if (npoints == 0) return SA_OK;
    const int bs = 64;
    k_poly_eval<<<(unsigned)((npoints + bs - 1) / bs), bs, 0, (cudaStream_t)stream>>>(
        (fe *)out, (const fe *)coeffs, (long long)ncoef, (const fe *)points, (long long)npoints);
    SA_LAUNCH_CHECK();
    return SA_OK;
}

}  // extern "C"

// ---- subproduct tree on the device (see the kernels above) ----
constexpr int TREE_MAX_LOG = 20;  // 2^20 points: ~1 GiB of tree, transforms and scratch
static int g_zf_direct_max = 512;       // up to here the one-CTA sweep kernel (SA_ZF_DIRECT_MAX with -DSA_TUNE)
static int g_interp_direct_max = 1024;  // up to here the k x k Lagrange kernels (SA_INTERP_DIRECT_MAX)
// Horner (one thread per point, ncoef * npoints products) up to this many products, the transposed tree walk above
// (SA_EVAL_TREE_MIN_LOG = log2 of the product count with -DSA_TUNE).  Measured (profiles/r02p_poly_sweep.jsonl, square
// jobs): 4096 points Horner 0.50 ms / walk 1.08 ms, 16384 points 2.01 / 1.36 ms, 65536 points 18.9 / 1.80 ms.
static double g_eval_tree_min = 189812531.0;  // 2^27.5
static void tree_config() {
#ifdef SA_TUNE
    static std::once_flag once;
    std::call_once(once, [] {
        if (const char *e = getenv("SA_ZF_DIRECT_MAX")) g_zf_direct_max = atoi(e);
        if (const char *e = getenv("SA_INTERP_DIRECT_MAX")) g_interp_direct_max = atoi(e);
        if (const char *e = getenv("SA_EVAL_TREE_MIN_LOG")) g_eval_tree_min = ldexp(1.0, atoi(e));
    });
#endif
}
// primitive 2^log-th root of unity: generator^(2^119 / 2^log), algebra.py:100-114
static void tree_root_of_unity(uint64_t out[2], int log) {
    // algebra.py:100-102: generator 85408008396924667383611388730472331217 has order 2^119; the table is built
    // once (a tree of 2^16 points asks ~60 times per call, each a chain of up to 118 host-side squarings)
    static uint64_t table[120][2];
    static std::once_flag once;
    std::call_once(once, [] {
        const uint64_t g[2] = {0xb5038f9c18f6f7d1ull, 0x4040fbed12ee470full};
        fe w = fe_to_mont(fe_from_limbs(g));
        for (int i = 119; i >= 0; i--) {
            const fe c = fe_from_mont(w);
            table[i][0] = (uint64_t)c.v[0] | ((uint64_t)c.v[1] << 32);
            table[i][1] = (uint64_t)c.v[2] | ((uint64_t)c.v[3] << 32);
            w = fe_montmul(w, w);
        }
    });
    out[0] = table[log][0];
    out[1] = table[log][1];
}
struct PolyTree {
    int logK = 0;
    long long k = 0, K = 0;
    fe *levels = nullptr;      // (logK + 1) * K: level j at levels + j * K
    fe *transforms = nullptr;  // logK * 2K: level j's node vectors zero-padded to 2m and transformed (or nullptr)
    fe *scratch = nullptr;     // 2K
};
static inline unsigned tree_grid(long long n) {
    long long g = (n + 255) / 256;
    return (unsigned)(g < 1 ? 1 : (g > 148 * 8 ? 148 * 8 : g));
}
// builds every level of the zerofier tree of domain[0..k) in `t` (buffers already assigned)
static int tree_build(PolyTree &t, const fe *domain, cudaStream_t st) {
    const long long K = t.K;
    int rc;
    k_tree_leaves<<<(unsigned)((K + 255) / 256), 256, 0, st>>>(t.levels, domain, t.k, K);
    SA_LAUNCH_CHECK();
    for (int j = 0; j < t.logK; j++) {
        uint64_t root[2];
        tree_root_of_unity(root, j + 1);
        fe *T = t.transforms ? t.transforms + (size_t)j * 2 * K : t.scratch;
        fe *child = t.levels + (size_t)j * K, *parent = t.levels + (size_t)(j + 1) * K;
        k_tree_pad<<<tree_grid(2 * K), 256, 0, st>>>(T, child, K, j);
        SA_LAUNCH_CHECK();
        if ((rc = sa_ntt(T, T, j + 1, root, 0, (size_t)(K >> j), st)) != SA_OK) return rc;
        k_tree_pairmul<<<tree_grid(K), 256, 0, st>>>(parent, T, K, j);
        SA_LAUNCH_CHECK();
        if ((rc = sa_ntt(parent, parent, j + 1, root, 1, (size_t)(K >> (j + 1)), st)) != SA_OK) return rc;
        k_tree_fix<<<tree_grid(K / 2), 256, 0, st>>>(parent, child, K, j, t.k, 0);
        SA_LAUNCH_CHECK();
    }
    return SA_OK;
}
static int tree_alloc(PolyTree &t, size_t k, bool keep_transforms, size_t extra_elems, fe **extra, cudaStream_t st) {
    t.k = (long long)k;
    t.logK = 0;
    while ((size_t(1) << t.logK) < k) t.logK++;
    if (t.logK > TREE_MAX_LOG) return SA_ESIZE;
    t.K = 1ll << t.logK;
    const size_t K = (size_t)t.K;
    const size_t lv = (size_t)(t.logK + 1) * K, tr = keep_transforms ? (size_t)t.logK * 2 * K : 0, sc = 2 * K;
    fe *ws = nullptr;
    int rc = get_workspace((void **)&ws, sizeof(fe) * (lv + tr + sc + extra_elems), st, 8);
    if (rc != SA_OK) return rc;
    t.levels = ws;
    t.transforms = keep_transforms ? ws + lv : nullptr;
    t.scratch = ws + lv + tr;
    if (extra) *extra = ws + lv + tr + sc;
    return SA_OK;
}

static inline size_t pow2_ceil(size_t x) {
    size_t p = 1;
    while (p < x) p <<= 1;
    return p;
}
// elements of extra workspace tree_multipoint needs for nf coefficients at the tree's k points
static size_t multipoint_extra(size_t nf, size_t k) {
    const size_t N = pow2_ceil(nf > k ? nf : k), K = pow2_ceil(k);
    return 4 * N + N + 2 * K + 16;
}
// vals[i] = f(d_i), i < k, for the tree `t` (built with transforms kept) whose root polynomial is z (k + 1
// coefficients); f has nf >= 1 coefficients.  `ws` = multipoint_extra(nf, k) elements.  See the kernels' comment.
static int tree_multipoint(const PolyTree &t, const fe *z, const fe *f, size_t nf, fe *vals, fe *ws, cudaStream_t st) {
    const long long k = t.k, K = t.K;
    const long long n = (long long)(nf > (size_t)k ? nf : (size_t)k), N = (long long)pow2_ceil((size_t)n);
    fe *W = ws, *alpha = W + 4 * N, *c0 = alpha + N, *c1 = c0 + K;
    int rc;
    uint64_t root[2];
    // alpha = 1 / rev_k(z) mod x^N by Newton: alpha_2s = alpha_s (2 - r alpha_s) mod x^2s in transforms of size 4s
    const fe one = fe_one();
    SA_CUDA(cudaMemcpyAsync(alpha, &one, sizeof(fe), cudaMemcpyHostToDevice, st));
    for (long long s = 1; s < N; s <<= 1) {
        const int lg = host_log2((size_t)(4 * s));
        tree_root_of_unity(root, lg);
        k_series_pad<<<tree_grid(8 * s), 256, 0, st>>>(W, z, k, alpha, s);
        SA_LAUNCH_CHECK();
        if ((rc = sa_ntt(W, W, lg, root, 0, 2, st)) != SA_OK) return rc;
        k_series_step<<<tree_grid(4 * s), 256, 0, st>>>(W, 4 * s);
        SA_LAUNCH_CHECK();
        if ((rc = sa_ntt(W, W, lg, root, 1, 1, st)) != SA_OK) return rc;
        SA_CUDA(cudaMemcpyAsync(alpha, W, sizeof(fe) * 2 * s, cudaMemcpyDeviceToDevice, st));
    }
    // s = rev_{n-1}(f) * alpha mod x^n; the walk starts from c_root[i] = s[n - k + i]
    {
        const long long n2 = 2 * N;
        const int lg = host_log2((size_t)n2);
        tree_root_of_unity(root, lg);
        k_eval_top_pad<<<tree_grid(2 * n2), 256, 0, st>>>(W, f, (long long)nf, alpha, n, n2);
        SA_LAUNCH_CHECK();
        if ((rc = sa_ntt(W, W, lg, root, 0, 2, st)) != SA_OK) return rc;
        k_pointwise_mul<<<tree_grid(n2), 256, 0, st>>>(W, W, W + n2, n2);
        SA_LAUNCH_CHECK();
        if ((rc = sa_ntt(W, W, lg, root, 1, 1, st)) != SA_OK) return rc;
        k_eval_root<<<(unsigned)((K + 255) / 256), 256, 0, st>>>(c0, W, n, k, K);
        SA_LAUNCH_CHECK();
    }
    // walk down: level j + 1 (nodes of 2m) -> level j (nodes of m); W is free again: chat = W[0, K), O = W[K, 3K)
    fe *cur = c0, *nxt = c1, *chat = W, *O = W + K;
    for (int j = t.logK - 1; j >= 0; j--) {
        tree_root_of_unity(root, j + 1);
        const fe *VT = t.transforms + (size_t)j * 2 * K;
        if ((rc = sa_ntt(chat, cur, j + 1, root, 0, (size_t)(K >> (j + 1)), st)) != SA_OK) return rc;
        k_tree_down<<<tree_grid(2 * K), 256, 0, st>>>(O, chat, VT, K, j);
        SA_LAUNCH_CHECK();
        if ((rc = sa_ntt(O, O, j + 1, root, 1, (size_t)(K >> j), st)) != SA_OK) return rc;
        k_tree_down_fix<<<tree_grid(K), 256, 0, st>>>(nxt, O, cur, K, j, k);
        SA_LAUNCH_CHECK();
        fe *tmp = cur;
        cur = nxt;
        nxt = tmp;
    }
    SA_CUDA(cudaMemcpyAsync(vals, cur, sizeof(fe) * (size_t)k, cudaMemcpyDeviceToDevice, st));
    return SA_OK;
}

extern "C" {

int sa_zerofier(void *out, const void *domain, size_t k, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    tree_config();
    if (k == 0) {  // the empty product (the drop-in answers Polynomial([]) before it gets here, ntt.py:70-71)
        const fe one = fe_one();
        SA_CUDA(cudaMemcpyAsync(out, &one, sizeof(fe), cudaMemcpyHostToDevice, st));
        SA_CUDA(cudaStreamSynchronize(st));
        return SA_OK;
    }
    if (k <= (size_t)g_zf_direct_max && k <= (size_t)ZF_MAXK) {
        const size_t smem = sizeof(fe) * (2 * k + 1);
        static std::atomic<bool> attr_done[SA_MAX_DEVICES];
        const int rc = optin_smem(k_zerofier, attr_done, sizeof(fe) * (2 * ZF_MAXK + 1));
        if (rc != SA_OK) return rc;
        k_zerofier<<<1, ZF_THREADS, smem, st>>>((fe *)out, (const fe *)domain, (int)k);
        SA_LAUNCH_CHECK();
        return SA_OK;
    }
    PolyTree t;
    int rc = tree_alloc(t, k, false, 0, nullptr, st);
    if (rc != SA_OK) return rc;
    if ((rc = tree_build(t, (const fe *)domain, st)) != SA_OK) return rc;
    k_tree_root<<<(unsigned)((k + 1 + 255) / 256), 256, 0, st>>>((fe *)out, t.levels + (size_t)t.logK * t.K, t.k, t.K);
    SA_LAUNCH_CHECK();
    return SA_OK;
}

static int interpolate_direct(void *out, const void *domain, const void *values, size_t k, cudaStream_t st) {
    // workspace: z (k+1) | w (k) | flag | QT (k*k)
    char *ws = nullptr;
    const size_t z_off = 0, w_off = sizeof(fe) * (k + 1), f_off = w_off + sizeof(fe) * k,
                 q_off = f_off + 16, total = q_off + sizeof(fe) * k * k;
    int rc = get_workspace((void **)&ws, total, st, 7);
    if (rc != SA_OK) return rc;
    fe *z = (fe *)(ws + z_off), *w = (fe *)(ws + w_off), *QT = (fe *)(ws + q_off);
    int *flag = (int *)(ws + f_off);
    if ((rc = sa_zerofier(z, domain, k, (void *)st)) != SA_OK) return rc;
    SA_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), st));
    const int bs = 128, grid = (int)((k + bs - 1) / bs);
    k_interp_weights<<<grid, bs, 0, st>>>(w, (const fe *)domain, (const fe *)values, z, (int)k, flag);
    SA_LAUNCH_CHECK();
    k_interp_rows<<<grid, bs, 0, st>>>(QT, (const fe *)domain, w, z, (int)k);
    SA_LAUNCH_CHECK();
    k_interp_colsum<<<(unsigned)k, 256, 0, st>>>((fe *)out, QT, (int)k);
    SA_LAUNCH_CHECK();
    int h = 0;
    SA_CUDA(cudaMemcpyAsync(&h, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
    SA_CUDA(cudaStreamSynchronize(st));
    return h ? SA_EDIVZERO : SA_OK;
}

// Lagrange interpolation through the subproduct tree, everything on the device:
//   M = prod (X - d_i) (tree), q_i = v_i / M'(d_i), and the interpolant sum_i q_i M / (X - d_i) is
//   combined bottom-up: P_node = P_L * M_R + P_R * M_L (the M's are the tree's nodes, their transforms
//   kept from the build).  M'(d_i) comes from one Horner kernel (k^2 / 2 multiply-adds, all points in
//   parallel); coinciding points give M'(d_i) = 0 -> SA_EDIVZERO like the division at ntt.py:124-125.
static int interpolate_tree(void *out, const void *domain, const void *values, size_t k, cudaStream_t st) {
    PolyTree t;
    fe *extra = nullptr;
    // extra: z (K + 1) | dz (K) | ev (K) | q (K) | P levels ping-pong (2 * K)
    const size_t Kpad = (size_t)1 << (k <= 1 ? 0 : (64 - __builtin_clzll((unsigned long long)(k - 1))));
    const bool walk = (double)k * (double)k >= g_eval_tree_min;  // M'(d_i): Horner is k^2 products
    int rc = tree_alloc(t, k, true, 6 * Kpad + 16 + (walk ? multipoint_extra(k, k) : 0), &extra, st);
    if (rc != SA_OK) return rc;
    const size_t K = (size_t)t.K;
    fe *z = extra, *dz = z + K + 1, *ev = dz + K, *q = ev + K, *Pa = q + K, *Pb = Pa + K, *mp = Pb + K + 16;
    if ((rc = tree_build(t, (const fe *)domain, st)) != SA_OK) return rc;
    k_tree_root<<<(unsigned)((k + 1 + 255) / 256), 256, 0, st>>>(z, t.levels + (size_t)t.logK * K, t.k, t.K);
    SA_LAUNCH_CHECK();
    k_derivative<<<(unsigned)((k + 255) / 256), 256, 0, st>>>(dz, z, (long long)k);
    SA_LAUNCH_CHECK();
    if (walk)
        rc = tree_multipoint(t, z, dz, k, ev, mp, st);
    else
        rc = poly_eval_horner(ev, dz, k, domain, k, (void *)st);
    if (rc != SA_OK) return rc;
    if ((rc = sa_pointwise_div(q, values, ev, k, (void *)st)) != SA_OK) return rc;  // SA_EDIVZERO: repeated point
    k_tree_qleaves<<<(unsigned)((K + 255) / 256), 256, 0, st>>>(Pa, q, t.k, t.K);
    SA_LAUNCH_CHECK();
    fe *cur = Pa, *nxt = Pb;
    for (int j = 0; j < t.logK; j++) {
        uint64_t root[2];
        tree_root_of_unity(root, j + 1);
        const fe *VT = t.transforms + (size_t)j * 2 * K;
        k_tree_pad<<<tree_grid(2 * (long long)K), 256, 0, st>>>(t.scratch, cur, t.K, j);
        SA_LAUNCH_CHECK();
        if ((rc = sa_ntt(t.scratch, t.scratch, j + 1, root, 0, K >> j, (void *)st)) != SA_OK) return rc;
        k_tree_cross<<<tree_grid((long long)K), 256, 0, st>>>(nxt, t.scratch, VT, t.K, j);
        SA_LAUNCH_CHECK();
        if ((rc = sa_ntt(nxt, nxt, j + 1, root, 1, K >> (j + 1), (void *)st)) != SA_OK) return rc;
        k_tree_fix<<<tree_grid((long long)K / 2), 256, 0, st>>>(nxt, cur, t.K, j, t.k, 1);
        SA_LAUNCH_CHECK();
        fe *tmp = cur;
        cur = nxt;
        nxt = tmp;
    }
    SA_CUDA(cudaMemcpyAsync(out, cur, sizeof(fe) * k, cudaMemcpyDeviceToDevice, st));
    return SA_OK;
}

int sa_interpolate(void *out, const void *domain, const void *values, size_t k, void *stream) {
    if (k == 0) return SA_OK;
    tree_config();
    cudaStream_t st = (cudaStream_t)stream;
    if (k <= (size_t)g_interp_direct_max && k <= (size_t)ZF_MAXK) return interpolate_direct(out, domain, values, k, st);
    if (k > ((size_t)1 << TREE_MAX_LOG)) return SA_ESIZE;
    return interpolate_tree(out, domain, values, k, st);
}

// fast_evaluate (ntt.py:82-100): Horner for small jobs, the transposed tree walk (tree_multipoint) for big ones
int sa_poly_eval_mode(void *out, const void *coeffs, size_t ncoef, const void *points, size_t npoints, int mode,
                      void *stream) {
    if (npoints == 0) return SA_OK;
    if (mode < 0 || mode > 2) return SA_ESIZE;
    tree_config();
    cudaStream_t st = (cudaStream_t)stream;
    const size_t nmax = ncoef > npoints ? ncoef : npoints;
    if (mode == 0)
        mode = (ncoef < 2 || npoints < 2 || (double)ncoef * (double)npoints < g_eval_tree_min ||
                nmax > ((size_t)1 << TREE_MAX_LOG)) ? 1 : 2;
    if (mode == 1) return poly_eval_horner(out, coeffs, ncoef, points, npoints, stream);
    if (nmax > ((size_t)1 << TREE_MAX_LOG)) return SA_ESIZE;
    if (ncoef == 0) {  // the zero polynomial
        SA_CUDA(cudaMemsetAsync(out, 0, sizeof(fe) * npoints, st));
        return SA_OK;
    }
    PolyTree t;
    fe *extra = nullptr;
    const size_t K = pow2_ceil(npoints);
    int rc = tree_alloc(t, npoints, true, K + 1 + 16 + multipoint_extra(ncoef, npoints), &extra, st);
    if (rc != SA_OK) return rc;
    fe *z = extra, *mp = z + K + 1 + 15;
    if ((rc = tree_build(t, (const fe *)points, st)) != SA_OK) return rc;
    k_tree_root<<<(unsigned)((npoints + 1 + 255) / 256), 256, 0, st>>>(z, t.levels + (size_t)t.logK * t.K, t.k, t.K);
    SA_LAUNCH_CHECK();
    return tree_multipoint(t, z, (const fe *)coeffs, ncoef, (fe *)out, mp, st);
}
int sa_poly_eval(void *out, const void *coeffs, size_t ncoef, const void *points, size_t npoints, void *stream) {
    return sa_poly_eval_mode(out, coeffs, ncoef, points, npoints, 0, stream);
}

// ---- Merkle / FRI ----
#ifdef SA_TUNE
// SA_MK_SHAPE="minlog:ipt:chunklog:red:coopmax,..." overrides the launch shape of levels with width >= 2^minlog
static void merkle_shape_env(MerkleArgs &a) {
    const char *e = getenv("SA_MK_SHAPE");
    if (!e) return;
    int best = -1, w = merkle_log2(a.width);
    while (*e) {
        int ml, ipt, cl, red, coop, used = 0;
        if (sscanf(e, "%d:%d:%d:%d:%d%n", &ml, &ipt, &cl, &red, &coop, &used) != 5) break;
        if (ml <= w && ml > best && cl <= w) {
            best = ml;
            a.ipt_log = ipt;
            a.chunk = 1 << cl;
            a.red_log = red;
            a.coop_max = coop;
        }
        e += used;
        if (*e == ',') e++;
    }
}
#endif
// arrival counters of k_merkle_chunk's fused top, one per (device, stream): zero whenever no launch
// of that stream is in flight (the last CTA resets it)
static std::map<std::pair<int, cudaStream_t>, unsigned int *> g_tickets;
static unsigned int *get_ticket(cudaStream_t st) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    std::lock_guard<std::mutex> lock(g_ws_mu);
    auto &slot = g_tickets[std::make_pair(dev, st)];
    if (!slot) {
        if (cudaMalloc((void **)&slot, 256) != cudaSuccess || cudaMemset(slot, 0, 256) != cudaSuccess) {
            slot = nullptr;
            cudaGetLastError();
        }
    }
    return slot;  // nullptr: fall back to one more launch
}
static int merkle_reduce(MerkleArgs a, cudaStream_t st, uint64_t *root_host = nullptr, unsigned long long seq = 0) {
    unsigned int *ticket = get_ticket(st);
    // first launch handles the bottom level in a.mode, later launches continue from digests
    while (true) {
        merkle_shape(a);
#ifdef SA_TUNE
        merkle_shape_env(a);
#endif
        // the launch that leaves at most MK_THREADS single-digest CTAs also reduces those (ticket)
        const long long left = merkle_next_width(a), grid = a.width / a.chunk;
        const bool fuse_top = left > 1 && left <= MK_THREADS && left == grid && ticket != nullptr;
        const bool last = left <= 1 || fuse_top;
        a.ticket = fuse_top ? ticket : nullptr;
        a.root_out = last ? root_host : nullptr;
        a.root_seq = seq;
        k_merkle_chunk<<<(unsigned)(a.width / a.chunk), MK_THREADS, 0, st>>>(a);
        SA_LAUNCH_CHECK();
        if (last) break;
        a.width = merkle_next_width(a);
        a.mode = 0;
    }
    return SA_OK;
}

int sa_merkle_tree(void *tree, const void *values, size_t n, void *stream) {
    if (!host_is_pow2(n)) return SA_ENOTPOW2;
    cudaStream_t st = (cudaStream_t)stream;
    SA_CUDA(cudaMemsetAsync(tree, 0, 64, st));
    MerkleArgs a;
    memset(&a, 0, sizeof(a));
    a.tree = (uint64_t *)tree;
    a.width = (long long)n;
    a.mode = 1;
    a.values = (const fe *)values;
    return merkle_reduce(a, st);
}

int sa_merkle_open(void *paths_out, const void *tree, size_t n, const uint64_t *indices_host, size_t k,
                   void *stream) {
    if (!host_is_pow2(n)) return SA_ENOTPOW2;
    for (size_t i = 0; i < k; i++)
        if (indices_host[i] >= n) return SA_EINDEX;
    const int depth = host_log2(n);
    if (k == 0 || depth == 0) return SA_OK;
    cudaStream_t st = (cudaStream_t)stream;
    uint64_t *idx = nullptr;
    keep_pool_memory();
    SA_CUDA(cudaMallocAsync((void **)&idx, 8 * k, st));
    SA_CUDA(cudaMemcpyAsync(idx, indices_host, 8 * k, cudaMemcpyHostToDevice, st));
    const long long total = (long long)k * depth * 8;
    k_merkle_paths<<<(unsigned)((total + 255) / 256), 256, 0, st>>>((uint64_t *)paths_out,
                                                                    (const uint64_t *)tree, (long long)n,
                                                                    depth, idx, (long long)k);
    SA_LAUNCH_CHECK();
    cudaFreeAsync(idx, st);
    return SA_OK;
}

int sa_gather(void *out, const void *values, size_t n, const uint64_t *indices_host, size_t k, void *stream) {
    for (size_t i = 0; i < k; i++)
        if (indices_host[i] >= n) return SA_EINDEX;
    if (k == 0) return SA_OK;
    cudaStream_t st = (cudaStream_t)stream;
    uint64_t *idx = nullptr;
    keep_pool_memory();
    SA_CUDA(cudaMallocAsync((void **)&idx, 8 * k, st));
    SA_CUDA(cudaMemcpyAsync(idx, indices_host, 8 * k, cudaMemcpyHostToDevice, st));
    k_gather<<<(unsigned)((k + 127) / 128), 128, 0, st>>>((fe *)out, (const fe *)values, idx, (long long)k);
    SA_LAUNCH_CHECK();
    cudaFreeAsync(idx, st);
    return SA_OK;
}

// x_i^-1 tables: xinv[i] = omega^-i (Montgomery), i < n/2, cached per (device, omega, n) in the LRU above
static int get_xinv(XinvPtr *out, const fe &omega, size_t n, cudaStream_t st) {
    int dev = 0;
    SA_CUDA(cudaGetDevice(&dev));
    const CacheKey key(1, dev, (uint64_t)n, (uint64_t)omega.v[0] | ((uint64_t)omega.v[1] << 32),
                       (uint64_t)omega.v[2] | ((uint64_t)omega.v[3] << 32), 0);
    if ((*out = cache_find<XinvTable>(key))) return SA_OK;
    const fe winv_m = fe_mont_inv(fe_to_mont(omega));
    XinvPtr made = std::make_shared<XinvTable>();
    made->device = dev;
    int rc = build_pow_table(*made, &made->tab, winv_m, fe_mont_one(), (long long)(n / 2), st);
    if (rc != SA_OK) return rc;
    SA_CUDA(cudaStreamSynchronize(st));  // complete before other streams can find it in the cache
    *out = cache_publish<XinvTable>(key, made);
    return SA_OK;
}

static int fri_scalars(fe *s_m, fe *inv2_m, const uint64_t alpha[2], const uint64_t offset[2]) {
    *inv2_m = fe_mont_inv(fe_to_mont(fe_from_u64(2)));
    const fe oinv_m = fe_mont_inv(fe_to_mont(fe_from_limbs(offset)));
    // alpha * 2^-1 * offset^-1, Montgomery form
    *s_m = fe_montmul(fe_montmul(fe_to_mont(fe_from_limbs(alpha)), *inv2_m), oinv_m);
    return SA_OK;
}

int sa_fri_fold(void *next, const void *cw, size_t n, const uint64_t alpha[2], const uint64_t offset[2],
                const uint64_t omega[2], void *stream) {
    if (!host_is_pow2(n) || n < 2) return SA_ENOTPOW2;
    cudaStream_t st = (cudaStream_t)stream;
    XinvPtr xinv;
    int rc = get_xinv(&xinv, fe_from_limbs(omega), n, st);
    if (rc != SA_OK) return rc;
    fe s_m, inv2_m;
    fri_scalars(&s_m, &inv2_m, alpha, offset);
    k_fri_fold<<<grid_for((long long)(n / 2), 128), 128, 0, st>>>((fe *)next, (const fe *)cw,
                                                                 (long long)(n / 2), xinv->tab, s_m, inv2_m);
    SA_LAUNCH_CHECK();
    return SA_OK;
}

int sa_fri_round(void *next, void *next_tree, const void *cw, size_t n, const uint64_t alpha[2],
                 const uint64_t offset[2], const uint64_t omega[2], void *stream) {
    if (!host_is_pow2(n) || n < 2) return SA_ENOTPOW2;
    cudaStream_t st = (cudaStream_t)stream;
    XinvPtr xinv;
    int rc = get_xinv(&xinv, fe_from_limbs(omega), n, st);
    if (rc != SA_OK) return rc;
    SA_CUDA(cudaMemsetAsync(next_tree, 0, 64, st));
    MerkleArgs a;
    memset(&a, 0, sizeof(a));
    a.tree = (uint64_t *)next_tree;
    a.width = (long long)(n / 2);
    a.mode = 2;
    a.prev = (const fe *)cw;
    a.next = (fe *)next;
    a.xinv = xinv->tab;
    fri_scalars(&a.s_m, &a.inv2_m, alpha, offset);
    return merkle_reduce(a, st);
}

// spin until the kernel has published root number `seq` (see merkle_publish_root); the stream is
// polled now and then so that a failed launch turns into an error instead of a hang
static int wait_for_root(uint64_t *root_host, unsigned long long seq, cudaStream_t st) {
    volatile uint64_t *flag = root_host + 8;
    for (unsigned spins = 1; *flag != seq; spins++) {
        if ((spins & 0xfff) == 0) {
            const cudaError_t q = cudaStreamQuery(st);
            if (q == cudaSuccess) {
                if (*flag == seq) break;
                g_last_error = "sa_fri_commit: the stream drained without publishing the round root";
                return SA_ECUDA;
            }
            if (q != cudaErrorNotReady) {
                g_last_error = std::string("sa_fri_commit: ") + cudaGetErrorString(q);
                return SA_ECUDA;
            }
        }
#if defined(__x86_64__)
        __builtin_ia32_pause();
#endif
    }
    std::atomic_thread_fence(std::memory_order_acquire);
    return SA_OK;
}

int sa_fri_commit(void *layers, void *trees, const void *codeword, size_t n, int rounds,
                  const uint64_t offset[2], const uint64_t omega[2], sa_fri_challenge_fn challenge, void *user,
                  void *stream) {
    if (!host_is_pow2(n) || rounds < 1 || (n >> (rounds - 1)) < 1) return SA_ESIZE;
    cudaStream_t st = (cudaStream_t)stream;
    // landing pad of the per-round root (8 words) + sequence number, written by the kernel itself
    static thread_local uint64_t *root_pinned = nullptr;
    static thread_local uint64_t *root_dev = nullptr;  // the same memory as the device addresses it
    static thread_local unsigned long long root_seq = 0;
    if (!root_pinned) {
        SA_CUDA(cudaHostAlloc((void **)&root_pinned, 256, cudaHostAllocMapped | cudaHostAllocPortable));
        memset(root_pinned, 0, 256);
    }
    SA_CUDA(cudaHostGetDevicePointer((void **)&root_dev, root_pinned, 0));  // per current device
    fe off = fe_from_limbs(offset), om = fe_from_limbs(omega);
    // host-side scalars of the fold: 2^-1 once, offset^-1 once and then squared along with offset
    // (a Fermat inversion on the host costs ~10 us; per round that was a fifth of the round trip)
    static const fe inv2_m = fe_mont_inv(fe_to_mont(fe_from_u64(2)));
    fe oinv_m = fe_mont_inv(fe_to_mont(off));
    const fe *cur = (const fe *)codeword;
    fe *layer_out = (fe *)layers;
    uint8_t *tree = (uint8_t *)trees;
    size_t len = n;
    int rc;
    static const bool trace = getenv("SA_FRI_TRACE") != nullptr;  // per-round host timeline on stderr
    auto now = [] { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    double t_mark = now();
    for (int r = 0; r < rounds; r++) {
        if (r == 0) {
            MerkleArgs a;
            memset(&a, 0, sizeof(a));
            a.tree = (uint64_t *)tree;
            a.width = (long long)len;
            a.mode = 1;
            a.values = cur;
            if ((rc = merkle_reduce(a, st, root_dev, ++root_seq)) != SA_OK) return rc;
        }
        const double t_launched = now();
        if ((rc = wait_for_root(root_pinned, root_seq, st)) != SA_OK) return rc;
        const double t_synced = now();
        uint64_t alpha[2] = {0, 0};
        const int want = r != rounds - 1;
        if (challenge(user, r, (const uint8_t *)root_pinned, alpha, want) != 0) return SA_ECALLBACK;
        if (trace) {
            const double t_cb = now();
            fprintf(stderr, "sa_fri_commit round %2d len %8zu: launch %.1f us, wait %.1f us, callback %.1f us\n", r, len,
                    t_launched - t_mark, t_synced - t_launched, t_cb - t_synced);
            t_mark = t_cb;
        }
        if (!want) break;
        // fold layer r into layer r+1 and build its tree: alpha / (2 offset), Montgomery form
        const fe s_m = fe_montmul(fe_montmul(fe_to_mont(fe_from_limbs(alpha)), inv2_m), oinv_m);
        uint8_t *next_tree = tree + 128 * len;  // this tree has 2 * len nodes of 64 bytes
        XinvPtr xinv;
        if ((rc = get_xinv(&xinv, om, len, st)) != SA_OK) return rc;
        MerkleArgs a;
        memset(&a, 0, sizeof(a));
        a.tree = (uint64_t *)next_tree;
        a.width = (long long)(len / 2);
        a.mode = 2;
        a.prev = cur;
        a.next = layer_out;
        a.xinv = xinv->tab;
        a.inv2_m = inv2_m;
        a.s_m = s_m;
        if ((rc = merkle_reduce(a, st, root_dev, ++root_seq)) != SA_OK) return rc;
        cur = layer_out;
        layer_out += len / 2;
        tree = next_tree;
        len /= 2;
        const fe om_m = fe_to_mont(om), off_m = fe_to_mont(off);
        om = fe_montmul(om_m, om);      // omega^2  (Montgomery form times canonical = canonical product)
        off = fe_montmul(off_m, off);   // offset^2
        oinv_m = fe_montmul(oinv_m, oinv_m);  // (offset^2)^-1, stays in Montgomery form
    }
    return SA_OK;
}

size_t sa_cache_limit(size_t bytes) {
    cache_config();
    std::lock_guard<std::mutex> lock(g_plan_mu);
    g_cache_limit = bytes;
    cache_make_room(0);
    return g_cache_bytes;
}
size_t sa_cache_bytes(void) {
    std::lock_guard<std::mutex> lock(g_plan_mu);
    return g_cache_bytes;
}
int sa_release_workspaces(void) {
    SA_CUDA(cudaDeviceSynchronize());
    int dev = 0;
    SA_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_ws_mu);
    for (auto it = g_ws.begin(); it != g_ws.end();) {
        if (std::get<0>(it->first) == dev) {
            if (it->second.first) cudaFree(it->second.first);
            it = g_ws.erase(it);
        } else {
            ++it;
        }
    }
    cudaGetLastError();
    return SA_OK;
}

long long sa_selftest_field(size_t count, uint64_t seed) {
    unsigned long long *d = nullptr, h = 0;
    SA_CUDA(cudaMalloc(&d, 8));
    SA_CUDA(cudaMemset(d, 0, 8));
    k_selftest_field<<<(unsigned)((count + 255) / 256), 256>>>(d, (long long)count, seed);
    SA_LAUNCH_CHECK();
    SA_CUDA(cudaMemcpy(&h, d, 8, cudaMemcpyDeviceToHost));
    cudaFree(d);
    return (long long)h;
}

}  // extern "C"
template <int OP>
static double microbench_op(int ilp, int iters, int blocks, int threads, fe *sink) {
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    auto run = [&](int it) {
        switch (ilp) {
            case 1: k_microbench<OP, 1><<<blocks, threads>>>(sink, it); break;
            case 2: k_microbench<OP, 2><<<blocks, threads>>>(sink, it); break;
            case 4: k_microbench<OP, 4><<<blocks, threads>>>(sink, it); break;
            default: k_microbench<OP, 8><<<blocks, threads>>>(sink, it); break;
        }
    };
    run(iters / 8 + 1);  // warm up
    cudaEventRecord(e0);
    run(iters);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return (double)ms;
}
extern "C" {
double sa_microbench(int op, int ilp, int iters, int blocks, int threads) {
    fe *sink = nullptr;
    if (cudaMalloc(&sink, sizeof(fe) * (size_t)blocks * (threads > MK_THREADS ? threads : MK_THREADS)) != cudaSuccess)
        return -1.0;
    double ms = -1.0;
    switch (op) {
        case 0: ms = microbench_op<0>(ilp, iters, blocks, threads, sink); break;
        case 1: ms = microbench_op<1>(ilp, iters, blocks, threads, sink); break;
        case 2: ms = microbench_op<2>(ilp, iters, blocks, threads, sink); break;
        case 3: ms = microbench_op<3>(ilp, iters, blocks, threads, sink); break;
        case 4: {  // blake2b node compressions (threads is fixed at MK_THREADS)
            cudaEvent_t e0, e1;
            cudaEventCreate(&e0);
            cudaEventCreate(&e1);
            auto run = [&](int it) {
                if (ilp >= 2)
                    k_microbench_b2<2><<<blocks, MK_THREADS>>>((uint64_t *)sink, it);
                else
                    k_microbench_b2<1><<<blocks, MK_THREADS>>>((uint64_t *)sink, it);
            };
            run(iters / 8 + 1);
            cudaEventRecord(e0);
            run(iters);
            cudaEventRecord(e1);
            cudaEventSynchronize(e1);
            float f = 0;
            cudaEventElapsedTime(&f, e0, e1);
            cudaEventDestroy(e0);
            cudaEventDestroy(e1);
            ms = (double)f;
            break;
        }
    }
    g_launches.fetch_add(2);
    if (cudaGetLastError() != cudaSuccess) ms = -1.0;
    cudaFree(sink);
    return ms;
}

}  // extern "C"
