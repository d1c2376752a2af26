/*
 * sa_b200.h -- C ABI of the B200 (sm_100a) NTT + FRI engine that stands in for the
 * hot path of aszepieniec/stark-anatomy (code/ntt.py, code/fri.py, code/merkle.py).
 *
 * The reference is pure Python and has no FFI: its boundary is the Python module
 * surface (SURVEY.md section 8b).  The entry points below are what a ctypes
 * binding for that path binds; stark-anatomy_b200/sa_engine.py is that binding
 * and INTEGRATION.md shows the stub a maintainer would add to the reference.
 *
 * Conventions
 *  - One field element = 16 bytes: two little-endian uint64 limbs (lo, hi) of the
 *    canonical residue in [0, p), p = 1 + 407 * 2^119 (code/algebra.py:96-98).
 *  - Scalars (roots, offsets, challenges) are passed as `const uint64_t x[2]`.
 *  - `void *` data pointers are DEVICE pointers unless the function name ends in
 *    `_host`; `stream` is a cudaStream_t (NULL = default stream).  Calls are
 *    asynchronous on `stream` unless stated otherwise.
 *  - Return value: 0 on success, otherwise one of the SA_E* codes; the Python
 *    binding turns SA_E* into the AssertionError (with the reference's message)
 *    the corresponding reference function raises.
 *  - No torch types, no C++ types: plain pointers and sizes.
 *  - Thread safety: entry points may be called from several host threads; the
 *    twiddle/plan caches are guarded by a mutex (tables are built outside of it).  Work submitted to different
 *    streams is independent (scratch buffers and the Merkle arrival counter are per
 *    device and stream); two threads must not be inside calls on the SAME stream at
 *    the same time.  sa_ntt_host calls on one device run one after the other
 *    (they share the copy streams - and the PCIe link).
 */
#ifndef SA_B200_H
#define SA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
    SA_OK = 0,
    SA_ENOTPOW2 = -1,   /* ntt.py:4   "cannot compute ntt of non-power-of-two sequence" */
    SA_EROOTORDER = -2, /* ntt.py:10  "primitive root must be nth root of unity, where n is len(values)" */
    SA_ENOTPRIM = -3,   /* ntt.py:11  "primitive root is not primitive nth root of unity, ..." */
    SA_EDIVZERO = -4,   /* algebra.py:92 "divide by zero" (element-wise division, ntt.py:172) */
    SA_EINDEX = -5,     /* merkle.py:18 "cannot open invalid index" */
    SA_ESIZE = -6,      /* unsupported size (log_n > 26, n == 0, ...) */
    SA_ECALLBACK = -7,  /* the challenge callback of sa_fri_commit returned non-zero */
    SA_ECUDA = -100     /* CUDA runtime error; sa_last_error() has the text */
};

/* Version / build info, e.g. "sa_b200 0.1 sm_100a". */
const char *sa_version(void);
/* Text of the last CUDA error seen by this thread's calls (empty string if none). */
const char *sa_last_error(void);
/* Number of kernel launches issued by this library since load (bench.py's gpu_launches). */
uint64_t sa_launch_count(void);

/* ---- code/ntt.py:3-18 ntt, code/ntt.py:20-30 intt -------------------------------------
 * out[b][i] = sum_j in[b][j] * root^(i*j), natural order in and out, for `batch`
 * contiguous transforms of n = 2^log_n elements.  inverse != 0 computes intt: the
 * transform with root^-1 followed by the multiplication with n^-1.
 * Validates root^n == 1 and root^(n/2) != 1 exactly like the reference's asserts.
 * in == out is allowed.  log_n in [0, 26].                                               */
int sa_ntt(void *out, const void *in, int log_n, const uint64_t root[2], int inverse, size_t batch,
           void *stream);
/* Multi-GPU assembly (SURVEY 8e; no reference counterpart: the reference is one thread on one CPU).
 * The same transforms, but the results are written to element offset `out_offset` of EVERY buffer
 * outs[0 .. nouts), nouts <= 8: outs[0] is memory of the current device, the others are buffers of
 * other GPUs mapped into this process (CUDA IPC / peer access over NVLink - stark-anatomy_b200/sa_dist.py
 * does the mapping with torch).  The stores to the peers are issued by the last pass of the
 * transform itself, tile by tile, so when every rank has run its shard of a batch each rank holds the
 * whole batch and no gather pass follows.  Completion on the peers is the caller's to synchronise
 * (a barrier across the ranks after the stream has drained).                                  */
int sa_ntt_multi(void *const *outs, int nouts, size_t out_offset, const void *in, int log_n,
                 const uint64_t root[2], int inverse, size_t batch, void *stream);
/* The same through ONE multicast address (NVLS: a multicast object that every rank's buffer is bound to, e.g.
 * torch.distributed._symmetric_memory's multicast_ptr): the last pass issues multimem.st, one store leaves the
 * GPU and the NVSwitch delivers it to every rank's buffer, the own one included.  `local` is this rank's own
 * buffer (same layout; intermediates of the three-pass sizes go there), log_n >= 1.                          */
int sa_ntt_mcast(void *mc, void *local, size_t out_offset, const void *in, int log_n, const uint64_t root[2],
                 int inverse, size_t batch, void *stream);
/* Buffers shared between the processes of one box (one process per GPU): sa_peer_alloc = cudaMalloc (zeroed) +
 * CUDA IPC handle (64 bytes, to be sent to the other processes, e.g. with all_gather_object); sa_peer_open maps
 * another process's buffer into the address space of the CURRENT device and enables peer access to its owner
 * over NVLink, so that this device's kernels (sa_ntt_multi) and copy engines (sa_copy_async) can write it;
 * sa_peer_close / sa_peer_free undo them.  sa_copy_async = cudaMemcpyAsync(cudaMemcpyDefault) on `stream`.   */
int sa_peer_alloc(void **ptr, size_t bytes, uint8_t handle_out[64]);
int sa_peer_open(void **ptr, const uint8_t handle[64]);
int sa_peer_close(void *ptr);
int sa_peer_free(void *ptr);
int sa_copy_async(void *dst, const void *src, size_t bytes, void *stream);
/* One kernel that reads `bytes` (multiple of 16, 16-byte aligned) at src once and stores them to every dsts[i],
 * i < ndst <= 7 (peer-mapped buffers): fully coalesced stores, a warp writes 512 contiguous bytes per
 * destination.  The push half of sa_dist's "p2p-push" assembly: transform i is pushed on a side stream while
 * transform i + 1 computes.  SA_PUSH_CTAS = CTAs of the push kernel (default 148).                          */
int sa_push(void *const *dsts, int ndst, const void *src, size_t bytes, void *stream);
/* The same through ONE multicast address (see sa_ntt_mcast): one multimem.st per 16 bytes, the NVSwitch replicates. */
int sa_push_mcast(void *mc_dst, const void *src, size_t bytes, void *stream);
/* Lets kernels of the CURRENT device store to memory of `peer_device` that is mapped into this process
 * (cudaDeviceEnablePeerAccess; fine if it already is enabled).  A buffer opened from an IPC handle belongs to
 * its owner's device ordinal in this process, and opening it under that ordinal does not enable access from
 * another device (sa_peer_open opens under the accessing device instead, which does).                        */
int sa_enable_peer_access(int peer_device);
/* Same through HOST buffers: H2D copy, transforms, D2H copy, synchronises before
 * returning (the end-to-end call bench.py times as `e2e`).                               */
int sa_ntt_host(void *out_host, const void *in_host, int log_n, const uint64_t root[2], int inverse,
                size_t batch, void *stream);
/* Host buffers for sa_ntt_host (no reference counterpart: the reference keeps Python lists).
 * Page-locked, and allocated on the NUMA node of the current CUDA device (the calling thread is
 * moved onto the CPUs listed in /sys/bus/pci/devices/<gpu>/local_cpulist for the allocation), so
 * that with one process per GPU the copies do not cross the socket interconnect (4 ranks:
 * 6.9e10 -> 9.6e10 butterflies/s end to end).  Any other host memory works too, pageable
 * memory at the speed of pageable copies.  NULL on failure (sa_last_error).               */
void *sa_host_alloc(size_t bytes);
int sa_host_free(void *p);

/* ---- element-wise pieces of fast_multiply / fast_coset_divide / fast_coset_evaluate ---- */
/* code/ntt.py:61  out[i] = a[i] * b[i]                                                   */
int sa_pointwise_mul(void *out, const void *a, const void *b, size_t n, void *stream);
/* code/ntt.py:172 out[i] = a[i] / b[i]; SA_EDIVZERO if some b[i] == 0 (synchronises).    */
int sa_pointwise_div(void *out, const void *a, const void *b, size_t n, void *stream);
/* code/univariate.py:153-154 as used at ntt.py:133,159-160,176: out[i] = in[i] * factor^i */
int sa_scale(void *out, const void *in, size_t n, const uint64_t factor[2], void *stream);
/* code/univariate.py:130-136 at many points (fast_evaluate's values, ntt.py:82-100):
 * out[j] = sum_i coeffs[i] * points[j]^i                                                 */
int sa_poly_eval(void *out, const void *coeffs, size_t ncoef, const void *points, size_t npoints,
                 void *stream);
/* The same with the algorithm chosen by the caller: mode 0 = what sa_poly_eval does (Horner, one thread per
 * point, below 2^27.5 coefficient-point products; above that the walk down the subproduct tree of the points,
 * max(ncoef, npoints) <= 2^20), 1 = Horner, 2 = the tree walk (ncoef, npoints >= 1).  The reference walks down a
 * remainder tree (ntt.py:82-100); the device walks down the TRANSPOSED interpolation tree (no divisions): one
 * power-series inverse at the root, then one batched transform pair per level.  Same values.                 */
int sa_poly_eval_mode(void *out, const void *coeffs, size_t ncoef, const void *points, size_t npoints, int mode,
                      void *stream);

/* code/ntt.py:66-80 fast_zerofier: out[0..k] = coefficients of prod_i (X - domain[i]) (monic,
 * k + 1 coefficients), k <= 2^20.  Small domains: one kernel; larger ones: the subproduct tree of
 * the reference, built level by level on the device with batched transforms (all nodes of a level
 * in one sa_ntt call).                                                                       */
int sa_zerofier(void *out, const void *domain, size_t k, void *stream);
/* code/ntt.py:102-130 fast_interpolate: out[0..k) = coefficients of the polynomial of degree
 * < k with value values[i] at domain[i], k <= 2^20.  SA_EDIVZERO when two domain points coincide
 * (the reference's element-wise division asserts there).  Small k: Lagrange kernels; larger k:
 * zerofier tree, weights v_i / M'(d_i), and a bottom-up combination over the same tree - one call,
 * everything on the device.  Synchronises.                                                    */
int sa_interpolate(void *out, const void *domain, const void *values, size_t k, void *stream);

/* ---- code/merkle.py:6-14 Merkle.commit -------------------------------------------------
 * Builds the whole blake2b-512 tree over n = 2^k leaves, leaf = H(decimal ASCII of the
 * value), node = H(left || right).  `tree` receives 2n nodes of 64 bytes in heap order:
 * node 1 is the root, node i has children 2i and 2i+1, leaf j is node n + j, node 0 is
 * unused.                                                                                 */
int sa_merkle_tree(void *tree, const void *values, size_t n, void *stream);
/* code/merkle.py:16-27 Merkle.open for k leaf indices (HOST array): paths_out receives
 * k * log2(n) digests of 64 bytes, siblings bottom-up per index (device memory).          */
int sa_merkle_open(void *paths_out, const void *tree, size_t n, const uint64_t *indices_host, size_t k,
                   void *stream);
/* out[i] = values[indices[i]] (the leaf triples of code/fri.py:104-105).                  */
int sa_gather(void *out, const void *values, size_t n, const uint64_t *indices_host, size_t k,
              void *stream);

/* ---- code/fri.py:85 split-and-fold, and the fused round of Fri.commit (fri.py:64-88) ----
 * next[i] = 2^-1 * ((1 + alpha/(offset*omega^i)) * cw[i] + (1 - alpha/(offset*omega^i)) * cw[n/2+i])
 * for i < n/2.  sa_fri_round additionally builds the Merkle tree of `next` (n/2 leaves,
 * n nodes of 64 bytes) in the same kernel that folds; sa_fri_fold only folds.             */
int sa_fri_fold(void *next, const void *cw, size_t n, const uint64_t alpha[2], const uint64_t offset[2],
                const uint64_t omega[2], void *stream);
int sa_fri_round(void *next, void *next_tree, const void *cw, size_t n, const uint64_t alpha[2],
                 const uint64_t offset[2], const uint64_t omega[2], void *stream);

/* ---- code/fri.py:56-96 Fri.commit, the whole round loop in one call -----------------------
 * Round 0 builds the Merkle tree of `codeword` (n = 2^k elements); every later round is the
 * fused fold + tree kernel on the previous layer.  After each round the 64-byte root is copied
 * to the host and `challenge(user, round, root, alpha_out, want_alpha)` is called: the caller
 * pushes the root into its proof stream (fri.py:72) and, when want_alpha != 0, writes the
 * Fiat-Shamir challenge alpha = field.sample(proof_stream.prover_fiat_shamir()) (fri.py:79)
 * into alpha_out; a non-zero return aborts the commit (SA_ECALLBACK).  omega / offset are
 * squared per round (fri.py:87-88).
 *   layers : device buffer for layers 1 .. rounds-1, layer r (n >> r elements) at element
 *            offset n - (n >> (r-1)), i.e. back to back;  total n - (n >> (rounds-1)) elements
 *   trees  : device buffer for the trees of layers 0 .. rounds-1, back to back, tree r has
 *            2 * (n >> r) nodes of 64 bytes;  total 4n - (4n >> rounds) nodes               */
typedef int (*sa_fri_challenge_fn)(void *user, int round, const uint8_t root[64], uint64_t alpha_out[2],
                                   int want_alpha);
int sa_fri_commit(void *layers, void *trees, const void *codeword, size_t n, int rounds,
                  const uint64_t offset[2], const uint64_t omega[2], sa_fri_challenge_fn challenge, void *user,
                  void *stream);

/* ---- device memory the library keeps between calls (no reference counterpart) ------------------
 * Twiddle tables (per device, log n, root, direction) and FRI x^-1 tables (per device, omega, n)
 * live in one least-recently-used cache bounded by bytes: default 4 GiB, SA_CACHE_LIMIT_MIB, or
 * sa_cache_limit(bytes), which also evicts down to the new limit right away and returns the bytes
 * still cached (sa_cache_limit(0) drops everything).  A table in use by an enqueued kernel is freed
 * only after that kernel has finished.  sa_cache_bytes() = bytes cached now.
 * sa_release_workspaces() synchronises the current device and frees its per-stream scratch buffers
 * (the n * batch intermediate of the multi-pass transforms, host-entry staging), which otherwise
 * only grow.                                                                                */
size_t sa_cache_limit(size_t bytes);
size_t sa_cache_bytes(void);
int sa_release_workspaces(void);

/* ---- self checks (used by tests / smoke) ------------------------------------------------
 * Runs the sm_100a carry-chain field arithmetic against the portable C++ version on
 * `count` pseudo-random pairs (plus edge cases) on the device; returns the number of
 * mismatches (0 = pass) or a negative SA_E* code.                                         */
long long sa_selftest_field(size_t count, uint64_t seed);
/* Micro-benchmark: n_threads threads each run `iters` dependent rounds of `ilp`
 * independent operations of kind op (0 montmul, 1 add, 2 sub, 3 butterfly; 4 = blake2b node
 * compressions, 256 threads per block whatever `threads` says, ilp 1 or 2).  Returns the
 * kernel time in milliseconds (negative on error).                                        */
double sa_microbench(int op, int ilp, int iters, int blocks, int threads);

#ifdef __cplusplus
}
#endif
#endif /* SA_B200_H */
