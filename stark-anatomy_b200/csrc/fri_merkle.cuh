// fri_merkle.cuh -- per-thread pieces of the FRI round kernel: split-and-fold
// (code/fri.py:85) and the chunked Merkle reduction (code/merkle.py:6-14).
// __host__ __device__ so tests/emu can drive the same code phase by phase.
#pragma once
#include "field.cuh"
#include "hash.cuh"

namespace sa {

constexpr int MK_THREADS = 256;  // threads per Merkle CTA
constexpr int MK_MAX_IPT_LOG = 3;  // a thread reduces at most 8 bottom nodes privately

// c'[i] = 2^-1 (a + b) + (alpha * 2^-1 * x_i^-1) (a - b)   ==  fri.py:85
//   inv2_m : 2^-1 in Montgomery form
//   t_m    : alpha * 2^-1 * (offset * omega^i)^-1 in Montgomery form
SA_HD fe fri_fold_one(const fe &a, const fe &b, const fe &t_m, const fe &inv2_m) {
    const fe s = fe_montmul(fe_add(a, b), inv2_m);
    const fe d = fe_montmul(fe_sub(a, b), t_m);
    return fe_add(s, d);
}

SA_HD fe merkle_ld_stream(const fe *p) {
#if defined(__CUDA_ARCH__)
    const uint4 v = __ldcg(reinterpret_cast<const uint4 *>(p));
    return fe_make(v.x, v.y, v.z, v.w);
#else
    return *p;
#endif
}

struct MerkleArgs {
    uint64_t *tree;      // heap layout, 8 words per node
    long long width;     // number of bottom nodes of this launch
    int chunk;           // bottom nodes per CTA (power of two, <= MK_THREADS << ipt_log)
    int ipt_log;         // log2 of the bottom nodes one thread reduces privately (0..3)
    int red_log;         // tree levels the CTA then reduces through shared memory (0..log2(chunk) - ipt_log);
                         // the launch leaves width >> (ipt_log + red_log) digests for the next one
    int coop_max;        // shared-memory levels of at most this many nodes are hashed four lanes per node
    int mode;            // 0: bottom digests already in tree; 1: leaves from `values`; 2: leaves from a fold
    const fe *values;    // mode 1: the codeword (width elements)
    const fe *prev;      // mode 2: the codeword being folded (2 * width elements)
    fe *next;            // mode 2: receives the folded codeword (width elements)
    const fe *xinv;      // mode 2: xinv[i] = omega^-i in Montgomery form, i < width
    fe s_m;              // mode 2: alpha * 2^-1 * offset^-1 in Montgomery form
    fe inv2_m;           // mode 2: 2^-1 in Montgomery form
    unsigned int *ticket;  // optional: CTA arrival counter (zero between launches); the CTA that arrives last
                         // also reduces the gridDim.x (<= MK_THREADS) subtree roots, saving a launch
    uint64_t *root_out;  // last launch of a tree, optional: host-mapped landing pad, receives the root
    unsigned long long root_seq;  // (8 words) and then this sequence number in word 8
};

// launch shape for a level of `width` bottom nodes: small levels are latency bound (one node per
// thread, 64..256-node CTAs so that 128-256 CTAs are in flight, each reducing its chunk to one digest); big ones are
// throughput bound: four leaves and their three parents per thread, barrier free, then only the three
// shared-memory levels that still fill whole warps (128, 64, 32 nodes) - the 32 digests a CTA leaves
// are picked up by the next launch, so no SM sits in a mostly idle dependency chain while thousands
// of leaves wait (profiles/r01g_merkle_shapes.txt)
SA_HD int merkle_log2(long long x) {
    int l = 0;
    while ((1ll << l) < x) l++;
    return l;
}
SA_HD void merkle_shape(MerkleArgs &a) {
    a.coop_max = MK_THREADS / 4;  // latency bound: a level of <= 64 nodes keeps all 256 lanes busy that way
    a.ipt_log = 0;
    if (a.width <= 64) {  // one CTA finishes the tree
        a.chunk = (int)a.width;
    } else if (a.width < (1 << 14)) {
        // dependency-chain regime, measured (profiles/r01g_merkle_small_shapes.txt): few leaves per CTA
        // spread the leaf hashes (a warp-wide compression occupies its scheduler for 2.3 us whatever
        // the number of active lanes) over many SMs, and the CTA that arrives last reduces the <= 256
        // subtree roots, so the tree is still one launch
        a.chunk = 64;
    } else if (a.width < (1 << 15)) {
        a.chunk = 128;
    } else if (a.width < (1 << 16)) {
        a.chunk = MK_THREADS;
    } else if (a.width < (1 << 18)) {
        a.ipt_log = 1;
        a.chunk = MK_THREADS << 1;
    } else {  // throughput bound
        a.ipt_log = 2;
        a.chunk = MK_THREADS << 2;
        a.red_log = 3;
        a.coop_max = 0;  // one thread per node issues fewer instructions per node
        return;
    }
    a.red_log = merkle_log2(a.chunk) - a.ipt_log;  // each CTA reduces its chunk to one digest
}
// width of the level a launch of shape `a` leaves behind
SA_HD long long merkle_next_width(const MerkleArgs &a) { return a.width >> (a.ipt_log + a.red_log); }

// digest of bottom node g of this launch: loads it (mode 0) or hashes the leaf (modes 1, 2) and
// writes it to the tree (and next[] in mode 2)
SA_HD void merkle_bottom(uint64_t d[8], const MerkleArgs &a, long long g) {
    uint64_t *node = a.tree + (a.width + g) * 8;
    if (a.mode == 0) {
        for (int i = 0; i < 8; i++) d[i] = node[i];
        return;
    }
    fe v;
    if (a.mode == 1) {
        v = a.values[g];
    } else {
        const fe t_m = fe_montmul(a.xinv[g], a.s_m);
        // (.cg: each element of the previous layer is read exactly once, so there is nothing to cache in L1)
        v = fri_fold_one(merkle_ld_stream(a.prev + g), merkle_ld_stream(a.prev + a.width + g), t_m, a.inv2_m);
        a.next[g] = v;
    }
    merkle_leaf_digest(d, v);
    for (int i = 0; i < 8; i++) node[i] = d[i];
}

// Private phase of thread t of CTA blk: reduce its 2^ipt_log bottom nodes to one digest (streaming:
// a slot per height), writing every node it creates to the tree.  root = the subtree digest.
SA_HD void merkle_private(uint64_t root[8], const MerkleArgs &a, long long blk, int t) {
    uint64_t slot[MK_MAX_IPT_LOG][8];
    const int ipt = 1 << a.ipt_log;
    uint64_t d[8];
    for (int j = 0; j < ipt; j++) {
        const long long g = blk * a.chunk + (long long)t * ipt + j;
        merkle_bottom(d, a, g);
        long long idx = a.width + g;
        int h = 0;
        while ((j >> h) & 1) {  // a left sibling of this height is waiting: combine
            uint64_t l[8];
            for (int i = 0; i < 8; i++) l[i] = slot[h][i];
            merkle_node_digest(d, l, d);
            idx >>= 1;
            for (int i = 0; i < 8; i++) a.tree[idx * 8 + i] = d[i];
            h++;
        }
        if (h < a.ipt_log)
            for (int i = 0; i < 8; i++) slot[h][i] = d[i];
    }
    for (int i = 0; i < 8; i++) root[i] = d[i];
}

}  // namespace sa
