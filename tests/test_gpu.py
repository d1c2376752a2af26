"""GPU parity tests (run on the B200 box: ``pytest -m gpu``).  Every check goes through the
C ABI (include/sa_b200.h) via sa_engine's ctypes binding and is compared bit-exactly with
the CPU oracle on the same seeded inputs, with the reference's golden digests, or through
size-independent properties at BASELINE.json's full sizes."""
import ctypes
import os
import random

import numpy as np
import pytest

import oracle as O
import dropin_cases as C
import sa_engine

pytestmark = pytest.mark.gpu
P = O.P
ROOT_DIR = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def eng():
    sa_engine.set_engine(None)
    e = sa_engine.get_engine()  # raises without CUDA / without the built library
    assert e.name == "cuda"
    return e


@pytest.fixture(autouse=True)
def _cuda_engine(eng):
    sa_engine.set_engine(eng)
    yield


def rand_np(seed, n):
    rng = np.random.default_rng(seed)
    lo = rng.integers(0, 1 << 64, size=n, dtype=np.uint64)
    hi = rng.integers(0, 0xCB80000000000000, size=n, dtype=np.uint64)  # < p's top limb => < p
    return np.stack([lo, hi], axis=1)


def up(eng, arr):
    return eng.upload(np.ascontiguousarray(arr).view(np.int64))


def down(eng, vec):
    return eng.download(vec).view(np.uint64)


def test_field_selftest(eng):
    assert eng.lib.sa_selftest_field(1 << 20, 12345) == 0
    assert eng.lib.sa_selftest_field(1 << 24, 987654321) == 0


def test_ntt_random_campaign(eng):
    """200 random (size, batch, direction, primitive root) combinations against the oracle"""
    rng = random.Random(4242)
    for it in range(200):
        log_n = rng.randrange(1, 15)
        n = 1 << log_n
        batch = rng.choice([1, 1, 2, 3, 5, 8, 13])
        inverse = rng.random() < 0.5
        w = pow(O.primitive_nth_root(n), 2 * rng.randrange(n // 2 if n > 2 else 1) + 1, P)  # odd power: still primitive
        x = rand_np(5000 + it, n * batch)
        if it % 7 == 0:
            x[rng.randrange(n * batch)] = O._fe(P - 1)
            x[rng.randrange(n * batch)] = 0
        got = down(eng, eng.ntt(up(eng, x), log_n, w, inverse=inverse, batch=batch))
        for b in range(batch):
            xb = x[b * n:(b + 1) * n]
            want = O.intt_np(w, xb) if inverse else O.ntt_np(w, xb)
            assert (got[b * n:(b + 1) * n] == want).all(), (it, log_n, batch, inverse)


@pytest.mark.parametrize("log_n", list(range(1, 21)))
def test_ntt_matches_oracle(eng, log_n):
    n = 1 << log_n
    w = O.primitive_nth_root(n)
    for batch in ([1, 3, 17] if log_n <= 12 else [1, 2] if log_n <= 16 else [1]):
        x = rand_np(1000 + log_n, n * batch)
        for inverse in (False, True):
            got = down(eng, eng.ntt(up(eng, x), log_n, w, inverse=inverse, batch=batch))
            for b in range(batch):
                xb = x[b * n:(b + 1) * n]
                want = O.intt_np(w, xb, parallel=True) if inverse else O.ntt_np(w, xb, parallel=True)
                assert (got[b * n:(b + 1) * n] == want).all(), (log_n, batch, inverse, b)


@pytest.mark.parametrize("log_n", [21, 22])
def test_ntt_three_pass_matches_oracle(eng, log_n):
    """above 2^20 the transform is a three-pass n1*n2*n3 split"""
    n = 1 << log_n
    w = O.primitive_nth_root(n)
    x = rand_np(2000 + log_n, n)
    vx = up(eng, x)
    y = eng.ntt(vx, log_n, w)
    assert (down(eng, y) == O.ntt_np(w, x, parallel=True)).all()
    assert bool((eng.ntt(y, log_n, w, inverse=True) == vx).all())


def test_ntt_2_24_roundtrip_in_place(eng):
    log_n = 24
    n = 1 << log_n
    w = O.primitive_nth_root(n)
    x = rand_np(24, n)
    v = up(eng, x)
    ref = v.clone()
    assert eng.lib.sa_ntt(v.data_ptr(), v.data_ptr(), log_n, sa_engine._limbs(w), 0, 1, eng._stream()) == 0
    assert not bool((v == ref).all())
    assert eng.lib.sa_ntt(v.data_ptr(), v.data_ptr(), log_n, sa_engine._limbs(w), 1, 1, eng._stream()) == 0
    assert bool((v == ref).all())
    with pytest.raises(Exception):
        eng.ntt(eng.empty(16), 27, w)


def test_ntt_2_26_maximum_size(eng):
    """the largest supported transform (three passes, 1 GiB per vector): a unit impulse at j must come out
    as c * w^(i*j) (checked at sampled indices with host pow), the all-ones vector as n * e_0, and a random
    vector must survive the round trip - no oracle run at this size"""
    import torch
    log_n = 26
    n = 1 << log_n
    w = O.primitive_nth_root(n)
    root = sa_engine._limbs(w)
    rng = random.Random(26)
    j, c = rng.randrange(n), rng.randrange(1, P)
    v = eng.zeros(n)
    s64 = lambda u: u - (1 << 64) if u >= (1 << 63) else u  # limb as the int64 torch stores
    v[j, 0] = s64(c & 0xFFFFFFFFFFFFFFFF)
    v[j, 1] = s64(c >> 64)
    out = eng.empty(n)
    assert eng.lib.sa_ntt(out.data_ptr(), v.data_ptr(), log_n, root, 0, 1, eng._stream()) == 0
    idx = [0, 1, n - 1, n // 2] + [rng.randrange(n) for _ in range(500)]
    got = eng.gather(out, idx).view(np.uint64)
    for k, i in enumerate(idx):
        want = c * pow(w, (i * j) % n, P) % P
        assert int(got[k][0]) | (int(got[k][1]) << 64) == want, i
    v.zero_()
    v[:, 0] = 1
    assert eng.lib.sa_ntt(out.data_ptr(), v.data_ptr(), log_n, root, 0, 1, eng._stream()) == 0
    assert int(out[0, 0]) == n and int(out[0, 1]) == 0 and not bool(out[1:].any())
    del v
    x = torch.randint(0, 1 << 62, (n, 2), dtype=torch.int64, device=eng.device)
    x[:, 1] &= (1 << 61) - 1
    ref = x.clone()
    assert eng.lib.sa_ntt(x.data_ptr(), x.data_ptr(), log_n, root, 0, 1, eng._stream()) == 0
    assert eng.lib.sa_ntt(x.data_ptr(), x.data_ptr(), log_n, root, 1, 1, eng._stream()) == 0
    assert bool((x == ref).all())


def test_ntt_edge_inputs_and_roots(eng):
    for log_n in (3, 10, 13):
        n = 1 << log_n
        w = O.primitive_nth_root(n)
        for name, x in (("zeros", np.zeros((n, 2), np.uint64)),
                        ("pm1", O.to_np([P - 1] * n)), ("delta", O.to_np([1] + [0] * (n - 1)))):
            assert (down(eng, eng.ntt(up(eng, x), log_n, w)) == O.ntt_np(w, x)).all(), name
        w2 = pow(w, 3, P)  # any primitive root, e.g. the squared roots fast_multiply derives
        x = rand_np(5, n)
        assert (down(eng, eng.ntt(up(eng, x), log_n, w2)) == O.ntt_np(w2, x)).all()
    x = up(eng, rand_np(6, 16))
    with pytest.raises(AssertionError, match="primitive root must be nth root of unity"):
        eng.ntt(x, 4, O.primitive_nth_root(64))
    with pytest.raises(AssertionError, match="not primitive nth root"):
        eng.ntt(x, 4, O.primitive_nth_root(4))


def test_ntt_in_place_and_host_entry(eng):
    import torch
    log_n, batch = 14, 4
    n = 1 << log_n
    w = O.primitive_nth_root(n)
    x = rand_np(77, n * batch)
    v = up(eng, x)
    rc = eng.lib.sa_ntt(v.data_ptr(), v.data_ptr(), log_n, sa_engine._limbs(w), 0, batch, eng._stream())
    assert rc == 0
    want = O.ntt_batch_np(w, x.reshape(batch, n, 2)).reshape(-1, 2)
    assert (down(eng, v) == want).all()
    out = np.zeros_like(x)
    rc = eng.lib.sa_ntt_host(out.ctypes.data, x.ctypes.data, log_n, sa_engine._limbs(w), 0, batch, eng._stream())
    assert rc == 0 and (out == want).all()
    torch.cuda.synchronize()


@pytest.mark.parametrize("log_n,batch,nouts", [(0, 3, 2), (3, 5, 3), (8, 7, 2), (10, 4, 8), (14, 3, 3), (20, 2, 8),
                                               (21, 1, 2)])
def test_ntt_multi_stores_every_destination(eng, log_n, batch, nouts):
    """sa_ntt_multi (multi-GPU assembly, sa_dist "p2p-store"): the last pass stores every result to the same
    offset of all destination buffers.  Here all destinations are on this device (on the 8-GPU box the others
    are peer-mapped buffers of the other ranks, tools/dist_check.py): each must equal the oracle's batch,
    everything outside the written range must stay untouched, forward and inverse."""
    import torch
    n = 1 << log_n
    w = O.primitive_nth_root(n) if n > 1 else 1
    x = rand_np(4000 + log_n, n * batch)
    want = O.ntt_batch_np(w, x.reshape(batch, n, 2)).reshape(-1, 2) if n > 1 else x
    pad = 5 * n + 3
    outs = [torch.full((pad + n * batch + 7, 2), -1, dtype=torch.int64, device=eng.device) for _ in range(nouts)]
    eng.ntt_multi(outs, pad, up(eng, x), log_n, w, batch=batch)
    for o in outs:
        got = down(eng, o)
        assert (got[pad:pad + n * batch] == want).all()
        assert (got[:pad] == np.uint64(2**64 - 1)).all() and (got[pad + n * batch:] == np.uint64(2**64 - 1)).all()
    if n > 1:
        back = [torch.zeros((n * batch, 2), dtype=torch.int64, device=eng.device) for _ in range(nouts)]
        eng.ntt_multi(back, 0, outs[-1][pad:pad + n * batch], log_n, w, inverse=True, batch=batch)
        for b in back:
            assert (down(eng, b) == x).all()
    with pytest.raises(AssertionError, match="unsupported size"):
        eng.ntt_multi(outs * 9, 0, up(eng, x), log_n, w, batch=batch)


def test_peer_buffers_single_process(eng):
    """the library-side pieces of sa_dist.PeerBuffers that one process can exercise: sa_peer_alloc (zeroed cudaMalloc
    + IPC handle), a torch view over it, sa_copy_async, sa_ntt_multi into it, free.  (Opening the handles from the
    other ranks needs several processes: tools/dist_check.py under torchrun.)"""
    import sa_dist
    n, batch = 1 << 12, 4
    pb = sa_dist.PeerBuffers(n * batch)
    assert pb.world == 1 and len(pb.local) == 2 and pb.ptrs[0][0] == pb.local[0].data_ptr()
    assert int(pb.local[0].abs().sum().item()) == 0
    x = rand_np(5150, n * batch)
    w = O.primitive_nth_root(n)
    local, ptrs = pb.next()
    eng.ntt_multi([ptrs[0]], 0, up(eng, x), 12, w, batch=batch)
    want = O.ntt_batch_np(w, x.reshape(batch, n, 2)).reshape(-1, 2)
    assert (down(eng, local) == want).all()
    local2, ptrs2 = pb.next()
    assert ptrs2[0] != ptrs[0]
    eng._check(eng.lib.sa_copy_async(ptrs2[0], ptrs[0], 16 * n * batch, eng._stream()))
    assert (down(eng, local2) == want).all()
    # sa_push: one read, several destinations (here three windows of the second buffer), ragged tail
    import ctypes
    import torch
    local2.zero_()
    nbytes = 16 * (n + 5)
    dsts = (ctypes.c_void_p * 3)(ptrs2[0], ptrs2[0] + 16 * (n + 8), ptrs2[0] + 16 * (2 * n + 16))
    eng._check(eng.lib.sa_push(dsts, 3, ptrs[0], nbytes, eng._stream()))
    got = down(eng, local2)
    for k in range(3):
        o = k * (n + 8)
        assert (got[o:o + n + 5] == want[:n + 5]).all() and (got[o + n + 5:o + n + 8] == 0).all()
    with pytest.raises(AssertionError, match="unsupported size"):
        eng._check(eng.lib.sa_push(dsts, 3, ptrs[0], 24, eng._stream()))
    # one to seven destinations, a length that is not a multiple of the grid stride; the others stay untouched
    for n in (1000, 70001):
        src = torch.randint(0, 1 << 62, (n, 2), dtype=torch.int64, device=eng.device)
        dst = torch.zeros((7 * (n + 3), 2), dtype=torch.int64, device=eng.device)
        for nd in (1, 3, 7):
            dst.zero_()
            ptrs = (ctypes.c_void_p * nd)(*[dst.data_ptr() + 16 * (n + 3) * i for i in range(nd)])
            eng._check(eng.lib.sa_push(ptrs, nd, src.data_ptr(), 16 * n, eng._stream()))
            for i in range(7):
                blk = dst[(n + 3) * i:(n + 3) * (i + 1)]
                assert bool((blk[:n] == src).all()) == (i < nd) and int(blk[n:].abs().sum()) == 0
    full = sa_dist.sharded_ntt(up(eng, x), 12, w, assemble="p2p-store", peers=pb)  # world 1: plain transform
    assert (down(eng, full) == want).all()
    pb.close()


@pytest.mark.parametrize("log_n,batch", [(16, 70), (18, 9), (12, 3), (21, 3), (22, 2)])
def test_ntt_host_entry_chunk_pipeline(eng, log_n, batch):
    """sa_ntt_host cuts a batch into ramped chunks over several copy streams (32 MiB chunks, first and
    last halved): ragged batch sizes, chunk boundaries and the single-chunk path against the oracle"""
    import torch
    n = 1 << log_n
    w = O.primitive_nth_root(n)
    x = rand_np(1200 + log_n, n * batch)
    want = O.ntt_batch_np(w, x.reshape(batch, n, 2)).reshape(-1, 2)
    # buffers from the library's allocator (page-locked, on the GPU's NUMA node)
    nbytes = x.nbytes
    p_in, p_out = eng.lib.sa_host_alloc(nbytes), eng.lib.sa_host_alloc(nbytes)
    assert p_in and p_out, eng.lib.sa_last_error()
    try:
        hx = np.ctypeslib.as_array((ctypes.c_uint64 * (nbytes // 8)).from_address(p_in)).reshape(-1, 2)
        hy = np.ctypeslib.as_array((ctypes.c_uint64 * (nbytes // 8)).from_address(p_out)).reshape(-1, 2)
        hx[:] = x
        for inverse in (0, 1):
            src = p_in if not inverse else p_out
            rc = eng.lib.sa_ntt_host(p_out, src, log_n, sa_engine._limbs(w), inverse, batch, eng._stream())
            assert rc == 0
            if not inverse:
                assert (hy == want).all()
        assert (hy == x).all()  # in-place inverse through the same pipeline
        del hx, hy
    finally:
        assert eng.lib.sa_host_free(p_in) == 0 and eng.lib.sa_host_free(p_out) == 0


@pytest.mark.parametrize("env", [{"SA_HOST_RAMP": "2"}, {"SA_HOST_CHUNK_MIB": "16"},
                                 {"SA_HOST_RAMP": "3", "SA_HOST_CHUNK_MIB": "64", "SA_HOST_STREAMS": "2"}])
def test_ntt_host_entry_pipeline_settings(eng, env):
    """the pipeline knobs are read once per process, so every setting runs in its own interpreter: chunk
    sizes whose ramp start rounds to zero transforms (round 1: an endless loop, ADVICE.md) and transforms
    larger than a chunk must all give the oracle's result"""
    import os
    import subprocess
    import sys
    code = r'''
import sys, ctypes, numpy as np
sys.path[:0] = [%r, %r]
import sa_engine, oracle as O
eng = sa_engine.get_engine()
for log_n, batch in ((20, 5), (21, 2), (16, 33)):
    n = 1 << log_n
    w = O.primitive_nth_root(n)
    rng = np.random.default_rng(log_n)
    x = np.stack([rng.integers(0, 1 << 64, size=n * batch, dtype=np.uint64),
                  rng.integers(0, 0xCB80000000000000, size=n * batch, dtype=np.uint64)], axis=1)
    out = np.zeros_like(x)
    rc = eng.lib.sa_ntt_host(out.ctypes.data, x.ctypes.data, log_n, sa_engine._limbs(w), 0, batch, None)
    assert rc == 0, rc
    assert (out == O.ntt_batch_np(w, x.reshape(batch, n, 2)).reshape(-1, 2)).all(), (log_n, batch)
print("PIPELINE_OK")
''' % (os.path.join(ROOT_DIR, "stark-anatomy_b200"), os.path.join(ROOT_DIR, "oracle"))
    out = subprocess.run([sys.executable, "-c", code], text=True, capture_output=True, timeout=600,
                         env=dict(os.environ, **env))
    assert "PIPELINE_OK" in out.stdout, out.stdout[-1000:] + out.stderr[-3000:]


def test_table_cache_is_bounded(eng):
    """1000 distinct roots (fast_multiply's order shrinking makes new ones all the time) must not grow
    HBM without bound: the plan / x^-1 table cache is an LRU bounded by sa_cache_limit"""
    import torch
    lib = eng.lib
    log_n, n = 12, 1 << 12
    base = O.primitive_nth_root(n)
    x = up(eng, rand_np(5, n))
    want0 = O.ntt_np(base, down(eng, x))
    limit = 4 << 20
    lib.sa_cache_limit(limit)
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    try:
        for k in range(1000):
            root = pow(base, 2 * k + 1, P)  # odd powers: 1000 distinct primitive n-th roots
            out = eng.ntt(x, log_n, root)
            assert lib.sa_cache_bytes() <= limit
            if k % 250 == 0:
                assert (down(eng, out) == O.ntt_np(root, down(eng, x))).all()
        torch.cuda.synchronize()
        assert free0 - torch.cuda.mem_get_info()[0] < 64 << 20  # (1000 plans would be ~100 MiB)
        assert (down(eng, eng.ntt(x, log_n, base)) == want0).all()  # an evicted plan is simply rebuilt
        assert lib.sa_cache_limit(0) == 0 and lib.sa_cache_bytes() == 0
    finally:
        lib.sa_cache_limit(4 << 30)
    assert lib.sa_release_workspaces() == 0
    assert (down(eng, eng.ntt(x, log_n, base)) == want0).all()


def test_ntt_host_entry_from_two_threads(eng):
    """two host threads in sa_ntt_host at once: the copy streams and their device buffers belong to one
    call at a time (per-device mutex), so both results must still be exact"""
    import threading
    log_n, batch = 18, 12  # 48 MiB per call: several pipelined chunks
    n = 1 << log_n
    w = O.primitive_nth_root(n)
    xs = [rand_np(1300 + i, n * batch) for i in range(2)]
    outs = [np.zeros_like(xs[0]), np.zeros_like(xs[1])]
    rcs = [None, None]

    def work(i):
        for _ in range(3):
            rcs[i] = eng.lib.sa_ntt_host(outs[i].ctypes.data, xs[i].ctypes.data, log_n, sa_engine._limbs(w), 0, batch, None)
    ts = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    for i in range(2):
        assert rcs[i] == 0
        assert (outs[i] == O.ntt_batch_np(w, xs[i].reshape(batch, n, 2)).reshape(-1, 2)).all()


def test_ntt_two_streams_and_threads(eng):
    """independent work on two CUDA streams from two host threads (per-stream workspaces, shared
    plan cache behind a mutex): results equal the oracle's"""
    import threading
    import torch
    log_n, batch = 16, 4
    n = 1 << log_n
    w = O.primitive_nth_root(n)
    xs = [rand_np(900 + i, n * batch) for i in range(2)]
    outs = [None, None]

    def work(i):
        st = torch.cuda.Stream()
        with torch.cuda.stream(st):
            v = up(eng, xs[i])
            for _ in range(20):  # keep both streams busy at the same time
                y = eng.ntt(v, log_n, w, batch=batch)
                v = eng.ntt(y, log_n, w, inverse=True, batch=batch)
            outs[i] = down(eng, eng.ntt(v, log_n, w, batch=batch))
        st.synchronize()
    ts = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    for i in range(2):
        want = O.ntt_batch_np(w, xs[i].reshape(batch, n, 2)).reshape(-1, 2)
        assert (outs[i] == want).all()


def test_ntt_2_20_golden_digest_and_roundtrip(eng):
    C.case_ntt_digests(1 << 20)


def test_ntt_2_20_batch_properties(eng):
    """full-size, size-independent properties: round trip and linearity on a batch of 2^20 transforms"""
    log_n, batch = 20, 4
    n = 1 << log_n
    w = O.primitive_nth_root(n)
    x = rand_np(21, n * batch)
    vx = up(eng, x)
    y = eng.ntt(vx, log_n, w, batch=batch)
    back = eng.ntt(y, log_n, w, inverse=True, batch=batch)
    assert bool((back == vx).all())
    # ntt(a) + ntt(b) == ntt(a + b) on the first two batch items (sum taken by the oracle's field add)
    a, b = x[:n], x[n:2 * n]
    s = O.to_np([(u + v) % P for u, v in zip(O.from_np(a[:4096]), O.from_np(b[:4096]))])
    ya, yb = down(eng, y[:n]), down(eng, y[n:2 * n])
    full_sum = O.pointwise_mul_np(np.ascontiguousarray(a), O.to_np([1] * n))  # copy through the oracle
    assert (full_sum == a).all()
    got_sum = down(eng, eng.ntt(up(eng, _field_add(a, b)), log_n, w))
    assert (got_sum == _field_add(ya, yb)).all()
    assert (s == _field_add(a[:4096], b[:4096])).all()


def _field_add(a, b):
    """vectorised (a + b) mod p on uint64[n,2] (numpy, test-side helper)"""
    alo, ahi = a[:, 0].astype(object), a[:, 1].astype(object)
    blo, bhi = b[:, 0].astype(object), b[:, 1].astype(object)
    s = (alo + (ahi << 64)) + (blo + (bhi << 64))
    s = np.where(s >= P, s - P, s)
    return np.stack([(s & 0xFFFFFFFFFFFFFFFF).astype(np.uint64), (s >> 64).astype(np.uint64)], axis=1)


def test_elementwise_ops(eng):
    for n in (1, 7, 1000, 1 << 16):
        a, b = rand_np(31, n), rand_np(32, n)
        b[b.sum(axis=1) == 0] = 1
        assert (down(eng, eng.pointwise_mul(up(eng, a), up(eng, b))) == O.pointwise_mul_np(a, b)).all()
        if n <= 1 << 12:
            assert (down(eng, eng.pointwise_div(up(eng, a), up(eng, b))) == O.pointwise_div_np(a, b)).all()
        f = random.Random(n).randrange(P)
        assert (down(eng, eng.scale(up(eng, a), f)) == O.scale_np(a, f)).all()
    a, b = rand_np(33, 4096), rand_np(34, 4096)
    b[1234] = 0
    with pytest.raises(AssertionError, match="divide by zero"):
        eng.pointwise_div(up(eng, a), up(eng, b))
    coeffs, pts = rand_np(35, 300), rand_np(36, 517)
    assert (down(eng, eng.poly_eval(up(eng, coeffs), up(eng, pts))) == O.poly_eval_np(coeffs, pts)).all()


@pytest.mark.parametrize("k", [1, 2, 3, 17, 284, 512, 513, 1000, 1024, 1025, 1500, 2048, 4096, 5000])
def test_zerofier_and_interpolate(eng, k):
    """sa_zerofier / sa_interpolate vs the oracle: the one-CTA / k x k kernels (k <= 512 / 1024) and the
    device subproduct tree above them (full and ragged trees: 513, 1025, 1500, 5000 points)"""
    dom = rand_np(70 + k, k)
    vals = rand_np(71 + k, k)
    z = down(eng, eng.zerofier(up(eng, dom)))
    assert z.shape[0] == k + 1 and (z == O.zerofier_np(dom)).all()
    if k <= 1500:
        got = down(eng, eng.interpolate(up(eng, dom), up(eng, vals)))
        assert got.shape[0] == k and (got == O.interpolate_np(dom, vals)).all()
    else:  # property check, the interpolant takes the prescribed values
        poly = eng.interpolate(up(eng, dom), up(eng, vals))
        assert (down(eng, eng.poly_eval(poly, up(eng, dom))) == vals).all()
        assert (down(eng, eng.poly_eval(up(eng, z), up(eng, dom))) == 0).all()
    if k >= 3:
        dom[k - 1] = dom[0]
        with pytest.raises(AssertionError, match="divide by zero"):
            eng.interpolate(up(eng, dom), up(eng, vals))


@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 8, 9, 17, 100, 256, 257, 513, 1000, 4097])
def test_poly_eval_tree_walk_matches_oracle(eng, k):
    """fast_evaluate's values (ntt.py:82-100) through the walk down the subproduct tree (sa_poly_eval_mode 2: the
    transposed interpolation tree, no divisions) vs the oracle's Horner: full and ragged trees, fewer / as many /
    more coefficients than points, the zero and constant polynomials, repeated points"""
    pts = rand_np(300 + k, k)
    if k >= 3:
        pts[k - 1] = pts[0]  # a repeated point is fine for evaluation
    for ncoef in sorted({1, 2, max(1, k - 1), k, k + 7, 3 * k + 1, 1 << (k.bit_length())}):
        coeffs = rand_np(400 + k + ncoef, ncoef)
        if ncoef > 2:
            coeffs[ncoef - 1] = 0  # a leading zero
        got = down(eng, eng.poly_eval(up(eng, coeffs), up(eng, pts), mode=2))
        assert (got == O.poly_eval_np(coeffs, pts)).all(), (k, ncoef)
        assert (got == down(eng, eng.poly_eval(up(eng, coeffs), up(eng, pts), mode=1))).all()
    zero = np.zeros((5, 2), dtype=np.uint64)
    assert (down(eng, eng.poly_eval(up(eng, zero), up(eng, pts), mode=2)) == 0).all()


@pytest.mark.parametrize("k,ncoef", [(1 << 15, 1 << 15), ((1 << 16) + 12345, 1 << 16), (1 << 14, (1 << 17) + 3),
                                     (1 << 18, 1 << 18)])
def test_poly_eval_tree_walk_large(eng, k, ncoef):
    """the size the library switches to the walk by itself (>= 2^29 coefficient-point products): the walk's values
    equal the Horner kernel's on a sample of the points and the oracle's on a few"""
    coeffs, pts = rand_np(500 + k % 89, ncoef), rand_np(501 + k % 89, k)
    vc, vp = up(eng, coeffs), up(eng, pts)
    got = eng.poly_eval(vc, vp)  # mode 0: the library's own choice at this size is the walk
    assert (down(eng, got) == down(eng, eng.poly_eval(vc, vp, mode=2))).all()
    step = max(1, k // 4096)
    assert (down(eng, got[::step].contiguous()) == down(eng, eng.poly_eval(vc, vp[::step].contiguous(), mode=1))).all()
    few = [0, 1, k // 2, k - 1]
    assert (down(eng, got)[few] == O.poly_eval_np(coeffs, pts[few])).all()


@pytest.mark.parametrize("k", [1 << 16, (1 << 16) + 12345, 1 << 18])
def test_zerofier_and_interpolate_large_by_property(eng, k):
    """one C call each at sizes the oracle's O(k^2) loops cannot reach: the zerofier is monic, vanishes on
    the domain, equals the product of the zerofiers of the two halves (fast_multiply, ntt.py:76-80); the
    interpolant has degree < k and takes the prescribed values (Horner kernel on the device)"""
    dom = rand_np(170 + k % 97, k)
    vals = rand_np(171 + k % 97, k)
    vd = up(eng, dom)
    z = eng.zerofier(vd)
    zh = down(eng, z)
    assert zh.shape[0] == k + 1 and (zh[k] == np.array([1, 0], dtype=np.uint64)).all()
    sample = vd if k <= 1 << 16 else vd[::37].contiguous()
    assert (down(eng, eng.poly_eval(z, sample)) == 0).all()
    half = k // 2
    zl, zr = eng.zerofier(vd[:half].contiguous()), eng.zerofier(vd[half:].contiguous())
    log_n = k.bit_length() + 1  # > deg(zl * zr)
    n = 1 << log_n
    w = O.primitive_nth_root(n)
    prod = eng.ntt(eng.pointwise_mul(eng.ntt(eng.pad(zl, n), log_n, w), eng.ntt(eng.pad(zr, n), log_n, w)), log_n, w,
                   inverse=True)
    assert (down(eng, prod)[:k + 1] == zh).all() and (down(eng, prod)[k + 1:] == 0).all()
    if k <= (1 << 16) + 12345:
        poly = eng.interpolate(vd, up(eng, vals))  # (M'(d_i) through the walk down the tree at this size)
        assert eng.length(poly) == k
        assert (down(eng, eng.poly_eval(poly, vd)) == vals).all()
        step = 53  # ... and independently of the walk: the Horner kernel on a sample of the points
        assert (down(eng, eng.poly_eval(poly, vd[::step].contiguous(), mode=1)) == vals[::step]).all()


@pytest.mark.parametrize("log_n", [0, 1, 2, 5, 6, 7, 9, 10, 11, 13, 14, 15, 16, 17, 18])
def test_merkle_tree_and_open(eng, log_n):
    n = 1 << log_n
    x = rand_np(50 + log_n, n)
    x[0] = 0
    if n > 4:
        x[1] = (7, 0)
        x[2] = O._fe(10**19)
        x[3] = O._fe(P - 1)
    tree = eng.merkle_tree(up(eng, x))
    want = O.merkle_tree_np(x)
    assert (tree.cpu().numpy()[1:] == want[1:]).all()
    assert eng.tree_root(tree) == want[1].tobytes()
    if n >= 2:
        idx = sorted({0, 1, n // 2, n - 1, random.Random(log_n).randrange(n)})
        assert eng.merkle_open(tree, idx) == [O.merkle_open(want, i) for i in idx]
        assert (eng.gather(up(eng, x), idx).view(np.uint64) == x[idx]).all()
        with pytest.raises(AssertionError, match="cannot open invalid index"):
            eng.merkle_open(tree, [n])


def test_merkle_tree_2_22_composes_from_halves(eng):
    """beyond the oracle's reach: the root over 2^22 leaves must be blake2b(root(left half) || root(right
    half)), every level-1 node of the big tree must be the root of the corresponding half, and an opened
    path must hash back to the root"""
    import hashlib
    import torch
    n = 1 << 22
    x = torch.randint(0, 1 << 62, (n, 2), dtype=torch.int64, device=eng.device)
    x[:, 1] &= (1 << 61) - 1
    big = eng.merkle_tree(x)
    left, right = eng.merkle_tree(x[:n // 2]), eng.merkle_tree(x[n // 2:])
    rl, rr = eng.tree_root(left), eng.tree_root(right)
    assert bytes(big[2].cpu().numpy().tobytes()) == rl and bytes(big[3].cpu().numpy().tobytes()) == rr
    assert eng.tree_root(big) == hashlib.blake2b(rl + rr).digest()
    i = 2718281
    path = eng.merkle_open(big, [i])[0]
    v = eng.gather(x, [i]).view(np.uint64)[0]
    acc = hashlib.blake2b(str(int(v[0]) | (int(v[1]) << 64)).encode()).digest()
    k = i
    for sib in path:
        acc = hashlib.blake2b(sib + acc if k & 1 else acc + sib).digest()
        k >>= 1
    assert acc == eng.tree_root(big)


def test_fri_commit_2_22_layers_fold_correctly(eng):
    """14 rounds on a 2^22 codeword (four times the golden case): every layer must be the split-and-fold
    of the previous one (fri.py:85, checked at sampled indices with host integers) and every published
    root must be node 1 of the retained tree"""
    import torch
    n, rounds = 1 << 22, 14
    omega, off = O.primitive_nth_root(n), O.GENERATOR
    rng = random.Random(2222)
    alphas = [rng.randrange(P) for _ in range(rounds)]
    cw = torch.randint(0, 1 << 62, (n, 2), dtype=torch.int64, device=eng.device)
    cw[:, 1] &= (1 << 61) - 1
    roots = []
    layers, trees = eng.fri_commit(cw, rounds, off, omega, lambda r, root, want: (roots.append(root), alphas[r])[1])
    assert len(layers) == rounds and len(roots) == rounds
    inv2 = pow(2, P - 2, P)
    val = lambda row: int(row[0]) | (int(row[1]) << 64)
    o, w, ln = off, omega, n
    for r in range(rounds):
        assert eng.tree_root(trees[r]) == roots[r]
        if r + 1 < rounds:
            half = ln // 2
            idx = [0, half - 1] + [rng.randrange(half) for _ in range(30)]
            a = eng.gather(layers[r], idx).view(np.uint64)
            b = eng.gather(layers[r], [i + half for i in idx]).view(np.uint64)
            c = eng.gather(layers[r + 1], idx).view(np.uint64)
            for k, i in enumerate(idx):
                t = alphas[r] * pow(o * pow(w, i, P) % P, P - 2, P) % P
                want = inv2 * ((1 + t) * val(a[k]) + (1 - t) * val(b[k])) % P
                assert val(c[k]) == want, (r, i)
            o, w, ln = o * o % P, w * w % P, half


def test_merkle_root_2_20_golden(eng):
    from conftest import load_golden
    c = [m for m in load_golden("merkle.json")["commit"] if m["n"] == 1 << 20][0]
    xs = C.seeded(1, 1 << 20)
    import sa_marshal
    tree = eng.merkle_tree(eng.upload(sa_marshal.pack(xs)))
    assert eng.tree_root(tree).hex() == c["root"]


@pytest.mark.parametrize("log_n", [1, 2, 6, 7, 8, 10, 11, 14, 15, 16, 17, 18])
def test_fri_round_and_fold(eng, log_n):
    n = 1 << log_n
    x = rand_np(60 + log_n, n)
    rng = random.Random(log_n)
    alpha, omega, off = rng.randrange(P), O.primitive_nth_root(n), O.GENERATOR
    want = O.fri_fold_np(x, alpha, off, omega)
    assert (down(eng, eng.fri_fold(up(eng, x), alpha, off, omega)) == want).all()
    nxt, tree = eng.fri_round(up(eng, x), alpha, off, omega)
    assert (down(eng, nxt) == want).all()
    assert (tree.cpu().numpy()[1:] == O.merkle_tree_np(want)[1:]).all()


def test_merkle_and_fri_commit_two_streams_and_threads(eng):
    """Merkle trees and whole FRI commits from two host threads on two streams at once: the fused-top
    arrival counter is per stream and the mapped root landing pad per thread, so neither may leak
    into the other's results"""
    import threading
    import torch
    log_n = 13
    n = 1 << log_n
    omega, off = O.primitive_nth_root(n), O.GENERATOR
    xs = [rand_np(700 + i, n) for i in range(2)]
    alphas = [[random.Random(710 + i).randrange(P) for _ in range(8)] for i in range(2)]
    got = [{"roots": [], "trees": []}, {"roots": [], "trees": []}]
    errs = []

    def work(i):
        try:
            st = torch.cuda.Stream()
            with torch.cuda.stream(st):
                v = up(eng, xs[i])
                for rep in range(10):
                    roots = []
                    eng.fri_commit(v, 8, off, omega, lambda r, root, want: (roots.append(root), alphas[i][r])[1])
                    got[i]["roots"].append(roots)
                    got[i]["trees"].append(eng.merkle_tree(v).cpu().numpy())
            st.synchronize()
        except BaseException as exc:  # surfaces in the main thread
            errs.append(exc)
    ts = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errs, errs
    for i in range(2):
        cw, o, w, want_roots = xs[i], off, omega, []
        for r in range(8):
            want_roots.append(O.merkle_tree_np(cw)[1].tobytes())
            if r < 7:
                cw = O.fri_fold_np(cw, alphas[i][r], o, w)
                o, w = o * o % P, w * w % P
        want_tree = O.merkle_tree_np(xs[i])
        for rep in range(10):
            assert got[i]["roots"][rep] == want_roots
            assert (got[i]["trees"][rep][1:] == want_tree[1:]).all()


# ---- the drop-in modules on the real engine, against the reference's golden outputs -------
def test_dropin_ntt_vectors(eng):
    C.case_ntt_vectors()
    C.case_ntt_asserts()


def test_dropin_poly(eng):
    C.case_poly()
    C.case_poly_asserts()


def test_dropin_poly_split_recursion(eng):
    C.case_poly_split_recursion()


def test_dropin_fast_multiply_digests(eng):
    C.case_fast_multiply_big(1 << 12)
    C.case_fast_multiply_big(1 << 20)  # BASELINE.md section 3 (654 s of reference time)


def test_dropin_fri_commit(eng):
    C.case_fri_commit(1 << 12)


def test_dropin_fri_commit_2_20_golden_roots(eng):
    C.case_fri_commit_2_20()  # BASELINE.md section 3 (73.1 s of reference time)


def test_fri_commit_callback_error_aborts_cleanly(eng):
    """a challenge callback that raises in the middle of a commit aborts it with that exception, and the engine
    stays usable"""
    n = 1 << 12
    rng = np.random.default_rng(9)
    cw = eng.upload(np.stack([rng.integers(0, 1 << 64, size=n, dtype=np.uint64),
                              rng.integers(0, 0xCB80000000000000, size=n, dtype=np.uint64)], axis=1).view(np.int64))

    class Boom(Exception):
        pass

    def on_root(r, root, want):
        if r == 3:
            raise Boom()
        return 12345

    with pytest.raises(Boom):
        eng.fri_commit(cw, 8, O.GENERATOR, O.primitive_nth_root(n), on_root)
    eng.synchronize()
    C.case_fri_commit(1 << 12)


def test_dropin_fri_prove_and_verify(eng):
    C.case_fri_prove(1 << 12)


def test_dropin_faststark_trace_replay(eng):
    C.case_faststark_trace_replay()


def test_dropin_recorded_faststark_and_rpsss_runs(eng):
    """the recorded calls of fast_stark.py's prove + verify and of fast_rpsss.py's keygen / sign / verify,
    replayed on the CUDA engine: the same proof and signature bytes as the pure reference"""
    C.case_faststark_proof_replay()
    C.case_rpsss_replay()


def test_dropin_merkle_class(eng):
    C.case_merkle_class()


def test_dropin_accel_polymul(eng):
    C.case_accel_polymul()


def test_dropin_device_list(eng):
    C.case_device_list()


def test_config5_unmodified_faststark_and_rpsss_on_the_cuda_engine(eng):
    """BASELINE config 5 on the real engine: the reference's fast_stark.py / fast_rpsss.py, unmodified (from
    the checkout whose code/ directory STARK_REFERENCE names; skipped without one), on top of the
    drop-in.  The seeded proof and the seeded signature must be the bytes the pure
    reference produced (tests/golden/faststark_trace.json, rpsss.json) and must verify; between
    fast_coset_evaluate and Fri.prove no 2^k-element list may cross the PCIe link (section 8 f3)."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    tool = os.path.join(root, "tools", "config5.py")
    out = subprocess.run([sys.executable, tool], text=True, capture_output=True, timeout=1500)
    res = json.loads(out.stdout[out.stdout.index("{"):]) if "{" in out.stdout else {}
    if res.get("unavailable"):
        pytest.skip(res["unavailable"])
    fs = res["faststark"]
    assert "error" not in fs, fs
    assert fs["byte_identical"] and fs["verify"] is True, fs
    for key in ("rpsss", "rpsss_accel"):
        r = res[key]
        assert "error" not in r, r
        assert r["byte_identical"], (key, r["signature_sha256"], r["golden_signature_sha256"])
        assert r["verify"] is True and r["verify_second"] is True and r["verify_other_document"] is False
        # what crossed the link during one sign: coefficient lists going up (each <= 1024 elements, far
        # fewer bytes than ONE 4096-element codeword per commitment would be), small trees / vectors coming down
        st = r["engine_during_sign"]
        if key == "rpsss":  # (with sa_accel the caller's Polynomial products upload their operands as well)
            assert st["h2d_bytes"] < 8 * 4096 * 16, st
    assert res["rpsss_accel"]["seconds"]["sign_warm"] < res["rpsss_accel"]["reference_seconds"]["sign"]


def test_dropin_reference_style_properties(eng):
    C.case_reference_style_properties(trials=20)


def test_kernels_were_launched(eng):
    assert eng.launch_count() > 100
