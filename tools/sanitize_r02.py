#!/usr/bin/env python3
"""Small-size exercise of round 2's new kernels for compute-sanitizer (memcheck / racecheck): TF_PEERS tile variants
(sa_ntt_multi), PDL launches, the subproduct tree (k_tree_*), the walk down it (sa_poly_eval_mode 2), sa_push, the FRI commit,
device lists.  Every result is checked against the oracle."""
import ctypes
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "stark-anatomy_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"), ROOT]
import numpy as np  # noqa: E402
import torch  # noqa: E402
import oracle as O  # noqa: E402
import sa_engine  # noqa: E402

eng = sa_engine.get_engine()


def rand(seed, n):
    rng = np.random.default_rng(seed)
    return np.stack([rng.integers(0, 1 << 64, size=n, dtype=np.uint64),
                     rng.integers(0, 0xCB80000000000000, size=n, dtype=np.uint64)], axis=1)


def up(a):
    return eng.upload(np.ascontiguousarray(a).view(np.int64))


def down(v):
    return eng.download(v).view(np.uint64)


# transforms incl. the peer-store variants (several destinations on this device) and a 2-pass size
for log_n, batch, nouts in ((6, 5, 3), (10, 3, 2), (12, 2, 3)):
    n = 1 << log_n
    x = rand(log_n, n * batch)
    w = O.primitive_nth_root(n)
    want = O.ntt_batch_np(w, x.reshape(batch, n, 2)).reshape(-1, 2)
    outs = [torch.zeros((n * batch + 9, 2), dtype=torch.int64, device=eng.device) for _ in range(nouts)]
    eng.ntt_multi(outs, 4, up(x), log_n, w, batch=batch)
    for o in outs:
        assert (down(o)[4:4 + n * batch] == want).all()
    assert (down(eng.ntt(eng.ntt(up(x), log_n, w, batch=batch), log_n, w, inverse=True, batch=batch)) == x).all()
print("transforms ok", flush=True)

# subproduct tree: ragged and full
for k in (600, 1024, 1100):
    dom, vals = rand(70 + k, k), rand(71 + k, k)
    z = down(eng.zerofier(up(dom)))
    assert (z == O.zerofier_np(dom)).all()
    if k >= 1100:
        got = down(eng.interpolate(up(dom), up(vals)))
        assert (got == O.interpolate_np(dom, vals)).all()
print("tree ok", flush=True)

# multi-point evaluation by the walk down the transposed tree (k_series_*, k_eval_*, k_tree_down*): ragged and full
# trees, fewer / more coefficients than points
for k, ncoef in ((1, 1), (5, 3), (64, 64), (100, 257), (600, 599), (1030, 2100)):
    pts, coeffs = rand(90 + k, k), rand(91 + k, ncoef)
    got = down(eng.poly_eval(up(coeffs), up(pts), mode=2))
    assert (got == O.poly_eval_np(coeffs, pts)).all(), (k, ncoef)
print("walk ok", flush=True)

# push kernel
src = up(rand(5, 1000))
dst = torch.zeros((3 * 1008, 2), dtype=torch.int64, device=eng.device)
ptrs = (ctypes.c_void_p * 3)(*[dst.data_ptr() + 16 * 1008 * i for i in range(3)])
eng._check(eng.lib.sa_push(ptrs, 3, src.data_ptr(), 16 * 1000, eng._stream()))
got = down(dst)
for i in range(3):
    assert (got[1008 * i:1008 * i + 1000] == down(src)).all()
print("push ok", flush=True)

# FRI commit + device lists through the drop-in
import dropin_cases as C  # noqa: E402
C.case_fri_commit(1 << 10)
C.case_device_list()
print("fri / device lists ok", flush=True)
