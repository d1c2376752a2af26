"""sa_engine -- ctypes binding of the C ABI (include/sa_b200.h) plus device memory.

This is the "reference-side binding a maintainer would add" (INTEGRATION.md):
plain pointers and sizes go to ``libsa_b200.so``; PyTorch is used only for
device memory (``torch.empty(..., device="cuda")``), host<->device copies and the
current CUDA stream.  There is no CPU fallback: creating the engine without a
CUDA device or without the built library raises.

Vectors are ``torch.int64`` tensors of shape [n, 2] on the GPU holding the
(lo, hi) limbs of canonical residues mod p = 1 + 407*2^119 (16 bytes/element).
"""
import ctypes
import os

P = 1 + 407 * (1 << 119)
_HERE = os.path.dirname(os.path.abspath(__file__))
# SA_B200_LIB: another build of the same C ABI (kernel experiments); default = the in-tree library
LIB_PATH = os.environ.get("SA_B200_LIB") or os.path.join(_HERE, "libsa_b200.so")

# include/sa_b200.h error codes -> the reference's assertion messages
SA_ERRORS = {
    -1: "cannot compute ntt of non-power-of-two sequence",                                   # ntt.py:4
    -2: "primitive root must be nth root of unity, where n is len(values)",                  # ntt.py:10
    -3: "primitive root is not primitive nth root of unity, where n is len(values)",         # ntt.py:11
    -4: "divide by zero",                                                                    # algebra.py:92
    -5: "cannot open invalid index",                                                         # merkle.py:18
    -6: "unsupported size",
}
FRI_CHALLENGE_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                                    ctypes.POINTER(ctypes.c_uint64), ctypes.c_int)

# every symbol include/sa_b200.h declares: (name, restype, argtypes)
_vp, _sz, _ci, _u64p = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.POINTER(ctypes.c_uint64)
SYMBOLS = [
    ("sa_version", ctypes.c_char_p, []),
    ("sa_last_error", ctypes.c_char_p, []),
    ("sa_launch_count", ctypes.c_uint64, []),
    ("sa_ntt", _ci, [_vp, _vp, _ci, _u64p, _ci, _sz, _vp]),
    ("sa_ntt_multi", _ci, [ctypes.POINTER(ctypes.c_void_p), _ci, _sz, _vp, _ci, _u64p, _ci, _sz, _vp]),
    ("sa_ntt_mcast", _ci, [_vp, _vp, _sz, _vp, _ci, _u64p, _ci, _sz, _vp]),
    ("sa_push_mcast", _ci, [_vp, _vp, _sz, _vp]),
    ("sa_enable_peer_access", _ci, [_ci]),
    ("sa_peer_alloc", _ci, [ctypes.POINTER(ctypes.c_void_p), _sz, ctypes.c_char_p]),
    ("sa_peer_open", _ci, [ctypes.POINTER(ctypes.c_void_p), ctypes.c_char_p]),
    ("sa_peer_close", _ci, [_vp]),
    ("sa_peer_free", _ci, [_vp]),
    ("sa_copy_async", _ci, [_vp, _vp, _sz, _vp]),
    ("sa_push", _ci, [ctypes.POINTER(ctypes.c_void_p), _ci, _vp, _sz, _vp]),
    ("sa_ntt_host", _ci, [_vp, _vp, _ci, _u64p, _ci, _sz, _vp]),
    ("sa_host_alloc", _vp, [_sz]),
    ("sa_host_free", _ci, [_vp]),
    ("sa_pointwise_mul", _ci, [_vp, _vp, _vp, _sz, _vp]),
    ("sa_pointwise_div", _ci, [_vp, _vp, _vp, _sz, _vp]),
    ("sa_scale", _ci, [_vp, _vp, _sz, _u64p, _vp]),
    ("sa_poly_eval", _ci, [_vp, _vp, _sz, _vp, _sz, _vp]),
    ("sa_poly_eval_mode", _ci, [_vp, _vp, _sz, _vp, _sz, _ci, _vp]),
    ("sa_zerofier", _ci, [_vp, _vp, _sz, _vp]),
    ("sa_interpolate", _ci, [_vp, _vp, _vp, _sz, _vp]),
    ("sa_merkle_tree", _ci, [_vp, _vp, _sz, _vp]),
    ("sa_merkle_open", _ci, [_vp, _vp, _sz, _u64p, _sz, _vp]),
    ("sa_gather", _ci, [_vp, _vp, _sz, _u64p, _sz, _vp]),
    ("sa_fri_fold", _ci, [_vp, _vp, _sz, _u64p, _u64p, _u64p, _vp]),
    ("sa_fri_round", _ci, [_vp, _vp, _vp, _sz, _u64p, _u64p, _u64p, _vp]),
    ("sa_fri_commit", _ci, [_vp, _vp, _vp, _sz, _ci, _u64p, _u64p, _vp, _vp, _vp]),
    ("sa_cache_limit", _sz, [_sz]),
    ("sa_cache_bytes", _sz, []),
    ("sa_release_workspaces", _ci, []),
    ("sa_selftest_field", ctypes.c_longlong, [_sz, ctypes.c_uint64]),
    ("sa_microbench", ctypes.c_double, [_ci, _ci, _ci, _ci, _ci]),
]


def load_library(path=LIB_PATH):
    """dlopen the C-ABI library and type every entry point (works without a GPU)."""
    if not os.path.exists(path):
        raise RuntimeError(
            "stark-anatomy_b200: %s is missing -- build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (nvcc, sm_100a). There is no CPU fallback." % path)
    lib = ctypes.CDLL(path)
    for name, restype, argtypes in SYMBOLS:
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    return lib


def _limbs(x):
    x = int(x)
    return (ctypes.c_uint64 * 2)(x & 0xFFFFFFFFFFFFFFFF, x >> 64)


class SaError(AssertionError):
    """Raised with the reference's assertion message for SA_E* codes."""


class CudaEngine:
    """Device-resident operations; one instance per process (one process per GPU)."""

    name = "cuda"

    def __init__(self, device=None):
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError("stark-anatomy_b200: no CUDA device visible; the engine has no CPU fallback")
        self.torch = torch
        self.lib = load_library()
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        # host<->device traffic this engine object has caused (calls and bytes); tools/config5.py and the
        # tests use it to show which boundary crossings are left (SURVEY 8 f3)
        self.stats = {"h2d_calls": 0, "h2d_bytes": 0, "d2h_calls": 0, "d2h_bytes": 0}

    def _count(self, kind, nbytes):
        self.stats[kind + "_calls"] += 1
        self.stats[kind + "_bytes"] += int(nbytes)

    # ------------------------------------------------------------ plumbing
    def _stream(self):
        # the C library works on the CURRENT device; make sure that is this engine's (a peer tensor rebuilt from
        # an IPC handle, or user code, may have left another device current)
        cuda = self.torch.cuda
        if cuda.current_device() != self.device.index:
            cuda.set_device(self.device)
        return ctypes.c_void_p(cuda.current_stream(self.device).cuda_stream)

    def _check(self, rc):
        if rc == 0:
            return
        if rc in SA_ERRORS:
            raise SaError(SA_ERRORS[rc])
        if rc == -7:
            raise RuntimeError("sa_b200: the challenge callback failed")
        raise RuntimeError("sa_b200: CUDA error: %s" % self.lib.sa_last_error().decode())

    def empty(self, n):
        return self.torch.empty((n, 2), dtype=self.torch.int64, device=self.device)

    def zeros(self, n):
        return self.torch.zeros((n, 2), dtype=self.torch.int64, device=self.device)

    def length(self, vec):
        return vec.shape[0]

    def upload(self, buf):
        """packed 16-byte elements (bytearray / numpy / pinned tensor) -> device vector"""
        torch = self.torch
        if isinstance(buf, torch.Tensor):
            if not buf.is_cuda:
                self._count("h2d", buf.numel() * buf.element_size())
            return buf.reshape(-1, 2).to(self.device, non_blocking=True)
        if len(buf) == 0:
            return self.empty(0)
        host = torch.frombuffer(buf, dtype=torch.int64).reshape(-1, 2)
        self._count("h2d", host.numel() * 8)
        return host.to(self.device)

    def download(self, vec):
        """device vector -> numpy uint64[n, 2] (buffer protocol, 16 bytes/element)"""
        self._count("d2h", vec.numel() * 8)
        return vec.contiguous().cpu().numpy()

    def pad(self, vec, n):
        """zero-extend to n elements"""
        if vec.shape[0] == n:
            return vec
        out = self.zeros(n)
        out[:vec.shape[0]] = vec
        return out

    def slice(self, vec, lo, hi):
        return vec[lo:hi]

    def concat(self, vecs):
        return self.torch.cat(vecs, dim=0)

    # ------------------------------------------------------------------ ntt
    def ntt(self, vec, log_n, root, inverse=False, batch=1):
        vec = vec.contiguous()
        out = self.empty(vec.shape[0])
        self._check(self.lib.sa_ntt(out.data_ptr(), vec.data_ptr(), log_n, _limbs(root), int(bool(inverse)),
                                    batch, self._stream()))
        return out

    def ntt_into(self, out, vec, log_n, root, inverse=False, batch=1):
        """sa_ntt into a caller-provided device vector (a slice of a larger buffer); out may alias vec"""
        assert out.is_contiguous() and vec.is_contiguous() and out.shape[0] == vec.shape[0]
        self._check(self.lib.sa_ntt(out.data_ptr(), vec.data_ptr(), log_n, _limbs(root), int(bool(inverse)), batch,
                                    self._stream()))
        return out

    def ntt_multi(self, outs, out_offset, vec, log_n, root, inverse=False, batch=1):
        """sa_ntt_multi: transform `vec` and store the result at element offset `out_offset` of every buffer in
        `outs` (outs[0] on this device, the others peer-mapped buffers of other GPUs; tensors or raw pointers)"""
        vec = vec.contiguous()
        ptrs = (ctypes.c_void_p * len(outs))(*[int(t) if isinstance(t, int) else int(t.data_ptr()) for t in outs])
        self._check(self.lib.sa_ntt_multi(ptrs, len(outs), out_offset, vec.data_ptr(), log_n, _limbs(root),
                                          int(bool(inverse)), batch, self._stream()))

    def ntt_mcast(self, mc_ptr, local, out_offset, vec, log_n, root, inverse=False, batch=1):
        """sa_ntt_mcast: transform `vec`, store the result through the multicast address `mc_ptr` (every rank's
        buffer receives it, this rank's `local` included) at element offset `out_offset`"""
        vec = vec.contiguous()
        self._check(self.lib.sa_ntt_mcast(ctypes.c_void_p(int(mc_ptr)), local.data_ptr(), out_offset, vec.data_ptr(),
                                          log_n, _limbs(root), int(bool(inverse)), batch, self._stream()))

    def wrap_pointer(self, ptr, nelems):
        """a device vector (torch.int64[n, 2]) over memory this process got from the C library"""
        class _Raw:
            __cuda_array_interface__ = {"shape": (nelems, 2), "typestr": "<i8", "data": (int(ptr), False), "version": 2}
        return self.torch.as_tensor(_Raw(), device=self.device)

    def pointwise_mul(self, a, b):
        out = self.empty(a.shape[0])
        self._check(self.lib.sa_pointwise_mul(out.data_ptr(), a.contiguous().data_ptr(),
                                              b.contiguous().data_ptr(), a.shape[0], self._stream()))
        return out

    def pointwise_div(self, a, b):
        out = self.empty(a.shape[0])
        self._check(self.lib.sa_pointwise_div(out.data_ptr(), a.contiguous().data_ptr(),
                                              b.contiguous().data_ptr(), a.shape[0], self._stream()))
        return out

    def scale(self, vec, factor):
        vec = vec.contiguous()
        out = self.empty(vec.shape[0])
        self._check(self.lib.sa_scale(out.data_ptr(), vec.data_ptr(), vec.shape[0], _limbs(factor), self._stream()))
        return out

    def poly_eval(self, coeffs, points, mode=0):
        """values of the polynomial at the points; mode 0 = the library chooses, 1 = Horner kernel, 2 = walk down
        the subproduct tree of the points (sa_poly_eval_mode)"""
        coeffs, points = coeffs.contiguous(), points.contiguous()
        out = self.empty(points.shape[0])
        self._check(self.lib.sa_poly_eval_mode(out.data_ptr(), coeffs.data_ptr(), coeffs.shape[0], points.data_ptr(),
                                               points.shape[0], int(mode), self._stream()))
        return out

    MAX_DIRECT_POINTS = 1 << 20  # sa_zerofier / sa_interpolate handle this many points per call

    def zerofier(self, domain):
        domain = domain.contiguous()
        out = self.empty(domain.shape[0] + 1)
        self._check(self.lib.sa_zerofier(out.data_ptr(), domain.data_ptr(), domain.shape[0], self._stream()))
        return out

    def interpolate(self, domain, values):
        domain, values = domain.contiguous(), values.contiguous()
        out = self.empty(domain.shape[0])
        self._check(self.lib.sa_interpolate(out.data_ptr(), domain.data_ptr(), values.data_ptr(), domain.shape[0],
                                            self._stream()))
        return out

    # --------------------------------------------------------------- merkle
    def _new_tree(self, n):
        return self.torch.empty((2 * n, 64), dtype=self.torch.uint8, device=self.device)

    def merkle_tree(self, vec):
        vec = vec.contiguous()
        n = vec.shape[0]
        tree = self._new_tree(n)
        self._check(self.lib.sa_merkle_tree(tree.data_ptr(), vec.data_ptr(), n, self._stream()))
        return tree

    def tree_root(self, tree):
        self._count("d2h", 64)
        return bytes(tree[1].cpu().numpy().tobytes())

    def download_tree(self, tree):
        """the whole heap-ordered tree as a host array uint8[2n, 64] (small trees: paths are then read on
        the host, O(log n) per opened index and no device round trip)"""
        self._count("d2h", tree.numel())
        return tree.cpu().numpy()

    def merkle_open(self, tree, indices):
        """authentication paths (lists of 64-byte digests, bottom-up) for leaf indices"""
        n = tree.shape[0] // 2
        k = len(indices)
        depth = n.bit_length() - 1
        if k == 0:
            return []
        if depth == 0:
            for i in indices:
                if not 0 <= i < n:
                    raise SaError(SA_ERRORS[-5])
            return [[] for _ in indices]
        for i in indices:
            if not 0 <= i < n:
                raise SaError(SA_ERRORS[-5])
        out = self.torch.empty((k, depth, 64), dtype=self.torch.uint8, device=self.device)
        idx = (ctypes.c_uint64 * k)(*indices)
        self._check(self.lib.sa_merkle_open(out.data_ptr(), tree.data_ptr(), n, idx, k, self._stream()))
        self._count("h2d", 8 * k)
        self._count("d2h", k * depth * 64)
        raw = out.cpu().numpy().tobytes()
        return [[raw[(q * depth + l) * 64:(q * depth + l + 1) * 64] for l in range(depth)] for q in range(k)]

    def gather(self, vec, indices):
        """values at `indices` -> numpy uint64[k, 2] on the host"""
        vec = vec.contiguous()
        k = len(indices)
        out = self.empty(k)
        if k:
            idx = (ctypes.c_uint64 * k)(*indices)
            self._check(self.lib.sa_gather(out.data_ptr(), vec.data_ptr(), vec.shape[0], idx, k, self._stream()))
            self._count("h2d", 8 * k)
            self._count("d2h", 16 * k)
        return out.cpu().numpy()

    # ------------------------------------------------------------------ fri
    def fri_fold(self, vec, alpha, offset, omega):
        vec = vec.contiguous()
        n = vec.shape[0]
        out = self.empty(n // 2)
        self._check(self.lib.sa_fri_fold(out.data_ptr(), vec.data_ptr(), n, _limbs(alpha), _limbs(offset),
                                         _limbs(omega), self._stream()))
        return out

    def fri_round(self, vec, alpha, offset, omega):
        """fold (fri.py:85) + Merkle tree of the folded codeword, one fused kernel"""
        vec = vec.contiguous()
        n = vec.shape[0]
        out = self.empty(n // 2)
        tree = self._new_tree(n // 2)
        self._check(self.lib.sa_fri_round(out.data_ptr(), tree.data_ptr(), vec.data_ptr(), n, _limbs(alpha),
                                          _limbs(offset), _limbs(omega), self._stream()))
        return out, tree

    def fri_commit(self, vec, rounds, offset, omega, on_root):
        """code/fri.py:56-96 round loop in one C call (sa_fri_commit).

        on_root(round, root_bytes, want_alpha) is called after every round with the 64-byte
        Merkle root; it returns the challenge alpha (int) when want_alpha.  Returns
        (layers, trees): device vectors / trees of layers 0 .. rounds-1 (layer 0 is `vec`)."""
        vec = vec.contiguous()
        n = vec.shape[0]
        layers = self.empty(max(n - (n >> (rounds - 1)), 1))
        trees = self.torch.empty((4 * n - ((4 * n) >> rounds), 64), dtype=self.torch.uint8, device=self.device)
        errors = []

        def challenge(_user, r, root_ptr, alpha_out, want):
            try:
                alpha = on_root(r, ctypes.string_at(root_ptr, 64), bool(want))
                if want:
                    alpha_out[0] = alpha & 0xFFFFFFFFFFFFFFFF
                    alpha_out[1] = alpha >> 64
                return 0
            except BaseException as exc:  # re-raised below, outside the C frame
                errors.append(exc)
                return 1
        cb = FRI_CHALLENGE_FN(challenge)
        rc = self.lib.sa_fri_commit(layers.data_ptr(), trees.data_ptr(), vec.data_ptr(), n, rounds, _limbs(offset),
                                    _limbs(omega), cb, None, self._stream())
        if errors:
            raise errors[0]
        self._check(rc)
        out_layers, out_trees = [vec], []
        lo, to, ln = 0, 0, n
        for r in range(rounds):
            out_trees.append(trees[to:to + 2 * ln])
            to += 2 * ln
            if r + 1 < rounds:
                out_layers.append(layers[lo:lo + ln // 2])
                lo += ln // 2
                ln //= 2
        return out_layers, out_trees

    def synchronize(self):
        self.torch.cuda.synchronize(self.device)

    def launch_count(self):
        return int(self.lib.sa_launch_count())


_ENGINE = None


def get_engine():
    """The process-wide engine; created on first use.  Raises without CUDA."""
    global _ENGINE
    if _ENGINE is None:
        _ENGINE = CudaEngine()
    return _ENGINE


def set_engine(engine):
    """Install an engine object (tests use this to exercise the host logic with a
    test double; the product never calls it)."""
    global _ENGINE
    _ENGINE = engine
    return engine
