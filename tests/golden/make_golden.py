#!/usr/bin/env python3
"""Generate tests/golden/*.json by running the UNMODIFIED Python reference.

Needs a checkout of the reference: STARK_REFERENCE names its code/ directory.
The fixtures pin the CPU oracle (tests/test_oracle.py), the CUDA engine
(tests/test_*_gpu.py) and the host mirror (tests/test_hostmirror.py) to the
reference's own outputs, so the tests themselves never need the reference.

    STARK_REFERENCE=<checkout>/code python tests/golden/make_golden.py    # ~2-3 minutes

Encoding: field elements are decimal strings, digests/bytes are hex strings.
Seeds are stated per case; inputs come from random.Random(seed).randrange(p).
"""
import hashlib
import json
import os
import pickle
import random
import subprocess
import sys

sys.dont_write_bytecode = True
REF = os.environ.get("STARK_REFERENCE")
if not REF or not os.path.isdir(REF):
    sys.exit("make_golden.py: set STARK_REFERENCE to the reference checkout's code/ directory")
sys.path.insert(0, REF)
HERE = os.path.dirname(os.path.abspath(__file__))

from algebra import Field, FieldElement            # noqa: E402
from univariate import Polynomial                  # noqa: E402
import ntt as refntt                               # noqa: E402
from merkle import Merkle                          # noqa: E402
from ip import ProofStream                         # noqa: E402
from fri import Fri                                # noqa: E402

field = Field.main()
P = field.p


def fe(v):
    return FieldElement(v, field)


def rand_elems(rng, n):
    return [fe(rng.randrange(P)) for _ in range(n)]


def enc(xs):
    return [str(x.value) for x in xs]


def vector_digest(xs):
    return hashlib.blake2b(b"".join(x.value.to_bytes(16, "little") for x in xs)).hexdigest()


def enc_obj(o):
    if isinstance(o, bytes):
        return {"b": o.hex()}
    if isinstance(o, FieldElement):
        return {"f": str(o.value)}
    if isinstance(o, list):
        return {"l": [enc_obj(x) for x in o]}
    if isinstance(o, tuple):
        return {"t": [enc_obj(x) for x in o]}
    if isinstance(o, int):
        return {"i": o}
    raise TypeError(type(o))


def dump(name, obj):
    path = os.path.join(HERE, name)
    with open(path, "w") as f:
        json.dump(obj, f, separators=(",", ":"))
    print(f"{name}: {os.path.getsize(path)} bytes")


def dump_gz(name, obj):
    """gzip-compressed JSON (mtime 0, so the same data gives the same bytes)"""
    import gzip
    path = os.path.join(HERE, name)
    with gzip.GzipFile(path, "wb", compresslevel=9, mtime=0) as f:
        f.write(json.dumps(obj, separators=(",", ":")).encode())
    print(f"{name}: {os.path.getsize(path)} bytes")


# --------------------------------------------------------------------- field
def gen_field():
    rng = random.Random(100)
    cases = []
    edge = [0, 1, 2, P - 1, P - 2, (1 << 64) - 1, 1 << 64, (1 << 127), (1 << 127) + 12345, 407 << 119]
    pairs = [(a, b) for a in edge for b in edge] + [(rng.randrange(P), rng.randrange(P)) for _ in range(200)]
    for a, b in pairs:
        A, B = fe(a), fe(b)
        cases.append({"a": str(a), "b": str(b), "add": str((A + B).value), "sub": str((A - B).value),
                      "mul": str((A * B).value), "inv": str(A.inverse().value),
                      "pow": str((A ^ (b % 1000003)).value), "neg": str((-A).value)})
    roots = {str(1 << k): str(field.primitive_nth_root(1 << k).value) for k in range(0, 25)}
    samples = []
    for n in (1, 16, 17, 32, 64):
        bs = bytes(rng.randrange(256) for _ in range(n))
        samples.append({"bytes": bs.hex(), "value": str(field.sample(bs).value)})
    dump("field.json", {"p": str(P), "generator": str(field.generator().value), "cases": cases,
                        "roots": roots, "samples": samples,
                        "bytes": [{"v": str(v), "s": bytes(fe(v)).decode()} for v in edge + [rng.randrange(P) for _ in range(20)]]})


# ----------------------------------------------------------------------- ntt
def gen_ntt():
    out = {"ntt": [], "intt": [], "digests": []}
    for logn in range(0, 11):
        n = 1 << logn
        rng = random.Random(200 + logn)
        xs = rand_elems(rng, n)
        w = field.primitive_nth_root(n)
        ys = refntt.ntt(w, xs) if n > 1 else xs
        out["ntt"].append({"seed": 200 + logn, "n": n, "root": str(w.value), "in": enc(xs), "out": enc(ys)})
        if n > 1:
            zs = refntt.intt(w, xs)
            out["intt"].append({"seed": 200 + logn, "n": n, "root": str(w.value), "in": enc(xs), "out": enc(zs)})
    # non-standard primitive roots (inverse root, odd power of the root)
    for logn, power in ((4, 3), (6, 5), (8, -1), (9, 7)):
        n = 1 << logn
        rng = random.Random(250 + logn)
        xs = rand_elems(rng, n)
        w = field.primitive_nth_root(n)
        w = w.inverse() if power < 0 else w ^ power
        out["ntt"].append({"seed": 250 + logn, "n": n, "root": str(w.value), "in": enc(xs), "out": enc(refntt.ntt(w, xs))})
    # special inputs
    n = 64
    w = field.primitive_nth_root(n)
    for name, xs in (("zeros", [fe(0)] * n), ("ones", [fe(1)] * n), ("pm1", [fe(P - 1)] * n),
                     ("delta", [fe(1)] + [fe(0)] * (n - 1)), ("ramp", [fe(i) for i in range(n)])):
        out["ntt"].append({"seed": name, "n": n, "root": str(w.value), "in": enc(xs), "out": enc(refntt.ntt(w, xs))})
    # digests of larger transforms (input recipe: BASELINE.md section 3)
    for logn, seed in ((12, 0), (13, 3), (14, 0)):
        n = 1 << logn
        rng = random.Random(seed)
        xs = rand_elems(rng, n)
        w = field.primitive_nth_root(n)
        out["digests"].append({"seed": seed, "n": n, "root": str(w.value),
                               "ntt": vector_digest(refntt.ntt(w, xs)), "intt": vector_digest(refntt.intt(w, xs))})
    # recorded in BASELINE.md section 3 (survey session, 189.7 s of reference time)
    out["digests"].append({"seed": 0, "n": 1 << 20, "root": str(field.primitive_nth_root(1 << 20).value),
                           "ntt": "ed47a03e33ff8db12b9ccc79462ac04f746786777569a830a8d88770caf632eeec98f286652134d42e1f5e976cde12f08175f879bf0ce134416a9aa97b1a8b06",
                           "source": "BASELINE.md section 3"})
    dump("ntt.json", out)


def gen_poly():
    out = {"multiply": [], "coset_evaluate": [], "coset_divide": [], "zerofier": [], "evaluate": [],
           "interpolate": [], "big": []}
    rng = random.Random(300)
    n = 64
    w = field.primitive_nth_root(n)
    shapes = [(0, 0), (3, 4), (3, 3), (7, 0), (5, 20), (31, 31), (17, 9), (30, 2), (12, 12), (1, 40)]
    for dl, dr in shapes:
        l = Polynomial(rand_elems(rng, dl + 1))
        r = Polynomial(rand_elems(rng, dr + 1))
        pr = refntt.fast_multiply(l, r, w, n)
        out["multiply"].append({"order": n, "root": str(w.value), "lhs": enc(l.coefficients), "rhs": enc(r.coefficients), "out": enc(pr.coefficients)})
    # trailing zero coefficients, zero operands, empty operand
    z = fe(0)
    specials = [
        (rand_elems(rng, 10) + [z, z, z], rand_elems(rng, 9) + [z]),
        ([z, z, z], rand_elems(rng, 5)),
        ([], rand_elems(rng, 5)),
        (rand_elems(rng, 3) + [z] * 4, rand_elems(rng, 2) + [z] * 5),   # degree < 8 with padding -> schoolbook length
        (rand_elems(rng, 6), [z, z, fe(1)]),
    ]
    for lc, rc in specials:
        pr = refntt.fast_multiply(Polynomial(lc), Polynomial(rc), w, n)
        out["multiply"].append({"order": n, "root": str(w.value), "lhs": enc(lc), "rhs": enc(rc), "out": enc(pr.coefficients)})
    # larger order with automatic shrink
    n2 = 1024
    w2 = field.primitive_nth_root(n2)
    for dl, dr in ((100, 27), (511, 500), (300, 8)):
        l = Polynomial(rand_elems(rng, dl + 1))
        r = Polynomial(rand_elems(rng, dr + 1))
        pr = refntt.fast_multiply(l, r, w2, n2)
        out["multiply"].append({"order": n2, "root": str(w2.value), "lhs": enc(l.coefficients), "rhs": enc(r.coefficients), "out": enc(pr.coefficients)})

    g = field.generator()
    for ncoef, order in ((1, 8), (5, 8), (8, 8), (20, 64), (64, 64), (100, 256), (283, 1024)):
        poly = Polynomial(rand_elems(rng, ncoef))
        wo = field.primitive_nth_root(order)
        vals = refntt.fast_coset_evaluate(poly, g, wo, order)
        out["coset_evaluate"].append({"order": order, "generator": str(wo.value), "offset": str(g.value), "coeffs": enc(poly.coefficients), "out": enc(vals)})
    vals = refntt.fast_coset_evaluate(Polynomial([]), g, field.primitive_nth_root(8), 8)
    out["coset_evaluate"].append({"order": 8, "generator": str(field.primitive_nth_root(8).value), "offset": str(g.value), "coeffs": [], "out": enc(vals)})

    for dq, dr, order in ((2, 3, 64), (20, 7, 64), (0, 31, 64), (31, 20, 64), (12, 1, 64), (300, 27, 1024), (100, 400, 1024)):
        wo = field.primitive_nth_root(order)
        q = Polynomial(rand_elems(rng, dq + 1))
        r = Polynomial(rand_elems(rng, dr + 1))
        prod = q * r
        quo = refntt.fast_coset_divide(prod, r, g, wo, order)
        assert quo == q
        out["coset_divide"].append({"order": order, "root": str(wo.value), "offset": str(g.value), "lhs": enc(prod.coefficients), "rhs": enc(r.coefficients), "out": enc(quo.coefficients)})
    # unclean division is not detected (ntt.py:137 comment): value still pinned
    wo = field.primitive_nth_root(64)
    lhs = Polynomial(rand_elems(rng, 30))
    rhs = Polynomial(rand_elems(rng, 10))
    quo = refntt.fast_coset_divide(lhs, rhs, g, wo, 64)
    out["coset_divide"].append({"order": 64, "root": str(wo.value), "offset": str(g.value), "lhs": enc(lhs.coefficients), "rhs": enc(rhs.coefficients), "out": enc(quo.coefficients), "unclean": True})
    quo = refntt.fast_coset_divide(Polynomial([]), rhs, g, wo, 64)
    out["coset_divide"].append({"order": 64, "root": str(wo.value), "offset": str(g.value), "lhs": [], "rhs": enc(rhs.coefficients), "out": enc(quo.coefficients)})

    n3 = 512
    w3 = field.primitive_nth_root(n3)
    for k in (0, 1, 2, 3, 7, 8, 9, 27, 64, 100):
        dom = rand_elems(rng, k)
        zf = refntt.fast_zerofier(dom, w3, n3)
        out["zerofier"].append({"order": n3, "root": str(w3.value), "domain": enc(dom), "out": enc(zf.coefficients)})
    for ncoef, k in ((1, 1), (5, 0), (10, 3), (40, 17), (64, 64), (30, 100)):
        poly = Polynomial(rand_elems(rng, ncoef))
        dom = rand_elems(rng, k)
        vals = refntt.fast_evaluate(poly, dom, w3, n3)
        out["evaluate"].append({"order": n3, "root": str(w3.value), "coeffs": enc(poly.coefficients), "domain": enc(dom), "out": enc(vals)})
    for k in (0, 1, 2, 3, 5, 16, 33, 71):
        dom = rand_elems(rng, k)
        vals = rand_elems(rng, k)
        poly = refntt.fast_interpolate(dom, vals, w3, n3)
        out["interpolate"].append({"order": n3, "root": str(w3.value), "domain": enc(dom), "values": enc(vals), "out": enc(poly.coefficients)})
    # interpolation on a subgroup prefix with some zero values (the shape fast_stark.py:86-90 uses)
    om = field.primitive_nth_root(64)
    dom = [om ^ i for i in range(40)]
    vals = rand_elems(rng, 40)
    vals[3] = fe(0)
    poly = refntt.fast_interpolate(dom, vals, om, 64)
    out["interpolate"].append({"order": 64, "root": str(om.value), "domain": enc(dom), "values": enc(vals), "out": enc(poly.coefficients)})

    # recorded in BASELINE.md section 3 (654.4 s of reference time)
    out["big"].append({"what": "fast_multiply", "seed": 2, "n": 1 << 20,
                       "digest": "6c676c90ad4d5582b54cf67188b08a16e6149f15d87fceeaf0fe26123de095312b14a1d91069bb35c18f053ae10fb6f0b6d43f5e57e788773708873374b0776b",
                       "source": "BASELINE.md section 3"})
    # a mid-size product computed now
    rng2 = random.Random(2)
    k = 1 << 12
    l = Polynomial(rand_elems(rng2, k // 2))
    r = Polynomial(rand_elems(rng2, k // 2))
    pr = refntt.fast_multiply(l, r, field.primitive_nth_root(k), k)
    out["big"].append({"what": "fast_multiply", "seed": 2, "n": k, "digest": vector_digest(pr.coefficients), "len": len(pr.coefficients)})
    dump("poly.json", out)


# -------------------------------------------------------------------- merkle
def gen_merkle():
    out = {"leaf": [], "commit": [], "open": []}
    rng = random.Random(400)
    for v in [0, 1, 9, 10, 12345678901234567890, P - 1, 10 ** 38, 10 ** 38 - 1, 10 ** 19, 10 ** 19 - 1] + [rng.randrange(P) for _ in range(10)] + [rng.randrange(10 ** k) for k in range(1, 39, 4)]:
        out["leaf"].append({"v": str(v), "digest": Merkle.H(bytes(fe(v))).hexdigest()})
    for logn in range(0, 9):
        n = 1 << logn
        xs = rand_elems(random.Random(410 + logn), n)
        out["commit"].append({"seed": 410 + logn, "n": n, "in": enc(xs), "root": Merkle.commit(xs).hex()})
        if n >= 2:
            for idx in sorted({0, 1, n // 2, n - 1, rng.randrange(n)}):
                out["open"].append({"seed": 410 + logn, "n": n, "index": idx, "path": [p.hex() for p in Merkle.open(idx, xs)]})
    for logn, seed in ((12, 1), (14, 1)):
        n = 1 << logn
        xs = rand_elems(random.Random(seed), n)
        out["commit"].append({"seed": seed, "n": n, "root": Merkle.commit(xs).hex()})
    out["commit"].append({"seed": 1, "n": 1 << 20, "source": "BASELINE.md section 3",
                          "root": "ed42d838c2164f94ef303eaafee84af247a3638e943cf4080f47078e5966ca1b1368eaea2524fbe3eb224cf6f1d8b0847257b45d73455e8acb9842108b9a151d"})
    out["commit"].append({"in": enc([fe(i) for i in range(1, 9)]), "n": 8, "seed": "1..8", "root": Merkle.commit([fe(i) for i in range(1, 9)]).hex()})
    dump("merkle.json", out)


# ----------------------------------------------------------------------- fri
def gen_fri():
    out = {"commit": [], "prove": [], "fold": []}
    g = field.generator()
    # single fold step (fri.py:85) on small vectors
    for logn in (1, 2, 5, 8):
        n = 1 << logn
        rng = random.Random(500 + logn)
        cw = rand_elems(rng, n)
        alpha = fe(rng.randrange(P))
        omega = field.primitive_nth_root(n)
        one, two = field.one(), fe(2)
        folded = [two.inverse() * ((one + alpha / (g * (omega ^ i))) * cw[i] + (one - alpha / (g * (omega ^ i))) * cw[n // 2 + i]) for i in range(n // 2)]
        out["fold"].append({"seed": 500 + logn, "n": n, "alpha": str(alpha.value), "offset": str(g.value), "omega": str(omega.value), "in": enc(cw), "out": enc(folded)})
    configs = [(256, 4, 17, 1), (64, 4, 2, 5), (1024, 4, 64, 1), (4096, 4, 64, 1), (4096, 8, 16, 7)]
    for (n, ef, tests, seed) in configs:
        omega = field.primitive_nth_root(n)
        cw = rand_elems(random.Random(seed), n)
        fri = Fri(g, omega, n, ef, tests)
        ps = ProofStream()
        layers = fri.commit(cw, ps)
        roots = [o for o in ps.objects if isinstance(o, bytes)]
        out["commit"].append({"seed": seed, "n": n, "ef": ef, "tests": tests, "rounds": fri.num_rounds(),
                              "roots": [r.hex() for r in roots], "last": enc(ps.objects[-1]),
                              "layer_lens": [len(l) for l in layers],
                              "layer_digests": [vector_digest(l) for l in layers],
                              "transcript_sha256": hashlib.sha256(pickle.dumps(ps.objects)).hexdigest()})
        # codeword of a low-degree polynomial (as in test_fri.py) for the prove fixture
        rng = random.Random(seed + 50)
        deg = n // ef - 1
        poly = Polynomial(rand_elems(rng, deg + 1))
        codeword = refntt.fast_coset_evaluate(poly, g, omega, n)
        ps = ProofStream()
        ps.push(b"prior-object")            # transcript need not start empty
        idx = fri.prove(codeword, ps)
        entry = {"seed": seed + 50, "n": n, "ef": ef, "tests": tests, "coeffs": enc(poly.coefficients),
                 "indices": idx, "num_objects": len(ps.objects),
                 "transcript_sha256": hashlib.sha256(pickle.dumps(ps.objects)).hexdigest(),
                 "verify": None}
        if n <= 1024:
            entry["objects"] = [enc_obj(o) for o in ps.objects]
        else:
            entry["object_sha256"] = [hashlib.sha256(pickle.dumps(o)).hexdigest() for o in ps.objects]
        if n <= 256:
            ps2 = ProofStream()
            ps2.objects = list(ps.objects)
            ps2.pull()
            pts = []
            entry["verify"] = bool(fri.verify(ps2, pts))
        out["prove"].append(entry)
    out["commit"].append({"seed": 1, "n": 1 << 20, "ef": 4, "tests": 64, "rounds": 12, "source": "BASELINE.md section 3",
                          "roots8": "ed42d838c2164f94 f7995d329c2f5805 11749815226e5328 3ea4670d830939a8 86180a2199d051bb d29430249f7f73ff b4fb6c618a93c045 6fc58a11714292c1 5bc94e4bab7b0760 b423d0f4d2cd164c b606d49ddf954697 6a4173dfdebb769d".split()})
    dump("fri.json", out)


# ------------------------------------------------- FastStark.prove call trace
def gen_faststark_trace():
    """Record every call fast_stark.py makes into the ntt.py / fri.py surfaces
    during one seeded FastStark.prove (test_fast_stark.py parameters), so the
    GPU box can replay them without the reference present."""
    import fast_stark as fs
    from rescue_prime import RescuePrime
    rng = random.Random(600)
    real_urandom = os.urandom
    os.urandom = lambda n: bytes(rng.getrandbits(8) for _ in range(n))
    try:
        calls = []

        def wrap(mod, name):
            orig = getattr(mod, name)

            def w(*a):
                res = orig(*a)
                calls.append((name, a, res))
                return res
            setattr(mod, name, w)
            return orig

        rp = RescuePrime()
        stark = fs.FastStark(field, 4, 2, 2, rp.m, rp.N + 1, transition_constraints_degree=3)
        names = ["fast_interpolate", "fast_coset_evaluate", "fast_coset_divide", "fast_zerofier"]
        origs = {nm: wrap(fs, nm) for nm in names}
        fri_obj = stark.fri
        fri_calls = []
        orig_prove = Fri.prove

        def prove_w(self, codeword, ps):
            before = len(ps.objects)
            prior = hashlib.sha256(pickle.dumps(ps.objects)).hexdigest()
            prior_objs = [enc_obj(o) for o in ps.objects]
            res = orig_prove(self, codeword, ps)
            fri_calls.append({"codeword": enc(codeword), "prior_objects": prior_objs, "prior_sha256": prior,
                              "indices": res, "pushed": [enc_obj(o) for o in ps.objects[before:]],
                              "after_sha256": hashlib.sha256(pickle.dumps(ps.objects)).hexdigest()})
            return res
        Fri.prove = prove_w

        tz, tzc, tzr = stark.preprocess()
        input_element = fe(rng.randrange(P))
        trace = rp.trace(input_element)
        output_element = rp.hash(input_element)
        air = rp.transition_constraints(stark.omicron)
        boundary = rp.boundary_constraints(output_element)
        proof = stark.prove(trace, air, boundary, tz, tzc)
        Fri.prove = orig_prove
        for nm in names:
            setattr(fs, nm, origs[nm])
        ok = stark.verify(proof, air, boundary, tzr)
        assert ok

        def enc_arg(a):
            if isinstance(a, Polynomial):
                return {"poly": enc(a.coefficients)}
            if isinstance(a, FieldElement):
                return {"f": str(a.value)}
            if isinstance(a, list):
                return {"l": enc(a)}
            if isinstance(a, int):
                return {"i": a}
            raise TypeError(type(a))
        rec = [{"fn": nm, "args": [enc_arg(x) for x in a], "out": enc_arg(res)} for nm, a, res in calls]
        dump("faststark_trace.json", {
            "params": {"expansion_factor": 4, "num_colinearity_checks": 2, "security_level": 2,
                       "num_registers": rp.m, "num_cycles": rp.N + 1, "transition_constraints_degree": 3,
                       "fri_domain_length": stark.fri_domain_length, "omicron_domain_length": stark.omicron_domain_length},
            "urandom_seed": 600, "calls": rec, "fri_prove": fri_calls,
            "proof_sha256": hashlib.sha256(proof).hexdigest(), "proof_len": len(proof), "verify": bool(ok)})
    finally:
        os.urandom = real_urandom


# ---------------------------------- full 64-byte roots of the 2^20 FRI ladder (BASELINE config 4)
def gen_fri_2_20():
    """Fri.commit of the reference on the seed-1 2^20 codeword (ef 4, 64 tests, 12 rounds): every
    round's full Merkle root and the digest of the last codeword.  ~75 s of reference time."""
    n = 1 << 20
    rng = random.Random(1)
    cw = [fe(rng.randrange(P)) for _ in range(n)]
    f = Fri(field.generator(), field.primitive_nth_root(n), n, 4, 64)
    ps = ProofStream()
    layers = f.commit(cw, ps)
    roots = [o.hex() for o in ps.objects if isinstance(o, bytes)]
    assert len(roots) == 12 and len(layers) == 12
    dump("fri_2_20.json", {"seed": 1, "n": n, "ef": 4, "tests": 64, "rounds": 12, "roots": roots,
                           "last_codeword_digest": vector_digest(ps.objects[-1]), "last_len": len(ps.objects[-1]),
                           "transcript_sha256": hashlib.sha256(pickle.dumps(ps.objects)).hexdigest()})


# ------------------------------------------ FastRPSSS keygen / sign (BASELINE config 5 parameters)
def gen_rpsss():
    """One seeded keygen + sign of the UNMODIFIED fast_rpsss.py (expansion 4, 64 colinearity checks,
    security level 128; FRI domain 4096, 4 rounds).  ~40 s of reference time; the 200 s reference
    verification is not run here (the signature is checked by the verifier in the GPU test)."""
    import time
    import fast_rpsss
    rng = random.Random(700)
    real_urandom = os.urandom
    os.urandom = lambda n: bytes(rng.getrandbits(8) for _ in range(n))
    try:
        t0 = time.perf_counter()
        r = fast_rpsss.FastRPSSS()
        t_init = time.perf_counter() - t0
        sk, pk = r.keygen()
        doc = b"Hello, World!"
        t0 = time.perf_counter()
        sig = r.sign(sk, doc)
        t_sign = time.perf_counter() - t0
        dump("rpsss.json", {"urandom_seed": 700, "document": doc.hex(), "sk": str(sk.value), "pk": str(pk.value),
                            "signature_sha256": hashlib.sha256(sig).hexdigest(), "signature_len": len(sig),
                            "fri_domain_length": r.stark.fri_domain_length,
                            "omicron_domain_length": r.stark.omicron_domain_length,
                            "reference_seconds": {"init_preprocess": round(t_init, 2), "sign": round(t_sign, 2),
                                                  "where": "dev container, 1 Xeon core, CPython 3.12"}})
    finally:
        os.urandom = real_urandom


# ---------------------------- recorded runs of fast_stark.py / fast_rpsss.py (tests/dropin_cases.py replays them)
def canon(x):
    """JSON-able canonical form of a value crossing the drop-in surface (independent of the classes' modules)"""
    if isinstance(x, bytes):
        return {"b": x.hex()}
    if isinstance(x, FieldElement):
        return {"f": str(x.value)}
    if isinstance(x, Polynomial):
        return {"poly": [str(c.value) for c in x.coefficients]}
    if isinstance(x, bool):
        return {"bool": x}
    if isinstance(x, int):
        return {"i": x}
    if isinstance(x, tuple):
        return {"t": [canon(v) for v in x]}
    if isinstance(x, list):
        return {"l": [canon(v) for v in x]}
    raise TypeError(type(x))


def canon_digest(x):
    return hashlib.sha256(json.dumps(canon(x), separators=(",", ":")).encode()).hexdigest()


class Recorder:
    """Records, in order, every top-level call the caller makes into the drop-in surface (the ntt.py functions,
    Merkle.commit / open, Fri.prove / verify), every object the caller pushes onto a proof stream (as a reference
    to the call result it came from where it did) and the Fiat-Shamir challenges drawn inside recorded calls
    together with the transcript state they were drawn from.  Arguments that are earlier results are stored as
    references, results as canonical digests."""

    def __init__(self):
        self.events, self.results, self.keep = [], {}, []
        self.elems, self.streams, self.depth, self.current = {}, {}, 0, None

    def _result(self, k, res):
        self.keep.append(res)
        self.results[id(res)] = k
        if isinstance(res, list):
            for i, e in enumerate(res):
                self.elems.setdefault(id(e), (k, i))

    def stream_id(self, ps):
        self.keep.append(ps)
        return self.streams.setdefault(id(ps), len(self.streams))

    def arg(self, a):
        if id(a) in self.results:
            return {"ref": self.results[id(a)]}
        if isinstance(a, ProofStream):
            return {"stream": self.stream_id(ps=a), "objects": canon_digest(list(a.objects)), "read_index": a.read_index}
        if isinstance(a, list) and not a:
            return {"out": []}
        return canon(a)

    def wrap(self, owner, name, label, method=False, static=False):
        orig = getattr(owner, name)
        rec = self

        def w(*a):
            if rec.depth:
                return orig(*a)
            args = a[1:] if method else a
            ev = {"fn": label, "args": [rec.arg(x) for x in args], "fs": []}
            if method:
                s = a[0]
                ev["fri"] = [canon(s.offset), canon(s.omega), s.domain_length, s.expansion_factor, s.num_colinearity_tests]
            streams = [x for x in args if isinstance(x, ProofStream)]
            before = len(streams[0].objects) if streams else 0
            rec.depth, rec.current = 1, ev
            try:
                res = orig(*a)
            finally:
                rec.depth, rec.current = 0, None
            ev["out"] = canon_digest(res)
            if label == "Fri.prove":
                ev["indices"] = res
            if streams:
                ev["pushed"] = canon_digest(list(streams[0].objects[before:]))
            if label == "Fri.verify":
                ev["out_list"] = canon_digest(args[1])
            rec._result(len(rec.events), res)
            rec.events.append(ev)
            return res
        setattr(owner, name, staticmethod(w) if static else w)

    def wrap_push(self, cls):
        orig = cls.push
        rec = self

        def push(ps, obj):
            if not rec.depth:
                if id(obj) in rec.results:
                    src = {"ref": rec.results[id(obj)]}
                elif id(obj) in rec.elems:
                    src = {"elem": list(rec.elems[id(obj)])}
                else:
                    src = canon(obj)
                rec.events.append({"push": rec.stream_id(ps), "obj": src})
            return orig(ps, obj)
        cls.push = push

    def wrap_fiat_shamir(self, cls):
        rec = self
        for kind in ("prover_fiat_shamir", "verifier_fiat_shamir"):
            orig = cls.__dict__.get(kind)
            if orig is None:
                continue

            def fs(ps, *a, _orig=orig, _kind=kind):
                out = _orig(ps, *a)
                if rec.current is not None:
                    seen = ps.objects if _kind == "prover_fiat_shamir" else ps.objects[:ps.read_index]
                    rec.current["fs"].append({"kind": _kind, "state": canon_digest(list(seen)), "out": out.hex()})
                return out
            setattr(cls, kind, fs)


def record_run(scenario):
    """run scenario() with the reference's modules instrumented; returns (its result, the recorded events)"""
    import fast_stark as fs
    import fri as reffri
    import merkle as refmerkle
    rec = Recorder()
    ntt_fns = [n for n in dir(fs) if n.startswith("fast_") and callable(getattr(fs, n))]
    classes = [ProofStream] + ProofStream.__subclasses__()
    saved = [(fs, n, getattr(fs, n)) for n in ntt_fns]
    saved += [(refmerkle.Merkle, n, refmerkle.Merkle.__dict__[n]) for n in ("commit", "open")]
    saved += [(reffri.Fri, n, reffri.Fri.__dict__[n]) for n in ("prove", "verify")]
    saved += [(c, n, c.__dict__[n]) for c in classes for n in ("push", "prover_fiat_shamir", "verifier_fiat_shamir")
              if n in c.__dict__]
    for n in ntt_fns:
        rec.wrap(fs, n, n)
    rec.wrap(refmerkle.Merkle, "commit", "Merkle.commit", static=True)
    rec.wrap(refmerkle.Merkle, "open", "Merkle.open", static=True)
    rec.wrap(reffri.Fri, "prove", "Fri.prove", method=True)
    rec.wrap(reffri.Fri, "verify", "Fri.verify", method=True)
    rec.wrap_push(ProofStream)
    for c in classes:
        rec.wrap_fiat_shamir(c)
    try:
        return scenario(rec), rec.events
    finally:
        for owner, n, f in saved:
            setattr(owner, n, f)


def seeded_urandom(seed):
    rng = random.Random(seed)
    return rng, (lambda n: bytes(rng.getrandbits(8) for _ in range(n)))


def gen_faststark_proof():
    """one seeded FastStark.prove + verify (test_fast_stark.py parameters, os.urandom seeded with 600, as in
    gen_faststark_trace) recorded for tests/dropin_cases.case_faststark_proof_replay"""
    import fast_stark as fs
    from rescue_prime import RescuePrime
    real_urandom = os.urandom
    rng, os.urandom = seeded_urandom(600)

    def scenario(rec):
        rp = RescuePrime()
        stark = fs.FastStark(field, 4, 2, 2, rp.m, rp.N + 1, transition_constraints_degree=3)
        tz, tzc, tzr = stark.preprocess()
        x = fe(rng.randrange(P))
        air = rp.transition_constraints(stark.omicron)
        boundary = rp.boundary_constraints(rp.hash(x))
        proof = stark.prove(rp.trace(x), air, boundary, tz, tzc)
        return proof, stark.verify(proof, air, boundary, tzr)
    try:
        (proof, ok), events = record_run(scenario)
    finally:
        os.urandom = real_urandom
    assert ok
    dump_gz("faststark_proof.json.gz", {"urandom_seed": 600, "events": events, "verify": ok,
                                  "proof_sha256": hashlib.sha256(proof).hexdigest(), "proof_len": len(proof)})


def gen_rpsss_run():
    """FastRPSSS keygen, sign(b"Hello, World!"), verify of that document and of b"Byebye." (os.urandom seeded
    with 700, as in gen_rpsss), recorded for tests/dropin_cases.case_rpsss_replay.  ~8 minutes."""
    import fast_rpsss
    real_urandom = os.urandom
    rng, os.urandom = seeded_urandom(700)

    def scenario(rec):
        r = fast_rpsss.FastRPSSS()
        sk, pk = r.keygen()
        sig = r.sign(sk, b"Hello, World!")
        return sig, r.verify(pk, b"Hello, World!", sig), r.verify(pk, b"Byebye.", sig)
    try:
        (sig, good, bad), events = record_run(scenario)
    finally:
        os.urandom = real_urandom
    assert good and not bad
    dump_gz("rpsss_run.json.gz", {"urandom_seed": 700, "events": events, "verify": good, "verify_other_document": bad,
                            "signature_sha256": hashlib.sha256(sig).hexdigest(), "signature_len": len(sig)})


# ------------------------------------------- value types, as tests/test_hostmirror.py exercises them
def gen_hostmirror():
    """sha256 and length of the text tests/test_hostmirror.py's SCRIPT prints with the reference's own
    algebra / univariate / merkle / ip modules; the mirror in stark-anatomy_b200/hostmirror must print the same"""
    sys.path.insert(0, os.path.dirname(HERE))
    from test_hostmirror import SCRIPT
    out = subprocess.check_output([sys.executable, "-c", SCRIPT, REF], text=True)
    dump("hostmirror.json", {"sha256": hashlib.sha256(out.encode()).hexdigest(), "len": len(out)})


if __name__ == "__main__":
    which = sys.argv[1:] or ["field", "ntt", "poly", "merkle", "fri", "faststark", "hostmirror", "faststark_proof"]
    if "field" in which:
        gen_field()
    if "ntt" in which:
        gen_ntt()
    if "poly" in which:
        gen_poly()
    if "merkle" in which:
        gen_merkle()
    if "fri" in which:
        gen_fri()
    if "faststark" in which:
        gen_faststark_trace()
    if "hostmirror" in which:
        gen_hostmirror()
    if "faststark_proof" in which:
        gen_faststark_proof()
    if "rpsss_run" in which:  # not in the default set: ~8 min
        gen_rpsss_run()
    if "fri20" in which:      # not in the default set: ~75 s
        gen_fri_2_20()
    if "rpsss" in which:      # not in the default set: ~40 s
        gen_rpsss()
