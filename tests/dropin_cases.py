"""Parity cases for the drop-in ``ntt`` / ``fri`` modules against tests/golden/*.json
(the reference's own outputs).  The same functions run twice:

  * tests/test_dropin_cpu.py  -- engine = tests/fake_engine.OracleEngine: checks the HOST
    logic (marshalling, list lengths, assertion messages, proof-stream pushes and
    pickle identity) without a GPU;
  * tests/test_dropin_gpu.py  -- engine = the CUDA engine: the parity tests proper.
"""
import gzip
import hashlib
import json
import os
import pickle
import random

import pytest

from conftest import GOLDEN, load_golden
from hostmirror_loader import load_host_types

T = load_host_types()
import ntt as N  # noqa: E402  (the drop-in, stark-anatomy_b200/ntt.py)
import fri as F  # noqa: E402

P = T.field.p


def vals(xs):
    return [x.value for x in xs]


def digest(xs):
    return hashlib.blake2b(b"".join(x.value.to_bytes(16, "little") for x in xs)).hexdigest()


def seeded(seed, n):
    rng = random.Random(seed)
    return [T.fe(rng.randrange(P)) for _ in range(n)]


# ------------------------------------------------------------------------ ntt
def case_ntt_vectors():
    g = load_golden("ntt.json")
    for c in g["ntt"]:
        xs = T.elems(c["in"])
        out = N.ntt(T.fe(c["root"]), xs)
        assert vals(out) == [int(v) for v in c["out"]], f"ntt n={c['n']} seed={c['seed']}"
        if c["n"] <= 1:
            assert out is xs  # ntt.py:5-6 returns the argument itself
        else:
            assert out is not xs and all(type(o) is T.FieldElement and o.field is T.field for o in out)
    for c in g["intt"]:
        xs = T.elems(c["in"])
        assert vals(N.intt(T.fe(c["root"]), xs)) == [int(v) for v in c["out"]], f"intt n={c['n']}"
    one = [T.fe(5)]
    assert N.intt(T.field.primitive_nth_root(1), one) is one


def case_ntt_asserts():
    with pytest.raises(AssertionError, match="cannot compute ntt of non-power-of-two sequence"):
        N.ntt(T.field.primitive_nth_root(4), T.elems([1, 2, 3]))
    with pytest.raises(AssertionError, match="cannot compute intt of non-power-of-two sequence"):
        N.intt(T.field.primitive_nth_root(4), T.elems([1, 2, 3]))
    with pytest.raises(AssertionError, match="primitive root must be nth root of unity"):
        N.ntt(T.field.primitive_nth_root(8), T.elems([1, 2, 3, 4]))
    with pytest.raises(AssertionError, match="primitive root is not primitive nth root of unity"):
        N.ntt(T.field.primitive_nth_root(2), T.elems([1, 2, 3, 4]))


def case_ntt_digests(max_n):
    for c in load_golden("ntt.json")["digests"]:
        if c["n"] > max_n:
            continue
        xs = seeded(c["seed"], c["n"])
        w = T.fe(c["root"])
        ys = N.ntt(w, xs)
        assert digest(ys) == c["ntt"], f"ntt digest n={c['n']}"
        if "intt" in c:
            assert digest(N.intt(w, xs)) == c["intt"]
        assert vals(N.intt(w, ys)) == vals(xs)  # round trip


def case_poly():
    g = load_golden("poly.json")
    for c in g["multiply"]:
        got = N.fast_multiply(T.poly(c["lhs"]), T.poly(c["rhs"]), T.fe(c["root"]), c["order"])
        assert vals(got.coefficients) == [int(v) for v in c["out"]], "fast_multiply"
    for c in g["coset_evaluate"]:
        got = N.fast_coset_evaluate(T.poly(c["coeffs"]), T.fe(c["offset"]), T.fe(c["generator"]), c["order"])
        assert vals(got) == [int(v) for v in c["out"]], "fast_coset_evaluate"
    for c in g["coset_divide"]:
        got = N.fast_coset_divide(T.poly(c["lhs"]), T.poly(c["rhs"]), T.fe(c["offset"]), T.fe(c["root"]), c["order"])
        assert vals(got.coefficients) == [int(v) for v in c["out"]], "fast_coset_divide"
    for c in g["zerofier"]:
        got = N.fast_zerofier(T.elems(c["domain"]), T.fe(c["root"]), c["order"])
        assert vals(got.coefficients) == [int(v) for v in c["out"]], "fast_zerofier"
    for c in g["evaluate"]:
        got = N.fast_evaluate(T.poly(c["coeffs"]), T.elems(c["domain"]), T.fe(c["root"]), c["order"])
        assert vals(got) == [int(v) for v in c["out"]], "fast_evaluate"
    for c in g["interpolate"]:
        got = N.fast_interpolate(T.elems(c["domain"]), T.elems(c["values"]), T.fe(c["root"]), c["order"])
        assert vals(got.coefficients) == [int(v) for v in c["out"]], "fast_interpolate"


def case_poly_split_recursion():
    """domains larger than one device call handles (sa_engine.MAX_DIRECT_POINTS) go through the
    reference's own halving recursion (ntt.py:76-80, :113-130) on top of the device pieces: force that
    path with a tiny limit and replay the golden zerofier / interpolate cases through it"""
    import sa_engine
    eng = sa_engine.get_engine()
    g = load_golden("poly.json")
    saved = eng.MAX_DIRECT_POINTS
    eng.MAX_DIRECT_POINTS = 3
    try:
        for c in g["zerofier"]:
            got = N.fast_zerofier(T.elems(c["domain"]), T.fe(c["root"]), c["order"])
            assert vals(got.coefficients) == [int(v) for v in c["out"]], "fast_zerofier (split)"
        for c in g["interpolate"]:
            got = N.fast_interpolate(T.elems(c["domain"]), T.elems(c["values"]), T.fe(c["root"]), c["order"])
            want = [int(v) for v in c["out"]]
            have = vals(got.coefficients)
            # the recursion's schoolbook combination may carry trailing zeros the direct kernel does not
            while len(have) > len(want) and have[-1] == 0:
                have.pop()
            assert have == want, "fast_interpolate (split)"
    finally:
        eng.MAX_DIRECT_POINTS = saved


def case_poly_asserts():
    w = T.field.primitive_nth_root(64)
    a, b = T.poly(range(1, 20)), T.poly(range(3, 12))
    with pytest.raises(AssertionError, match="supplied root does not have supplied order"):
        N.fast_multiply(a, b, w, 32)
    with pytest.raises(AssertionError, match="supplied root is not primitive root of supplied order"):
        N.fast_multiply(a, b, w, 128)
    with pytest.raises(AssertionError, match="cannot divide by zero polynomial"):
        N.fast_coset_divide(a, T.poly([0, 0]), T.field.generator(), w, 64)
    with pytest.raises(AssertionError, match="cannot divide by polynomial of larger degree"):
        N.fast_coset_divide(b, a, T.field.generator(), w, 64)
    with pytest.raises(AssertionError, match="cannot interpolate over domain of different length"):
        N.fast_interpolate(T.elems([1, 2]), T.elems([1]), w, 64)
    # a divisor codeword with a zero entry: algebra.py:92 "divide by zero"
    zero_at_coset = T.poly([(-T.field.generator()).value, 1])  # X - g vanishes at g*w^0
    big = T.poly(range(1, 30))
    with pytest.raises(AssertionError, match="divide by zero"):
        N.fast_coset_divide(big * T.poly([1] * 9), zero_at_coset * T.poly([1] * 9), T.field.generator(), w, 64)


def case_fast_multiply_big(n):
    c = [c for c in load_golden("poly.json")["big"] if c["n"] == n][0]
    rng = random.Random(c["seed"])
    lhs = T.Polynomial([T.fe(rng.randrange(P)) for _ in range(n // 2)])
    rhs = T.Polynomial([T.fe(rng.randrange(P)) for _ in range(n // 2)])
    got = N.fast_multiply(lhs, rhs, T.field.primitive_nth_root(n), n)
    assert len(got.coefficients) == n - 1
    assert digest(got.coefficients) == c["digest"]


# ------------------------------------------------------------------------ fri
def case_fri_commit(max_n):
    for c in load_golden("fri.json")["commit"]:
        if c["n"] > max_n or "roots" not in c:
            continue
        n = c["n"]
        cw = seeded(c["seed"], n)
        fri = F.Fri(T.field.generator(), T.field.primitive_nth_root(n), n, c["ef"], c["tests"])
        assert fri.num_rounds() == c["rounds"]
        ps = F.ProofStream()
        layers = fri.commit(cw, ps)
        roots = [o for o in ps.objects if isinstance(o, bytes)]
        assert [r.hex() for r in roots] == c["roots"]
        assert type(ps.objects[-1]) is list and vals(ps.objects[-1]) == [int(v) for v in c["last"]]
        assert layers[0] is cw and layers[-1] is ps.objects[-1]  # fri.py:82,91-96 aliasing
        assert [len(l) for l in layers] == c["layer_lens"]
        assert [digest(list(l)) for l in layers] == c["layer_digests"]
        assert hashlib.sha256(pickle.dumps(ps.objects)).hexdigest() == c["transcript_sha256"]


def case_fri_commit_2_20():
    """BASELINE config 4: all 12 full 64-byte roots, the last codeword and the pickled transcript of the
    reference's own Fri.commit on the seed-1 2^20 codeword (tests/golden/fri_2_20.json)"""
    c = load_golden("fri_2_20.json")
    n = 1 << 20
    cw = seeded(1, n)
    fri = F.Fri(T.field.generator(), T.field.primitive_nth_root(n), n, 4, 64)
    ps = F.ProofStream()
    layers = fri.commit(cw, ps)
    roots = [o for o in ps.objects if isinstance(o, bytes)]
    assert [r.hex() for r in roots] == c["roots"]
    assert len(ps.objects[-1]) == c["last_len"] and digest(ps.objects[-1]) == c["last_codeword_digest"]
    assert hashlib.sha256(pickle.dumps(ps.objects)).hexdigest() == c["transcript_sha256"]
    assert [len(l) for l in layers] == [n >> r for r in range(12)]
    # the same ladder from a device-resident codeword (what fast_coset_evaluate hands to Fri.prove)
    dev = F.DeviceCodeword(N._engine().upload(__import__("sa_marshal").pack(cw)), None, T.field)
    ps2 = F.ProofStream()
    fri.commit(dev, ps2)
    assert pickle.dumps(ps2.objects) == pickle.dumps(ps.objects)


def case_fri_prove(max_n, with_verify=True):
    for c in load_golden("fri.json")["prove"]:
        if c["n"] > max_n:
            continue
        n = c["n"]
        omega = T.field.primitive_nth_root(n)
        g = T.field.generator()
        codeword = N.fast_coset_evaluate(T.poly(c["coeffs"]), g, omega, n)
        fri = F.Fri(g, omega, n, c["ef"], c["tests"])
        ps = F.ProofStream()
        ps.push(b"prior-object")
        indices = fri.prove(codeword, ps)
        assert indices == c["indices"]
        assert len(ps.objects) == c["num_objects"]
        if "objects" in c:
            want = [T.dec_obj(o) for o in c["objects"]]
            for i, (got_o, want_o) in enumerate(zip(ps.objects, want)):
                assert pickle.dumps(got_o) == pickle.dumps(want_o), f"object {i} differs"
        else:
            assert [hashlib.sha256(pickle.dumps(o)).hexdigest() for o in ps.objects] == c["object_sha256"]
        # byte-identical transcript, including pickle's object-identity (memo) structure
        assert hashlib.sha256(pickle.dumps(ps.objects)).hexdigest() == c["transcript_sha256"]
        if with_verify and n <= 1024:
            vs = F.ProofStream()
            vs.objects = list(ps.objects)
            vs.pull()
            points = []
            assert fri.verify(vs, points) is True
            for (i, y) in points:  # returned points lie on the polynomial (test_fri.py:44-50)
                assert T.poly(c["coeffs"]).evaluate(g * (omega ^ i)) == y
            # corrupt the codeword -> verifier must reject (test_fri.py:52-58)
            bad = list(codeword)
            for i in range(0, n // 3):
                bad[i] = T.field.zero()
            bs = F.ProofStream()
            fri.prove(bad, bs)
            assert fri.verify(bs, []) is False


def case_faststark_trace_replay():
    """Replay every call fast_stark.py made into the ntt/fri surfaces during a seeded
    FastStark.prove (recorded from the unmodified reference) and compare results."""
    g = load_golden("faststark_trace.json")

    def dec(a):
        (k, v), = a.items()
        if k == "poly":
            return T.poly(v)
        if k == "f":
            return T.fe(v)
        if k == "l":
            return T.elems(v)
        return v
    for call in g["calls"]:
        args = [dec(a) for a in call["args"]]
        got = getattr(N, call["fn"])(*args)
        (k, want), = call["out"].items()
        got_vals = vals(got.coefficients) if k == "poly" else vals(got)
        assert got_vals == [int(v) for v in want], call["fn"]
    p = g["params"]
    for rec in g["fri_prove"]:
        n = p["fri_domain_length"]
        fri = F.Fri(T.field.generator(), T.field.primitive_nth_root(n), n, p["expansion_factor"],
                    p["num_colinearity_checks"])
        ps = F.ProofStream()
        ps.objects = [T.dec_obj(o) for o in rec["prior_objects"]]
        assert hashlib.sha256(pickle.dumps(ps.objects)).hexdigest() == rec["prior_sha256"]
        before = len(ps.objects)
        idx = fri.prove(T.elems(rec["codeword"]), ps)
        assert idx == rec["indices"]
        want = [T.dec_obj(o) for o in rec["pushed"]]
        assert [pickle.dumps(o) for o in ps.objects[before:]] == [pickle.dumps(o) for o in want]


# ------------------------------------------ recorded runs of fast_stark.py / fast_rpsss.py
def canon(x):
    """the canonical form make_golden.py's Recorder digests (the same rules, on the drop-in's types)"""
    import sa_devlist
    if isinstance(x, bytes):
        return {"b": x.hex()}
    if isinstance(x, T.FieldElement):
        return {"f": str(x.value)}
    if isinstance(x, T.Polynomial):
        return {"poly": [str(c.value) for c in x.coefficients]}
    if isinstance(x, bool):
        return {"bool": x}
    if isinstance(x, int):
        return {"i": x}
    if isinstance(x, tuple):
        return {"t": [canon(v) for v in x]}
    if isinstance(x, (list, sa_devlist.DeviceCodeword)):
        return {"l": [canon(v) for v in x]}
    raise TypeError(type(x))


def canon_digest(x):
    return hashlib.sha256(json.dumps(canon(x), separators=(",", ":")).encode()).hexdigest()


def decode(c):
    (k, v), = c.items()
    if k == "b":
        return bytes.fromhex(v)
    if k == "f":
        return T.fe(v)
    if k == "poly":
        return T.poly(v)
    if k in ("i", "bool"):
        return v
    if k == "t":
        return tuple(decode(x) for x in v)
    if k == "l":
        return [decode(x) for x in v]
    raise ValueError(k)


class ReplayStream(F.ProofStream):
    """A proof stream whose Fiat-Shamir challenges are the recorded ones; each is handed out only if the
    transcript it is drawn from is, digest for digest, the one the reference drew it from."""

    def __init__(self, objects=(), read_index=0):
        F.ProofStream.__init__(self)
        self.objects, self.read_index, self.challenges = list(objects), read_index, []

    def _challenge(self, kind, seen):
        assert self.challenges, "a challenge the reference did not draw"
        c = self.challenges.pop(0)
        assert c["kind"] == kind and c["state"] == canon_digest(list(seen)), "transcript differs at a challenge"
        return bytes.fromhex(c["out"])

    def prover_fiat_shamir(self, num_bytes=32):
        return self._challenge("prover_fiat_shamir", self.objects)

    def verifier_fiat_shamir(self, num_bytes=32):
        return self._challenge("verifier_fiat_shamir", self.objects[:self.read_index])


def replay_recorded(name):
    """Replay a run of the unmodified caller recorded by make_golden.py (Recorder): every call it made into the
    drop-in surface, in order, with the drop-in's own earlier results as the arguments that were results, must
    give the reference's result (digest), push what the reference pushed and draw the challenges it drew; the
    caller's own pushes are rebuilt from the drop-in's results.  Returns the recorded file and the streams."""
    with gzip.open(os.path.join(GOLDEN, name), "rt") as f:
        g = json.load(f)
    results, streams = {}, {}  # event index -> the drop-in's result; stream number -> ReplayStream

    def arg(a):
        if "ref" in a:
            return results[a["ref"]]
        if "out" in a:
            return []
        if "stream" in a:
            ps = streams.get(a["stream"])
            if ps is None:  # a stream the caller filled itself (a deserialized proof): one with the same objects
                src = [s for s in streams.values() if canon_digest(s.objects) == a["objects"]]
                assert src, "no replayed stream holds the objects this call was given"
                ps = streams[a["stream"]] = ReplayStream(src[0].objects)
            ps.read_index = a["read_index"]
            assert canon_digest(ps.objects) == a["objects"]
            return ps
        return decode(a)
    for i, ev in enumerate(g["events"]):
        if "push" in ev:
            ps = streams.setdefault(ev["push"], ReplayStream())
            src = ev["obj"]
            ps.push(results[src["ref"]] if "ref" in src else
                    results[src["elem"][0]][src["elem"][1]] if "elem" in src else decode(src))
            continue
        fn, args = ev["fn"], [arg(a) for a in ev["args"]]
        where = "event %d (%s)" % (i, fn)
        stream = next((a for a in args if isinstance(a, ReplayStream)), None)
        before = len(stream.objects) if stream is not None else 0
        if stream is not None:
            stream.challenges = list(ev["fs"])
        if fn.startswith("fast_"):
            got = getattr(N, fn)(*args)
        elif fn.startswith("Merkle."):
            got = getattr(F.Merkle, fn[7:])(*args)
        else:
            off, om, n, ef, tests = ev["fri"]
            got = getattr(F.Fri(decode(off), decode(om), n, ef, tests), fn[4:])(*args)
        assert canon_digest(got) == ev["out"], where
        if stream is not None:
            assert not stream.challenges, where + ": fewer challenges than the reference drew"
            assert canon_digest(stream.objects[before:]) == ev["pushed"], where
        if fn == "Fri.verify":
            assert canon_digest(args[1]) == ev["out_list"], where
        results[i] = got
    return g, streams


def case_faststark_proof_replay():
    """fast_stark.py's seeded prove + verify (tests/golden/faststark_proof.json.gz): the proof assembled from the
    drop-in's results is the reference's proof, byte for byte, and the verifier's FRI check accepts it"""
    g, streams = replay_recorded("faststark_proof.json.gz")
    proof = streams[0].serialize()
    assert hashlib.sha256(proof).hexdigest() == g["proof_sha256"] and len(proof) == g["proof_len"]
    verdicts = [e["out"] for e in g["events"] if e.get("fn") == "Fri.verify"]
    assert g["verify"] is True and verdicts == [canon_digest(True)]


def case_rpsss_replay():
    """fast_rpsss.py's seeded keygen, sign and two verifies (tests/golden/rpsss_run.json.gz): the signature
    assembled from the drop-in's results is the reference's, byte for byte; every FRI verdict is the reference's"""
    g, streams = replay_recorded("rpsss_run.json.gz")
    sig = streams[0].serialize()
    assert hashlib.sha256(sig).hexdigest() == g["signature_sha256"] == load_golden("rpsss.json")["signature_sha256"]
    assert len(sig) == g["signature_len"]
    assert g["verify"] is True and g["verify_other_document"] is False


# --------------------------------------------------------------------- merkle
def case_merkle_class():
    """fri.Merkle (GPU commit/open for field elements) against the reference's outputs"""
    g = load_golden("merkle.json")
    by_key = {}
    for c in g["commit"]:
        if "in" in c:
            xs = T.elems(c["in"])
        elif c["n"] <= 1 << 14:
            xs = seeded(c["seed"], c["n"])
        else:
            continue
        by_key[(str(c["seed"]), c["n"])] = xs
        assert F.Merkle.commit(xs).hex() == c["root"]
    for c in g["open"]:
        xs = by_key[(str(c["seed"]), c["n"])]
        path = F.Merkle.open(c["index"], xs)
        assert [p.hex() for p in path] == c["path"]
        assert F.Merkle.verify(F.Merkle.commit(xs), c["index"], path, xs[c["index"]])
        assert not F.Merkle.verify(F.Merkle.commit(xs), c["index"] ^ 1, path, xs[c["index"]])
    xs = seeded(9, 64)
    with pytest.raises(AssertionError, match="cannot open invalid index"):
        F.Merkle.open(64, xs)
    # raw byte strings (code/test_merkle.py's data) stay on the caller's host class
    import os
    data = [os.urandom(int(os.urandom(1)[0]) + 1) for _ in range(16)]
    root = F.Merkle.commit(data)
    for i in range(16):
        assert F.Merkle.verify(root, i, F.Merkle.open(i, data), data[i])


# ----------------------------------------------------- device-resident lists
def case_device_list():
    """sa_devlist.DeviceCodeword: the list-like ntt / intt / fast_coset_evaluate return (section 8 f3)"""
    import sa_devlist
    import sa_engine
    n = 256
    w = T.field.primitive_nth_root(n)
    xs = seeded(31, n)
    out = N.ntt(w, xs)
    assert isinstance(out, sa_devlist.DeviceCodeword) and not isinstance(out, list)
    ref = load_golden  # noqa: F841
    plain = list(out)
    assert len(out) == n and vals(plain) == vals(N.ntt(w, list(xs)))
    # list protocol
    assert out[3] is out[3] and out[-1] is out[n - 1] and out[3].value == plain[3].value
    assert all(type(o) is T.FieldElement and o.field is T.field for o in out)
    assert out == plain and plain == out and not (out != plain) and out != plain[:-1]
    assert vals(out[10:20]) == vals(plain[10:20]) and type(out[10:20]) is list
    assert vals(out + [T.fe(1)]) == vals(plain) + [1] and vals([T.fe(1)] + out) == [1] + vals(plain)
    assert plain[5] in out and out.index(plain[5]) == 5 and out.count(plain[5]) == 1
    assert vals(reversed(out)) == vals(plain)[::-1]
    with pytest.raises(IndexError):
        out[n]
    assert pickle.loads(pickle.dumps(out)) == plain
    # the chain stays on the device: intt(ntt(x)) == x, no element is created in between
    eng = sa_engine.get_engine()
    back = N.intt(w, N.ntt(w, xs))
    assert vals(back) == vals(xs)
    # a big one is read through gathers, identity per index is stable, tolist keeps identities
    big_n = 1 << 15
    big = N.ntt(T.field.primitive_nth_root(big_n), seeded(32, big_n))
    a, b = big[12345], big[7]
    assert big[12345] is a and big._full is None
    full = big.tolist()
    assert full[12345] is a and full[7] is b and big[100] is full[100]
    # Merkle on a device list == the host class on the plain list; opens come from the attached tree
    host = F._HostMerkle
    assert F.Merkle.commit(out) == host.commit(plain)
    for i in (0, 1, 77, n - 1):
        assert F.Merkle.open(i, out) == host.open(i, plain)
        assert F.Merkle.verify(F.Merkle.commit(out), i, F.Merkle.open(i, out), out[i])
    with pytest.raises(AssertionError, match="cannot open invalid index"):
        F.Merkle.open(n, out)
    big_tree = F.Merkle.commit(big)
    assert big_tree == host.commit(full) and F.Merkle.open(4242, big) == host.open(4242, full)
    # mutation: the host list becomes the truth, the device copy and tree are rebuilt on demand
    out[0] = T.fe(123)
    plain[0] = T.fe(123)
    assert out == plain and len(out) == n
    assert F.Merkle.commit(out) == host.commit(plain) and F.Merkle.open(0, out) == host.open(0, plain)
    assert vals(N.intt(w, out)) == vals(N.intt(w, plain))
    out.append(T.fe(5))
    assert len(out) == n + 1 and out[-1].value == 5
    # a plain list modified in place after Fri.commit is re-hashed by query, like merkle.py:26-27
    m = 64
    cw = seeded(33, m)
    fri = F.Fri(T.field.generator(), T.field.primitive_nth_root(m), m, 2, 4)
    ps = F.ProofStream()
    layers = fri.commit(cw, ps)
    idx = [1, 5, 9, 13]
    cw[1] = T.fe(999)
    qs = F.ProofStream()
    fri.query(layers[0], layers[1], idx, qs)
    assert qs.objects[4] == host.open(1, cw)
    # SA_B200_DEVICE_LISTS=0 behaviour: plain lists
    sa_devlist.ENABLED = False
    try:
        assert type(N.ntt(w, xs)) is list
    finally:
        sa_devlist.ENABLED = True


# ----------------------------------------------------------------- sa_accel
def case_accel_polymul():
    """opt-in device Polynomial.__mul__ (section 8 f2) == the schoolbook product, same lengths"""
    import sa_accel
    rng = random.Random(77)

    def rnd(n, zero_tail=0):
        return T.Polynomial([T.fe(rng.randrange(P)) for _ in range(n)] + [T.field.zero()] * zero_tail)
    shapes = [(1, 1), (40, 70), (64, 64), (100, 3, 5), (283, 283), (850, 28), (1, 3000), (1025, 1024, 2)]
    pairs = []
    for sh in shapes:
        tail = sh[2] if len(sh) > 2 else 0
        pairs.append((rnd(sh[0], tail), rnd(sh[1])))
    want = [vals((a * b).coefficients) for a, b in pairs]
    assert sa_accel._original_mul is None
    sa_accel.enable(threshold=1)
    try:
        for (a, b), w in zip(pairs, want):
            got = a * b
            assert vals(got.coefficients) == w and len(got.coefficients) == len(a.coefficients) + len(b.coefficients) - 1
        assert (T.Polynomial([]) * pairs[0][0]).coefficients == []
        x = T.Polynomial([T.field.zero(), T.field.one()])
        assert vals(((x ^ 5) * pairs[1][0]).coefficients) == [0] * 5 + vals(pairs[1][0].coefficients)
    finally:
        sa_accel.disable()
    assert T.Polynomial.__mul__ is not sa_accel.device_mul


# ------------------------------------------- the reference's own test strategy
def case_reference_style_properties(trials=5):
    """Randomised cross-checks in the style of code/test_ntt.py, code/test_merkle.py (fresh
    os.urandom inputs every run; fast path == slow path of the host value types)."""
    import os
    field = T.field

    def sample(nbytes=17):
        return field.sample(os.urandom(nbytes))

    # test_ntt.py:6-19  ntt == evaluation on the powers of the root
    n = 1 << 8
    w = field.primitive_nth_root(n)
    coeffs = [sample() for _ in range(n)]
    assert N.ntt(w, coeffs) == T.Polynomial(coeffs).evaluate_domain([w ^ i for i in range(n)])
    # test_ntt.py:21-32  intt(ntt(x)) == x
    n = 1 << 7
    w = field.primitive_nth_root(n)
    values = [sample(1) for _ in range(n)]
    assert N.intt(w, N.ntt(w, values)) == values
    # test_ntt.py:34-70  multiply == schoolbook, divide recovers the factor
    n = 1 << 6
    w = field.primitive_nth_root(n)
    for _ in range(trials):
        lhs = T.Polynomial([sample() for _ in range(os.urandom(1)[0] % (n // 2) + 1)])
        rhs = T.Polynomial([sample() for _ in range(os.urandom(1)[0] % (n // 2) + 1)])
        product = N.fast_multiply(lhs, rhs, w, n)
        assert product == lhs * rhs
        if not lhs.is_zero() and not rhs.is_zero():
            assert N.fast_coset_divide(product, lhs, field.generator(), w, n) == rhs
    # test_ntt.py:72-96  fast_evaluate(fast_interpolate(domain, values), domain) == values
    n = 1 << 9
    w = field.primitive_nth_root(n)
    for _ in range(2):
        k = int.from_bytes(os.urandom(2), "big") % 200 + 1
        seen, domain = set(), []
        while len(domain) < k:
            d = sample()
            if d.value not in seen:
                seen.add(d.value)
                domain.append(d)
        vals_ = [sample() for _ in range(k)]
        poly = N.fast_interpolate(domain, vals_, w, n)
        assert N.fast_evaluate(poly, domain, w, n) == vals_
        assert N.fast_evaluate(N.fast_zerofier(domain, w, n), domain, w, n) == [field.zero()] * k
    # test_ntt.py:98-116  coset evaluation == pointwise evaluation on offset * <omega>
    n = 1 << 5
    w = field.primitive_nth_root(n)
    poly = T.Polynomial([sample() for _ in range(n // 2)])
    got = N.fast_coset_evaluate(poly, field.generator(), w, n)
    assert got == [poly.evaluate(field.generator() * (w ^ i)) for i in range(n)]
    # test_merkle.py:4-47 with field-element leaves: every index opens and verifies; tampering fails
    n = 64
    data = [sample() for _ in range(n)]
    root = F.Merkle.commit(data)
    for i in range(n):
        path = F.Merkle.open(i, data)
        assert F.Merkle.verify(root, i, path, data[i])
        assert not F.Merkle.verify(root, i, path, sample())           # wrong leaf
        assert not F.Merkle.verify(root, (i + 1) % n, path, data[i])  # wrong index
        bad = list(path)
        bad[os.urandom(1)[0] % len(bad)] = os.urandom(64)
        assert not F.Merkle.verify(root, i, bad, data[i])             # wrong path element
    assert not F.Merkle.verify(os.urandom(64), 0, F.Merkle.open(0, data), data[0])  # wrong root
