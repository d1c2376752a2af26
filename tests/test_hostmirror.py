"""The host mirror (stark-anatomy_b200/hostmirror) behaves like the reference's value
types and pickles to the same bytes: SCRIPT's output with the mirror must be the text the
reference's own modules printed (its sha256 and length: tests/golden/hostmirror.json, made by make_golden.py)."""
import hashlib
import os
import subprocess
import sys
import textwrap

from conftest import ROOT, load_golden

MIRROR = os.path.join(ROOT, "stark-anatomy_b200", "hostmirror")

SCRIPT = textwrap.dedent('''
    import sys, pickle, random, hashlib, json
    sys.dont_write_bytecode = True
    sys.path.insert(0, sys.argv[1])
    from algebra import Field, FieldElement, xgcd
    from univariate import Polynomial, test_colinearity
    from merkle import Merkle
    from ip import ProofStream
    f = Field.main(); P = f.p; rng = random.Random(3)
    F = lambda v: FieldElement(v, f)
    out = []
    for _ in range(200):
        a, b = rng.randrange(P), rng.randrange(1, P)
        A, B = F(a), F(b)
        out += [(A + B).value, (A - B).value, (A * B).value, (A / B).value, (-A).value, A.inverse().value,
                (A ^ rng.randrange(2000)).value, bytes(A).decode(), str(A), A == B, A.is_zero()]
    out += [F(0).inverse().value, F(7) == F(7), xgcd(240, 46)]
    out += [f.primitive_nth_root(1 << k).value for k in range(0, 22)] + [f.generator().value]
    out += [f.sample(bytes(range(k))).value for k in (1, 16, 17, 40)]
    def co(p): return [c.value for c in p.coefficients]
    for _ in range(60):
        a = [rng.randrange(P) if rng.random() < 0.8 else 0 for _ in range(rng.randrange(0, 12))]
        b = [rng.randrange(P) if rng.random() < 0.8 else 0 for _ in range(rng.randrange(1, 8))]
        A, B = Polynomial([F(v) for v in a]), Polynomial([F(v) for v in b])
        x = F(rng.randrange(P))
        out += [A.degree(), A.is_zero(), co(A * B), co(A + B), co(A - B), co(-A), A.evaluate(x).value,
                co(A.scale(x)), co(A ^ 3), A == B, A == Polynomial([F(v) for v in a] + [F(0)])]
        if B.degree() >= 0:
            q, r = Polynomial.divide(A, B)
            out += [co(q), r.degree(), co(r)[:r.degree() + 1]]
            out += [co((A * B) / B) if A.degree() >= 0 else None, (A % B).degree()]
    for n in (1, 2, 3, 6):
        dom = [F(rng.randrange(P)) for _ in range(n)]; vals = [F(rng.randrange(P)) for _ in range(n)]
        ip = Polynomial.interpolate_domain(dom, vals)
        out += [ip.degree(), co(ip)[:ip.degree() + 1], co(Polynomial.zerofier_domain(dom))]
    out += [test_colinearity([(F(1), F(2)), (F(2), F(4)), (F(3), F(6))]),
            test_colinearity([(F(1), F(2)), (F(2), F(4)), (F(3), F(7))]),
            test_colinearity([(F(1), F(5)), (F(2), F(5)), (F(3), F(5))])]
    for n in (2, 4, 16):
        data = [F(rng.randrange(P)) for _ in range(n)]
        root = Merkle.commit(data)
        out += [root.hex()] + [[p.hex() for p in Merkle.open(i, data)] for i in range(n)]
        out += [Merkle.verify(root, i, Merkle.open(i, data), data[i]) for i in range(n)]
        out += [Merkle.verify(root, 0, Merkle.open(1, data), data[0])]
    ps = ProofStream()
    xs = [F(rng.randrange(P)) for _ in range(5)]
    for o in (b"root", xs, (xs[0], xs[1], xs[2]), [b"a" * 64, b"b" * 64]):
        ps.push(o)
    out += [ps.serialize().hex(), ps.prover_fiat_shamir().hex(), ps.pull().hex(), ps.verifier_fiat_shamir().hex()]
    print(json.dumps(out, default=str))
''')


def test_mirror_matches_reference_including_pickles():
    ref = load_golden("hostmirror.json")
    mir = subprocess.check_output([sys.executable, "-c", SCRIPT, MIRROR], text=True)
    assert len(mir) == ref["len"] and hashlib.sha256(mir.encode()).hexdigest() == ref["sha256"]
