"""Host-logic tests of the drop-in modules (no GPU): the engine is replaced by the
oracle-backed test double from tests/fake_engine.py.  Everything here is checked
against the reference's own outputs in tests/golden/."""
import hashlib
import os
import random
import subprocess
import sys

import pytest

import dropin_cases as C
import sa_engine
from fake_engine import OracleEngine
from conftest import load_golden, ROOT
from hostmirror_loader import HAVE_REFERENCE, REFERENCE

# these run the reference's own modules unmodified on top of the drop-in, so they need a checkout of it
needs_reference = pytest.mark.skipif(not HAVE_REFERENCE, reason="STARK_REFERENCE does not name the reference's code/ directory")


def drop_cached_trees():
    """fri.Merkle caches device trees by data fingerprint, and a tree belongs to the engine that built it:
    none may cross an engine swap (the GPU tests commit the same golden data on the CUDA engine)"""
    C.F.Merkle._trees.clear()
    C.F.Merkle._cache_bytes = 0


@pytest.fixture(autouse=True)
def double_engine():
    prev = sa_engine._ENGINE
    drop_cached_trees()
    sa_engine.set_engine(OracleEngine())
    yield
    sa_engine.set_engine(prev)
    drop_cached_trees()


def test_ntt_vectors():
    C.case_ntt_vectors()


def test_ntt_asserts():
    C.case_ntt_asserts()


def test_ntt_digests():
    C.case_ntt_digests(1 << 14)


def test_poly():
    C.case_poly()


def test_poly_asserts():
    C.case_poly_asserts()


def test_poly_split_recursion():
    C.case_poly_split_recursion()


def test_fast_multiply_4096():
    C.case_fast_multiply_big(1 << 12)


def test_fri_commit():
    C.case_fri_commit(1 << 12)


def test_fri_prove_and_verify():
    C.case_fri_prove(1 << 12)


def test_faststark_trace_replay():
    C.case_faststark_trace_replay()


def test_merkle_class():
    C.case_merkle_class()


def test_accel_polymul():
    C.case_accel_polymul()


def test_device_list():
    C.case_device_list()


def test_reference_style_properties():
    C.case_reference_style_properties()


def test_engine_use_is_recorded():
    """the drop-in really goes through the engine object (no hidden host arithmetic)"""
    eng = sa_engine.get_engine()
    C.N.ntt(C.T.field.primitive_nth_root(16), C.seeded(1, 16))
    assert ("ntt", 4, False, 1) in eng.calls


def test_default_engine_fails_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    sa_engine.set_engine(None)
    with pytest.raises(RuntimeError, match="no CUDA device"):
        C.N.ntt(C.T.field.primitive_nth_root(16), C.seeded(1, 16))


def test_unmodified_fast_stark_prove_is_byte_identical():
    """code/fast_stark.py, UNMODIFIED, with the drop-in ahead of it on sys.path and os.urandom seeded as in
    tests/golden/make_golden.py: the proof must be the same bytes the pure reference produced, and the
    reference verifier must accept it.  Every call fast_stark.py made into the drop-in during that prove and
    verify is recorded in tests/golden/faststark_proof.json.gz; replaying them rebuilds the proof from the
    drop-in's results.  With STARK_REFERENCE set, fast_stark.py itself runs on the drop-in as well."""
    C.case_faststark_proof_replay()
    assert len(sa_engine.get_engine().calls) > 10
    if not HAVE_REFERENCE:
        return
    code = r'''
import sys, os, random, hashlib
sys.dont_write_bytecode = True
sys.path[:0] = [%(pkg)r, %(ref)r, %(oracle)r, %(tests)r]
import sa_engine
from fake_engine import OracleEngine
sa_engine.set_engine(OracleEngine())
import fast_stark as fs, fri, ntt
assert fri.__file__.startswith(%(pkg)r) and ntt.__file__.startswith(%(pkg)r)
assert fs.__file__.startswith(%(ref)r)
assert fs.fast_coset_evaluate is ntt.fast_coset_evaluate and fs.Fri is fri.Fri
from rescue_prime import RescuePrime
from algebra import Field, FieldElement
field = Field.main()
rng = random.Random(600)
os.urandom = lambda n: bytes(rng.getrandbits(8) for _ in range(n))
rp = RescuePrime()
stark = fs.FastStark(field, 4, 2, 2, rp.m, rp.N + 1, transition_constraints_degree=3)
tz, tzc, tzr = stark.preprocess()
x = FieldElement(rng.randrange(field.p), field)
trace = rp.trace(x)
air = rp.transition_constraints(stark.omicron)
boundary = rp.boundary_constraints(rp.hash(x))
proof = stark.prove(trace, air, boundary, tz, tzc)
ok = stark.verify(proof, air, boundary, tzr)
print(hashlib.sha256(proof).hexdigest(), len(proof), ok, len(sa_engine.get_engine().calls))
''' % {"pkg": os.path.join(ROOT, "stark-anatomy_b200"), "ref": REFERENCE,
       "oracle": os.path.join(ROOT, "oracle"), "tests": os.path.join(ROOT, "tests")}
    out = subprocess.check_output([sys.executable, "-c", code], text=True).split()
    g = load_golden("faststark_trace.json")
    assert out[0] == g["proof_sha256"] and int(out[1]) == g["proof_len"]
    assert out[2] == "True" and int(out[3]) > 10
    # same again with the opt-in device Polynomial.__mul__ (section 8 f2): still the same bytes
    env = dict(os.environ, SA_B200_ACCEL_POLYMUL="1")
    out2 = subprocess.check_output([sys.executable, "-c", code], text=True, env=env).split()
    assert out2[:3] == out[:3] and int(out2[3]) > int(out[3])


@needs_reference
@pytest.mark.parametrize("ref_test", ["test_ntt.py", "test_fri.py", "test_merkle.py"])
def test_reference_own_tests_pass_against_the_dropin(ref_test):
    """The reference's OWN test files (code/test_ntt.py, test_fri.py, test_merkle.py), unmodified,
    collected from the read-only checkout with the drop-in directory ahead of code/ on sys.path:
    their `from ntt import *` / `from fri import *` bind to stark-anatomy_b200/ntt.py and fri.py
    (engine = the oracle-backed double, as everywhere in this file)."""
    code = r'''
import sys
sys.dont_write_bytecode = True
sys.path[:0] = [%(pkg)r, %(ref)r, %(oracle)r, %(tests)r]
import sa_engine
from fake_engine import OracleEngine
sa_engine.set_engine(OracleEngine())
import ntt, fri
assert ntt.__file__.startswith(%(pkg)r) and fri.__file__.startswith(%(pkg)r)
import pytest
# (--confcutdir: collection does not walk the directories above the reference, which may not be listable)
rc = pytest.main([%(target)r, "-q", "-x", "-k", "not colinearity", "-p", "no:cacheprovider",
                  "--rootdir", %(ref)r, "--confcutdir", %(ref)r, "-c", "/dev/null", "--import-mode=importlib"])
eng = sa_engine.get_engine()
print("RC", int(rc), "ENGINE_CALLS", len(eng.calls))
''' % {"pkg": os.path.join(ROOT, "stark-anatomy_b200"), "ref": REFERENCE,
       "oracle": os.path.join(ROOT, "oracle"), "tests": os.path.join(ROOT, "tests"),
       "target": os.path.join(REFERENCE, ref_test)}
    out = subprocess.run([sys.executable, "-c", code], text=True, capture_output=True, timeout=900,
                         cwd=os.path.join(ROOT, "tests"))
    tail = out.stdout.strip().splitlines()[-1].split() if out.stdout.strip() else []
    assert tail[:2] == ["RC", "0"], out.stdout[-2000:] + out.stderr[-2000:]
    if ref_test != "test_merkle.py":  # (test_merkle.py hashes raw byte strings: stays on the host class)
        assert int(tail[3]) > 0, "the reference test did not reach the engine"


def test_unmodified_fast_rpsss_sign_and_verify():
    """BASELINE config 5's functional check: code/fast_rpsss.py and code/fast_stark.py, unmodified, on top
    of the drop-in: keygen -> sign -> verify is True, and a signature does not verify for another document.
    (Reference alone: sign 29 s, verify 206 s.)  The calls they made into the drop-in during a seeded run are
    recorded in tests/golden/rpsss_run.json.gz; replaying them rebuilds the signature from the drop-in's results.
    With STARK_REFERENCE set, the two modules themselves run on the drop-in as well (with the opt-in device
    Polynomial.__mul__)."""
    C.case_rpsss_replay()
    assert len(sa_engine.get_engine().calls) > 50
    if not HAVE_REFERENCE:
        return
    code = r'''
import sys
sys.dont_write_bytecode = True
sys.path[:0] = [%(pkg)r, %(ref)r, %(oracle)r, %(tests)r]
import sa_engine
from fake_engine import OracleEngine
sa_engine.set_engine(OracleEngine())
import fast_rpsss, fast_stark, fri
assert fast_rpsss.__file__.startswith(%(ref)r) and fast_stark.__file__.startswith(%(ref)r)
assert fast_stark.Fri is fri.Fri and fri.__file__.startswith(%(pkg)r)
r = fast_rpsss.FastRPSSS()
sk, pk = r.keygen()
sig = r.sign(sk, b"Hello, World!")
print("RESULT", r.verify(pk, b"Hello, World!", sig), r.verify(pk, b"Byebye.", sig), len(sa_engine.get_engine().calls))
''' % {"pkg": os.path.join(ROOT, "stark-anatomy_b200"), "ref": REFERENCE,
       "oracle": os.path.join(ROOT, "oracle"), "tests": os.path.join(ROOT, "tests")}
    env = dict(os.environ, SA_B200_ACCEL_POLYMUL="1")
    out = subprocess.run([sys.executable, "-c", code], text=True, capture_output=True, timeout=900, env=env)
    line = [l for l in out.stdout.splitlines() if l.startswith("RESULT")]
    assert line, out.stdout[-2000:] + out.stderr[-2000:]
    _, good, bad, calls = line[0].split()
    assert good == "True" and bad == "False" and int(calls) > 50
