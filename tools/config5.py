#!/usr/bin/env python3
"""BASELINE config 5 on the real CUDA engine: the reference's code/fast_stark.py and code/fast_rpsss.py,
UNMODIFIED (imported from the checkout of the reference whose code/ directory STARK_REFERENCE names), with the
drop-in ntt.py / fri.py ahead of them on sys.path and the default engine (CUDA, no test double).

    python tools/config5.py [--out gpurun_out/r02_config5.json] [--skip-rpsss]

Scenarios (each in its own interpreter, so module state such as sa_accel cannot leak between them):
  faststark   seeded os.urandom (600), test_fast_stark.py parameters: the proof must have the sha256 the pure
              reference produced (tests/golden/faststark_trace.json) and the reference verifier logic accepts it
  rpsss       seeded os.urandom (700): FastRPSSS() (preprocess), keygen, sign(b"Hello, World!"), verify, verify
              of another document; signature sha256 == tests/golden/rpsss.json; wall times of every step
  rpsss+accel the same with the opt-in device Polynomial.__mul__ (sa_accel)
The JSON this prints / writes is what profiles/r02_config5.json holds.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "stark-anatomy_b200")


def find_reference():
    cand = os.environ.get("STARK_REFERENCE")
    return cand if cand and os.path.isdir(cand) else None


COMMON = r'''
import sys, os, random, hashlib, json, time
sys.dont_write_bytecode = True
sys.path[:0] = [%(pkg)r, %(ref)r]
import sa_engine
eng = sa_engine.get_engine()          # the CUDA engine; raises without a GPU
assert eng.name == "cuda"
import fast_stark as fs, fri, ntt
assert fri.__file__.startswith(%(pkg)r) and ntt.__file__.startswith(%(pkg)r), (fri.__file__, ntt.__file__)
assert fs.__file__.startswith(%(ref)r), fs.__file__
assert fs.fast_coset_evaluate is ntt.fast_coset_evaluate and fs.Fri is fri.Fri and fs.Merkle is fri.Merkle
from algebra import Field, FieldElement
field = Field.main()
def stats():
    s = dict(getattr(eng, "stats", {}))
    s["kernel_launches"] = eng.launch_count()
    return s
def delta(a, b):
    return {k: b[k] - a.get(k, 0) for k in b}
'''

FASTSTARK = COMMON + r'''
from rescue_prime import RescuePrime
rng = random.Random(600)
os.urandom = lambda n: bytes(rng.getrandbits(8) for _ in range(n))
rp = RescuePrime()
stark = fs.FastStark(field, 4, 2, 2, rp.m, rp.N + 1, transition_constraints_degree=3)
t0 = time.perf_counter(); tz, tzc, tzr = stark.preprocess(); t_pre = time.perf_counter() - t0
x = FieldElement(rng.randrange(field.p), field)
trace = rp.trace(x)
air = rp.transition_constraints(stark.omicron)
boundary = rp.boundary_constraints(rp.hash(x))
s0 = stats()
t0 = time.perf_counter(); proof = stark.prove(trace, air, boundary, tz, tzc); t_prove = time.perf_counter() - t0
s1 = stats()
t0 = time.perf_counter(); ok = stark.verify(proof, air, boundary, tzr); t_verify = time.perf_counter() - t0
print("RESULT " + json.dumps({"proof_sha256": hashlib.sha256(proof).hexdigest(), "proof_len": len(proof), "verify": bool(ok),
      "seconds": {"preprocess": t_pre, "prove": t_prove, "verify": t_verify}, "engine_during_prove": delta(s0, s1)}))
'''

RPSSS = COMMON + r'''
import fast_rpsss
assert fast_rpsss.__file__.startswith(%(ref)r)
rng = random.Random(700)
os.urandom = lambda n: bytes(rng.getrandbits(8) for _ in range(n))
if %(accel)r:
    import sa_accel
    sa_accel.enable()
t0 = time.perf_counter(); r = fast_rpsss.FastRPSSS(); t_init = time.perf_counter() - t0
sk, pk = r.keygen()
doc = b"Hello, World!"
s0 = stats()
t0 = time.perf_counter(); sig = r.sign(sk, doc); t_sign = time.perf_counter() - t0
s1 = stats()
t0 = time.perf_counter(); good = r.verify(pk, doc, sig); t_verify = time.perf_counter() - t0
bad = r.verify(pk, b"Byebye.", sig)
# a second signature: steady state (plans, twiddle tables and pools are warm)
t0 = time.perf_counter(); sig2 = r.sign(sk, b"second document"); t_sign2 = time.perf_counter() - t0
good2 = r.verify(pk, b"second document", sig2)
print("RESULT " + json.dumps({"signature_sha256": hashlib.sha256(sig).hexdigest(), "signature_len": len(sig),
      "pk": str(pk.value), "verify": bool(good), "verify_other_document": bool(bad), "verify_second": bool(good2),
      "accel_polymul": bool(%(accel)r),
      "seconds": {"init_preprocess": t_init, "sign": t_sign, "sign_warm": t_sign2, "verify": t_verify},
      "engine_during_sign": delta(s0, s1)}))
'''


def run(code, timeout=1800):
    out = subprocess.run([sys.executable, "-c", code], text=True, capture_output=True, timeout=timeout)
    line = [l for l in out.stdout.splitlines() if l.startswith("RESULT ")]
    if not line:
        return {"error": (out.stdout[-1500:] + out.stderr[-3000:])}
    return json.loads(line[0][7:])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--skip-rpsss", action="store_true")
    args = ap.parse_args()
    ref = find_reference()
    if ref is None:
        print(json.dumps({"unavailable": "STARK_REFERENCE does not name the reference's code/ directory"}))
        return 0
    fmt = {"pkg": PKG, "ref": ref}
    golden = os.path.join(ROOT, "tests", "golden")
    res = {"reference_dir": ref, "what": "unmodified code/fast_stark.py + code/fast_rpsss.py on the CUDA engine (drop-in ntt.py / fri.py)"}
    with open(os.path.join(golden, "faststark_trace.json")) as f:
        g = json.load(f)
    fsr = run(FASTSTARK % fmt)
    fsr["golden_proof_sha256"] = g["proof_sha256"]
    fsr["byte_identical"] = fsr.get("proof_sha256") == g["proof_sha256"] and fsr.get("proof_len") == g["proof_len"]
    res["faststark"] = fsr
    if not args.skip_rpsss:
        gp = os.path.join(golden, "rpsss.json")
        gr = json.load(open(gp)) if os.path.exists(gp) else {}
        for accel in (False, True):
            r = run(RPSSS % dict(fmt, accel=accel))
            r["golden_signature_sha256"] = gr.get("signature_sha256")
            r["byte_identical"] = bool(gr) and r.get("signature_sha256") == gr.get("signature_sha256")
            r["reference_seconds"] = gr.get("reference_seconds")
            res["rpsss_accel" if accel else "rpsss"] = r
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    ok = res["faststark"].get("byte_identical") and res["faststark"].get("verify")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
