"""Test helper: load the host value types the drop-in modules will use.

``load_host_types()`` puts stark-anatomy_b200/ (and, when STARK_REFERENCE names a
checkout of the reference's code/ directory, that directory behind it) on sys.path
exactly like a user of the drop-in would, imports the drop-in ``ntt`` / ``fri``
modules and returns a small namespace with the value types plus JSON fixture decoders.
Without STARK_REFERENCE the drop-in uses its own host mirror of the value types.
"""
import importlib
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "stark-anatomy_b200")

# the reference's flat module directory; also enables the tests that run its modules unmodified
REFERENCE = os.environ.get("STARK_REFERENCE", "")
HAVE_REFERENCE = bool(REFERENCE) and os.path.isdir(REFERENCE)


def setup_paths(use_reference=True):
    """drop-in first, then (optionally) the reference's flat module directory"""
    sys.dont_write_bytecode = True
    if use_reference and HAVE_REFERENCE and REFERENCE not in sys.path:
        sys.path.insert(0, REFERENCE)
    if PKG in sys.path:
        sys.path.remove(PKG)
    sys.path.insert(0, PKG)


def load_host_types(use_reference=True):
    setup_paths(use_reference)
    sa_host = importlib.import_module("sa_host")
    ns = types.SimpleNamespace()
    ns.algebra = sa_host.algebra
    ns.univariate = sa_host.univariate
    ns.Field = sa_host.algebra.Field
    ns.FieldElement = sa_host.algebra.FieldElement
    ns.Polynomial = sa_host.univariate.Polynomial
    ns.field = ns.Field.main()
    ns.using_reference_types = "hostmirror" not in (sa_host.algebra.__file__ or "")

    def fe(v):
        return ns.FieldElement(int(v), ns.field)

    def dec_obj(o):
        (k, v), = o.items()
        if k == "b":
            return bytes.fromhex(v)
        if k == "f":
            return fe(v)
        if k == "l":
            return [dec_obj(x) for x in v]
        if k == "t":
            return tuple(dec_obj(x) for x in v)
        if k == "i":
            return v
        raise ValueError(k)
    ns.fe = fe
    ns.dec_obj = dec_obj
    ns.elems = lambda xs: [fe(x) for x in xs]
    ns.poly = lambda xs: ns.Polynomial([fe(x) for x in xs])
    return ns
