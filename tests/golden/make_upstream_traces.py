#!/usr/bin/env python3
"""Record the reference's own unit tests as call traces (tests/golden/upstream_*_trace.json).

    PHE_SOURCE_DIR=<checkout of python-paillier 1.5.0> python tests/golden/make_upstream_traces.py

Runs phe/tests/paillier_test.py, util_test.py and math_test.py of that checkout on its own, unmodified ``phe``
(default key size lowered to KEY_BITS, the same key-generation sweeps left out as in the replaying tests) and records:
  api   every call the test code makes into PaillierPublicKey / PaillierPrivateKey / EncryptedNumber / EncodedNumber and
        phe.util, with arguments, the random r values ``get_random_lt_n`` drew inside it, and the result or exception;
  seam  every call ``phe`` makes into its bigint seam (powmod / mulmod / invert in phe.util and phe.paillier), tagged
        with the test class that made it, plus the calls of a known-answer check and of a 1024-bit round trip.
A seeded sample (per API function, per test class for the seam) keeps the files to about 330 KB in all.  tests/test_reference_suite_dropin.py replays the api trace on this package,
tests/test_phe_seam_unmodified.py the seam trace through integration/phe_b200_backend.py.
"""
import importlib.util
import json
import os
import random
import sys
import unittest

SRC = os.environ["PHE_SOURCE_DIR"]
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, SRC)
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import phe                                            # noqa: E402
from phe import encoding, paillier, util              # noqa: E402
from oracle.trace import Unsupported, dump            # noqa: E402

KEY_BITS = 1152
SKIP = ("testKeyUniqueness", "testDefaultKeySize", "testStaticPrivateKeySize", "Fallbacks")
API = [(paillier.PaillierPublicKey, ("raw_encrypt", "encrypt")),
       (paillier.PaillierPrivateKey, ("raw_decrypt", "decrypt")),
       (paillier.EncryptedNumber, ("__add__", "__radd__", "__mul__", "__rmul__", "__sub__", "__rsub__", "__truediv__",
                                   "decrease_exponent_to")),
       (encoding.EncodedNumber, ("decode", "decrease_exponent_to"))]
UTIL = ("powmod", "mulmod", "invert", "isqrt", "improved_i_sqrt", "extended_euclidean_algorithm", "base64url_encode",
        "base64url_decode", "base64_to_int", "int_to_base64", "is_prime")
SEAM = ("powmod", "mulmod", "invert")

state = {"depth": 0, "drawn": None, "api": [], "seam": [], "keys": {}, "cls": None, "mod": None}


def _record(name, args, kwargs, fn):
    top = state["depth"] == 0
    if top:
        state["drawn"] = []
    state["depth"] += 1
    out, exc = None, None
    try:
        out = fn(*args, **kwargs)
        return out
    except Exception as e:                          # noqa: BLE001
        exc = e
        raise
    finally:
        state["depth"] -= 1
        if top:
            try:
                rec = {"f": name, "a": [dump(a) for a in args], "k": {k: dump(v) for k, v in kwargs.items()},
                       "r": [hex(r) for r in state["drawn"]], "m": state["mod"]}
                if exc is None:
                    rec["out"] = dump(out)
                else:
                    rec["exc"] = type(exc).__name__
                state["api"].append(rec)
            except Unsupported:
                pass


def _wrap_method(cls, meth):
    orig = cls.__dict__[meth]

    def w(*a, **k):
        return _record("%s.%s" % (cls.__name__, meth), a, k, orig)
    setattr(cls, meth, w)


def _wrap_encode():
    orig = encoding.EncodedNumber.__dict__["encode"].__func__

    def w(cls, *a, **k):
        return _record("EncodedNumber.encode", (cls,) + a, k, lambda c, *aa, **kk: orig(c, *aa, **kk))
    encoding.EncodedNumber.encode = classmethod(w)


def _wrap_util(name):
    orig = getattr(util, name)
    setattr(util, name, lambda *a, **k: _record("util." + name, a, k, orig))


def _wrap_seam(mod, name):
    orig = getattr(mod, name)

    def w(*a):
        rec = {"cls": state["cls"], "f": name, "a": [hex(x) if x >= 0 else "-" + hex(-x) for x in a]}
        try:
            o = orig(*a)
        except ZeroDivisionError:
            rec["exc"] = "ZeroDivisionError"
            state["seam"].append(rec)
            raise
        rec["out"] = hex(o)
        state["seam"].append(rec)
        return o
    setattr(mod, name, w)


def _install():
    for cls, meths in API:
        for m in meths:
            _wrap_method(cls, m)
    _wrap_encode()
    orig_draw = paillier.PaillierPublicKey.get_random_lt_n

    def draw(self):
        r = orig_draw(self)
        if state["drawn"] is not None:
            state["drawn"].append(r)
        return r
    paillier.PaillierPublicKey.get_random_lt_n = draw
    orig_init = paillier.PaillierPrivateKey.__init__

    def init(self, public_key, p, q):
        orig_init(self, public_key, p, q)
        state["keys"][hex(public_key.n)] = [hex(p), hex(q)]
    paillier.PaillierPrivateKey.__init__ = init
    orig_gen = paillier.generate_paillier_keypair

    def gen(private_keyring=None, n_length=None):
        return orig_gen(private_keyring, n_length=n_length or KEY_BITS)
    paillier.generate_paillier_keypair = phe.generate_paillier_keypair = gen
    for mod in (paillier, util):
        for name in SEAM:
            _wrap_seam(mod, name)          # phe.paillier imported the seam by name: both bindings are recorded
    for name in UTIL:                      # after the seam: util.powmod called from a test records both ways
        _wrap_util(name)


def _run(module):
    spec = importlib.util.spec_from_file_location("upstream_" + module, os.path.join(SRC, "phe", "tests", module + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    res = unittest.TestResult()
    state["mod"] = module
    for suite in unittest.defaultTestLoader.loadTestsFromModule(mod):
        cases = [case for case in suite if not any(s in case.id() for s in SKIP)]
        if cases:
            state["cls"] = type(cases[0]).__name__          # one suite per test class (runs its setUpClass)
            unittest.TestSuite(cases).run(res)
    assert not res.failures and not res.errors, (res.failures[:2], res.errors[:2])
    return res.testsRun


def _sample(records, budget, seed):
    """Every record when they fit `budget` bytes of JSON, else a seeded sample in the original order."""
    size = [len(json.dumps(r)) for r in records]
    if sum(size) <= budget:
        return records
    order = list(range(len(records)))
    random.Random(seed).shuffle(order)
    keep, used = set(), 0
    for i in order:
        if used + size[i] <= budget:
            keep.add(i)
            used += size[i]
    return [r for i, r in enumerate(records) if i in keep]


def _per(records, key, budget, seed):
    """_sample within each group of records with the same `key`, `budget` bytes per group."""
    return [r for k in sorted({r[key] for r in records}) for r in _sample([r for r in records if r[key] == k], budget, seed)]


def _seam_flows():
    """The seam calls of the reference's known answer (phe/tests/paillier_test.py:128-136) and of a 1024-bit round trip."""
    flows = {}
    for name, fn in (("known_answer", lambda: _known_answer()), ("roundtrip_1024", lambda: _roundtrip())):
        start = len(state["seam"])
        state["cls"] = name
        fn()
        flows[name] = state["seam"][start:]
        del state["seam"][start:]
    return flows


def _known_answer():
    pk = paillier.PaillierPublicKey(126869)
    sk = paillier.PaillierPrivateKey(pk, 293, 433)
    assert pk.raw_encrypt(10100, 74384) == 935906717 and sk.raw_decrypt(935906717) == 10100


def _roundtrip():
    pk, sk = paillier.generate_paillier_keypair(n_length=1024)
    c = pk.encrypt(-123456.75)
    assert sk.decrypt(c + 0.25) == -123456.5


def main():
    _install()
    flows = _seam_flows()
    state["api"].clear()
    runs = {m: _run(m) for m in ("paillier_test", "util_test", "math_test")}
    paillier_calls = [r for r in state["api"] if r["m"] == "paillier_test"]
    util_calls = [r for r in state["api"] if r["m"] != "paillier_test"]          # util_test and math_test
    api = {"phe_version": phe.__version__, "key_bits": KEY_BITS, "tests_run": runs, "keys": state["keys"],
           "calls_recorded": {"paillier": len(paillier_calls), "util_math": len(util_calls)},
           "paillier": _per(paillier_calls, "f", 12000, 1),
           "util_math": _per(util_calls, "f", 6000, 2)}
    used = json.dumps([api["paillier"], api["util_math"]])
    api["keys"] = {n: pq for n, pq in api["keys"].items() if '"%s"' % n in used}      # the keys the kept calls use
    seam = {"phe_version": phe.__version__, "key_bits": KEY_BITS, "calls_recorded": len(state["seam"]),
            "flows": flows,
            "calls": _per(state["seam"], "cls", 6000, 3)}
    for name, obj in (("upstream_api_trace.json", api), ("upstream_seam_trace.json", seam)):
        with open(os.path.join(HERE, name), "w") as f:
            json.dump(obj, f, separators=(",", ":"))
        print(name, os.path.getsize(os.path.join(HERE, name)), "bytes")
    print(runs, api["calls_recorded"], {"seam": seam["calls_recorded"], "kept": len(seam["calls"])},
          {"kept": [len(api["paillier"]), len(api["util_math"])]})


if __name__ == "__main__":
    main()
