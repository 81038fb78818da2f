"""The boundary exercised the way the reference would bind it: the three bigint seam functions of the unmodified phe
package (phe/util.py:38,53,85, imported by name at phe/paillier.py:29) rebound to integration/phe_b200_backend.py --
the ctypes stub INTEGRATION.md section 1 quotes -- exactly as the reference's own tests flip backends
(phe/tests/util_test.py:64-75).  tests/golden/make_upstream_traces.py ran the reference's unit tests on the unmodified
reference and recorded every seam call its phe made (arguments and result, tagged with the test class); here every
recorded call goes through the backend and must give the same result.  The engine is the test-only host simulation of
the device code."""
import importlib.util
import os
import sys
import types

import pytest

from oracle.golden import load_golden


@pytest.fixture(scope="module")
def backend():
    import __graft_entry__ as ge
    spec = importlib.util.spec_from_file_location("phe_b200_backend", os.path.join(ge.ROOT, "integration", "phe_b200_backend.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.load(ge.build_hostsim())
    return mod, load_golden("upstream_seam_trace.json")


def _h(s):
    return -int(s[1:], 16) if s.startswith("-") else int(s, 16)


def _replay(fns, calls):
    bad = []
    for c in calls:
        try:
            got = hex(fns[c["f"]](*[_h(a) for a in c["a"]]))
        except ZeroDivisionError:
            got = "ZeroDivisionError"
        if got != c.get("out", c.get("exc")):
            bad.append((c["cls"], c["f"], c["a"], got))
    return bad


def test_seam_is_rebound_and_counts_calls(backend):
    """install() rebinds the seam in phe.util and phe.paillier (a stand-in package with phe's module layout: the
    backend touches nothing else), uninstall() restores it; the seam calls of the reference's known answer
    (phe/tests/paillier_test.py:128-136) and of a 1024-bit encrypt / add / decrypt go through the engine."""
    be, trace = backend
    names = ("powmod", "mulmod", "invert")
    pkg, pu, pp = (types.ModuleType(n) for n in ("phe", "phe.util", "phe.paillier"))
    pkg.util, pkg.paillier = pu, pp
    originals = {n: (lambda *a: None) for n in names}
    for mod in (pu, pp):
        for n in names:
            setattr(mod, n, originals[n])
    saved = {k: sys.modules.get(k) for k in ("phe", "phe.util", "phe.paillier")}
    sys.modules.update({"phe": pkg, "phe.util": pu, "phe.paillier": pp})
    try:
        be.install(pkg)
        assert pp.powmod is be.powmod and pp.mulmod is be.mulmod and pp.invert is be.invert
        assert pu.powmod is be.powmod and pu.mulmod is be.mulmod and pu.invert is be.invert
        calls = {"n": 0}
        lib = be._lib

        class LibProxy:
            def __getattr__(self, name):
                fn = getattr(lib, name)
                if name != "pai_mod_powmod_host":
                    return fn

                def counted(*a):
                    calls["n"] += 1
                    return fn(*a)
                return counted
        be._lib = LibProxy()
        try:
            fns = {n: getattr(pp, n) for n in names}
            assert not _replay(fns, trace["flows"]["known_answer"])
            assert calls["n"] >= 2                    # r^n mod n^2 and the decrypt's powmod
            calls["n"] = 0
            assert not _replay(fns, trace["flows"]["roundtrip_1024"])
            assert calls["n"] >= 5                    # hp, hq (key constants), r^n, and the CRT pair
        finally:
            be._lib = lib
        be.uninstall(pkg)
        assert all(getattr(mod, n) is originals[n] for mod in (pu, pp) for n in names)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def test_reference_test_classes_on_unmodified_phe(backend):
    be, trace = backend
    calls = trace["calls"]
    classes = {c["cls"] for c in calls}
    assert {"PaillierTestRawEncryption", "PaillierTestEncryptedNumber", "TestKeyring", "TestIssue62", "PaillierUtilTest",
            "ArithmeticTest"} <= classes and len(calls) >= 100
    assert {c["f"] for c in calls} == {"powmod", "mulmod", "invert"}
    bad = _replay({"powmod": be.powmod, "mulmod": be.mulmod, "invert": be.invert}, calls)
    assert not bad, (len(bad), bad[:2])
