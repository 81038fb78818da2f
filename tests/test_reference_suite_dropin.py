"""The REFERENCE'S OWN unit tests (phe/tests/paillier_test.py, util_test.py, math_test.py) replayed on the drop-in
package, with the kernels on the test-only host simulation.  tests/golden/make_upstream_traces.py ran those tests on
the unmodified reference and recorded every call their code made into the phe API (keys, arguments, the random r each
encryption drew, the result or the exception raised); here every recorded call is made again on this package and must
give the same result, bit for bit, or raise the same exception.  Key sizes are reduced to 1152 bits (the simulation is
~100x slower than the GPU), nothing else is changed."""
import importlib

import pytest

from oracle.golden import load_golden
from oracle.trace import Loader, dump


@pytest.fixture(scope="module")
def trace(pkg):
    import __graft_entry__ as ge
    engine_mod = importlib.import_module("python-paillier_b200.engine")
    engine_mod._set_engine_for_tests(pkg.Engine(ge.build_hostsim()))
    yield load_golden("upstream_api_trace.json")
    engine_mod._set_engine_for_tests(None)


@pytest.fixture(params=["thread-per-ciphertext", "warp-per-ciphertext"])
def kernel_family(request, monkeypatch):
    """The scalar phe API is a batch of one: on the GPU it runs on the warp-per-ciphertext kernels (pai_coop.cuh);
    PAI_COOP_MAX=0 forces the throughput kernels.  The reference's tests must pass on both."""
    monkeypatch.setenv("PAI_COOP_MAX", "0" if request.param.startswith("thread") else "1000000")


def _replay(pkg, records, keys):
    """Re-make every recorded call on this package; returns the calls whose result differs."""
    util = importlib.import_module("python-paillier_b200.util")
    ld = Loader(pkg, keys)
    bad = []
    for rec in records:
        args = [ld.load(a) for a in rec["a"]]
        kw = {k: ld.load(v) for k, v in rec["k"].items()}
        owner, meth = rec["f"].split(".", 1)
        fn = getattr(util, meth) if owner == "util" else getattr(args.pop(0), meth)
        if rec["r"] and meth in ("encrypt", "raw_encrypt") and len(args) < (3 if meth == "encrypt" else 2) \
                and kw.get("r_value") is None:
            kw["r_value"] = int(rec["r"][0], 16)      # the r the reference drew (it obfuscates with it)
        try:
            got, exc = dump(fn(*args, **kw)), None
        except Exception as e:                        # noqa: BLE001
            got, exc = None, type(e).__name__
        if (exc != rec["exc"]) if "exc" in rec else (exc is not None or got != rec["out"]):
            bad.append((rec["f"], rec.get("exc", rec.get("out")), exc or got))
    return bad


def test_reference_paillier_tests(pkg, trace, kernel_family):
    recs = trace["paillier"]
    assert trace["tests_run"]["paillier_test"] > 150 and len(recs) > 100
    assert {r["f"].split(".")[0] for r in recs} >= {"PaillierPublicKey", "PaillierPrivateKey", "EncryptedNumber", "EncodedNumber"}
    bad = _replay(pkg, recs, trace["keys"])
    assert not bad, (len(bad), bad[:3])


def test_reference_util_and_math_tests(pkg, trace, kernel_family):
    recs = trace["util_math"]
    assert trace["tests_run"]["util_test"] >= 5 and trace["tests_run"]["math_test"] >= 2 and len(recs) > 200
    assert {r["m"] for r in recs} == {"util_test", "math_test"}
    bad = _replay(pkg, recs, trace["keys"])
    assert not bad, (len(bad), bad[:3])
