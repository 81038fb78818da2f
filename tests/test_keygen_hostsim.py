"""Batched key generation (SURVEY.md 8f rank 4): pai_miller_rabin / util.is_prime_batch / getprimeover_batch /
generate_paillier_keypairs on the host simulation -- probable-prime agreement with the reference's is_prime
(phe/util.py:420-443) on primes, composites, Carmichael numbers and strong pseudoprimes to small bases."""
import importlib

import pytest

from oracle.golden import H, load_golden


@pytest.fixture(scope="module")
def env(pkg):
    import __graft_entry__ as ge
    engine_mod = importlib.import_module("python-paillier_b200.engine")
    engine_mod._set_engine_for_tests(pkg.Engine(ge.build_hostsim()))
    yield importlib.import_module("python-paillier_b200.util"), engine_mod
    engine_mod._set_engine_for_tests(None)


def test_miller_rabin_batch_agrees_with_the_reference(pkg, env):
    """Verdicts of the reference's is_prime on the same candidates are stored in tests/golden/is_prime_reference.json."""
    util, engine_mod = env
    fx = load_golden("is_prime_reference.json")
    primes, composites, randoms = ([H(c) for c in fx[k]] for k in ("known_primes", "known_composites", "random"))
    got = util.is_prime_batch(primes + composites + randoms)
    assert got == fx["is_prime"]
    assert got[:len(primes)] == [True] * len(primes) and not any(got[len(primes):len(primes) + len(composites)])
    # raw kernel on survivors only (no trial division): the pseudoprimes must still fall to random bases
    raw = engine_mod.miller_rabin_batch([3215031751, 2 ** 127 - 1, 3825123056546413051, 318665857834031151167461, 2 ** 61 - 1], rounds=25)
    assert raw == [False, True, False, False, True]


def test_batched_keygen(pkg, env):
    util, _ = env
    ps = util.getprimeover_batch(160, 5)
    assert len(ps) == 5 and len(set(ps)) == 5 and all(p.bit_length() == 160 and util.is_prime(p) for p in ps)
    keys = pkg.generate_paillier_keypairs(3, n_length=320)
    assert len({pk.n for pk, _ in keys}) == 3
    for pk, sk in keys:
        assert pk.n.bit_length() == 320 and sk.p * sk.q == pk.n
        assert sk.decrypt(pk.encrypt(-12.5) + 3) == -9.5
    pk, sk = pkg.generate_paillier_keypair(n_length=512)        # the scalar entry point keeps the reference's host-side loop
    assert pk.n.bit_length() == 512 and sk.decrypt(pk.encrypt(7)) == 7
