#!/usr/bin/env python3
"""Generate the golden fixtures in tests/golden/ by running the UNMODIFIED reference.

It needs a checkout of python-paillier 1.5.0, named by PHE_SOURCE_DIR:

    PHE_SOURCE_DIR=<checkout> python tests/golden/make_golden.py            # writes tests/golden/*.json

Everything is produced by ``phe`` 1.5.0 imported from that checkout (pure-Python
bigint branch, phe/util.py:47-48 -- gmpy2 is not installable offline; both branches
return identical integers, see oracle/paillier_oracle.py).  Keys come from the
reference's own ``generate_paillier_keypair`` (phe/paillier.py:37-68) and are persisted
because it draws from ``SystemRandom``.  Integers are stored as hex strings.
"""
import json
import os
import random
import sys

sys.path.insert(0, os.environ["PHE_SOURCE_DIR"])
import phe                                            # noqa: E402
from phe import paillier, util                        # noqa: E402
import numpy as np                                    # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
assert not util.HAVE_GMP


def H(x):
    return hex(x)


def edge_plain(pk):
    n = pk.n
    return [0, 1, 2, n - 1, n - 2, pk.max_int, pk.max_int + 1, n - pk.max_int, n - pk.max_int - 1,
            n // 2, n, n + 1, 2 * n + 5, -1, -(n // 5)]


def make_key_fixture(kb, nvec, seed):
    pk, sk = paillier.generate_paillier_keypair(n_length=kb)
    rng = random.Random(seed)
    n, nsq = pk.n, pk.nsquare
    fx = {"key_bits": kb, "n": H(n), "p": H(sk.p), "q": H(sk.q),
          "psquare": H(sk.psquare), "qsquare": H(sk.qsquare), "p_inverse": H(sk.p_inverse),
          "hp": H(sk.hp), "hq": H(sk.hq), "max_int": H(pk.max_int), "phe_version": phe.__version__}

    # raw_encrypt / raw_decrypt (phe/paillier.py:102-139, 328-354)
    enc = []
    plains = edge_plain(pk) + [rng.randrange(0, n) for _ in range(nvec)]
    for i, m in enumerate(plains):
        r = rng.randrange(1, n)
        if i == 0:
            r = 1
        if i == 1:
            r = n - 1
        c = pk.raw_encrypt(m, r_value=r)
        d = sk.raw_decrypt(c)
        assert d == m % n
        enc.append({"m": H(m) if m >= 0 else "-" + H(-m), "r": H(r), "c": H(c), "d": H(d)})
    fx["encrypt"] = enc

    # raw_decrypt of arbitrary integers, incl. degenerate ones (no range check in the reference)
    dec = []
    for c in [0, 1, 2, n, sk.p, sk.q, sk.p * 3, sk.psquare, sk.qsquare * 2 % nsq, nsq - 1, nsq - n,
              (1 << (2 * kb)) - 1 if (1 << (2 * kb)) - 1 >= nsq else nsq - 2] + \
             [rng.randrange(0, nsq) for _ in range(nvec // 2)]:
        dec.append({"c": H(c), "d": H(sk.raw_decrypt(c))})
    fx["decrypt_any"] = dec

    # _raw_add (phe/paillier.py:705-719)
    e = paillier.EncryptedNumber(pk, 1, 0)
    add = []
    cts = [int(x["c"], 16) for x in enc]
    pairs = [(0, 0), (0, 1), (1, 1), (nsq - 1, nsq - 1), (nsq - 1, 1), (n, n), (n + 1, nsq - n - 1)]
    pairs += [(rng.choice(cts), rng.choice(cts)) for _ in range(nvec // 2)]
    pairs += [(rng.randrange(0, nsq), rng.randrange(0, nsq)) for _ in range(nvec // 2)]
    for a, b in pairs:
        add.append({"a": H(a), "b": H(b), "s": H(e._raw_add(a, b))})
    fx["add"] = add

    # _raw_mul (phe/paillier.py:721-751): positive, negative (invert branch) and edge scalars
    mul = []
    ks = [0, 1, 2, 3, 15, 16, 17, 255, 256, 2 ** 31, 2 ** 32 - 1, 2 ** 32, 2 ** 64 - 1, 2 ** 64, pk.max_int,
          pk.max_int + 1, n - pk.max_int - 1, n - pk.max_int, n - 1, n - 2, n - 2 ** 40, 16 ** 7, 16 ** 13]
    ks += [rng.getrandbits(rng.choice([8, 31, 32, 33, 53, 56, 63, 64, 65, 100, 256, kb // 2])) for _ in range(nvec // 2)]
    ks += [n - rng.getrandbits(rng.choice([8, 32, 53, 64, 100])) - 1 for _ in range(nvec // 4)]
    ks += [rng.randrange(0, n) for _ in range(4)]
    ks = [k % n for k in ks]
    for i, k in enumerate(ks):
        c = cts[(5 + i) % len(cts)] if i % 5 else rng.randrange(1, nsq)
        obj = paillier.EncryptedNumber(pk, c, 0)
        try:
            out = obj._raw_mul(k)
        except ZeroDivisionError:
            mul.append({"c": H(c), "k": H(k), "error": "ZeroDivisionError"})
            continue
        mul.append({"c": H(c), "k": H(k), "o": H(out)})
    # non-invertible ciphertexts on the negative branch -> ZeroDivisionError (phe/util.py:96-97,101-102)
    for c in [0, n, sk.p, sk.q * 7, sk.psquare]:
        obj = paillier.EncryptedNumber(pk, c, 0)
        try:
            out = obj._raw_mul(n - 5)
            mul.append({"c": H(c), "k": H(n - 5), "o": H(out)})
        except ZeroDivisionError:
            mul.append({"c": H(c), "k": H(n - 5), "error": "ZeroDivisionError"})
    fx["mul"] = mul

    # the three seam functions on this key's moduli (phe/util.py:38-103)
    seam = {"powmod": [], "mulmod": [], "invert": []}
    for _ in range(8):
        a, b = rng.randrange(0, nsq), rng.randrange(0, n)
        seam["powmod"].append({"a": H(a), "b": H(b), "c": H(nsq), "o": H(util.powmod(a, b, nsq))})
        a = rng.randrange(0, nsq)
        seam["powmod"].append({"a": H(a), "b": H(sk.p - 1), "c": H(sk.psquare), "o": H(util.powmod(a, sk.p - 1, sk.psquare))})
        a, b = rng.randrange(0, nsq), rng.randrange(0, nsq)
        seam["mulmod"].append({"a": H(a), "b": H(b), "c": H(nsq), "o": H(util.mulmod(a, b, nsq))})
        a = rng.randrange(1, nsq)
        try:
            seam["invert"].append({"a": H(a), "b": H(nsq), "o": H(util.invert(a, nsq))})
        except ZeroDivisionError:
            seam["invert"].append({"a": H(a), "b": H(nsq), "error": "ZeroDivisionError"})
    seam["powmod"].append({"a": H(1), "b": H(n), "c": H(nsq), "o": H(util.powmod(1, n, nsq))})
    seam["invert"].append({"a": H(sk.p), "b": H(sk.q), "o": H(util.invert(sk.p, sk.q))})
    fx["seam"] = seam
    return fx, pk, sk


def make_api_fixture(pk, sk, seed):
    """EncodedNumber / EncryptedNumber behaviour through the public API with injected r
    (phe/encoding.py:110-233, phe/paillier.py:145-194, 490-529, 570-601)."""
    rng = random.Random(seed)
    n = pk.n
    out = {"n": H(n), "p": H(sk.p), "q": H(sk.q), "encode": [], "ops": []}
    vals = [0, 1, -1, 2 ** 31 - 1, -2 ** 31, 12345678901234567890, 0.0, 1.0, -1.0, 3.141592653589793, -2.718281828459045,
            1e-10, -1e-10, 1e10, 1.5e300, 2.5e-300, 0.1, 0.2, 1 / 3, float(2 ** 53), 123456.789, -0.000123]
    vals += [rng.gauss(0, 0.1) for _ in range(20)] + [rng.randrange(-2 ** 40, 2 ** 40) for _ in range(10)]
    for v in vals:
        enc = phe.EncodedNumber.encode(pk, v)
        rec = {"v": repr(v), "encoding": H(enc.encoding), "exponent": enc.exponent, "decoded": repr(enc.decode())}
        if isinstance(v, float) and v != 0:
            for key, kw in (("prec_1e-6", {"precision": 1e-6}), ("maxexp_-20", {"max_exponent": -20})):
                try:
                    e2 = phe.EncodedNumber.encode(pk, v, **kw)
                    rec[key] = [H(e2.encoding), e2.exponent]
                except ValueError:
                    rec[key] = "ValueError"
        out["encode"].append(rec)
    # operator semantics with deterministic r: a+b, a+scalar, a*scalar, a-b, a/scalar
    pairs = [(1.5, 2.25), (3, 4), (-7, 2.5), (0.1, 0.2), (1e-5, 123456), (-1.25, -3.5), (2 ** 40, -0.375), (1e3, 1e-3)]
    for a, b in pairs:
        ra, rb = rng.randrange(1, n), rng.randrange(1, n)
        ea, eb = pk.encrypt(a, r_value=ra), pk.encrypt(b, r_value=rb)
        s, m, d, q = ea + eb, ea * b, ea - eb, ea / 4
        sc = ea + b
        out["ops"].append({
            "a": repr(a), "b": repr(b), "ra": H(ra), "rb": H(rb),
            "ea": [H(ea.ciphertext(False)), ea.exponent], "eb": [H(eb.ciphertext(False)), eb.exponent],
            "add": [H(s.ciphertext(False)), s.exponent, repr(sk.decrypt(s))],
            "add_scalar": [H(sc.ciphertext(False)), sc.exponent, repr(sk.decrypt(sc))],
            "mul": [H(m.ciphertext(False)), m.exponent, repr(sk.decrypt(m))],
            "sub": [H(d.ciphertext(False)), d.exponent, repr(sk.decrypt(d))],
            "div4": [H(q.ciphertext(False)), q.exponent, repr(sk.decrypt(q))],
        })
    return out


def make_config1(pk, sk):
    """BASELINE.json configs[0]: 1024-bit key, 256 int32 plaintexts, encrypt + decrypt round trip."""
    rng = random.Random(20240901)
    xs = np.random.RandomState(0).randint(-2 ** 31, 2 ** 31, 256).tolist()
    rows = []
    for x in xs:
        r = rng.randrange(1, pk.n)
        e = pk.encrypt(int(x), r_value=r)
        assert sk.decrypt(e) == x
        rows.append({"x": int(x), "r": H(r), "c": H(e.ciphertext(False)), "exponent": e.exponent})
    return {"n": H(pk.n), "p": H(sk.p), "q": H(sk.q), "rows": rows}


def make_is_prime():
    """The reference's probable-prime test (phe/util.py:421-443) on known primes, Carmichael numbers, strong
    pseudoprimes to small bases, semiprimes and random odd numbers (all above its small-prime table)."""
    rng = random.Random(5)
    primes = [2 ** 127 - 1, 2 ** 521 - 1, (1 << 255) - 19, 2 ** 89 - 1]
    carmichael = [561, 41041, 825265, 321197185, 5394826801, 232250619601, 9746347772161, 1436697831295441,
                  60977817398996785, 7156857700403137441, 1791562810662585767521, 87674969936234821377601]
    strong_pseudo = [3215031751, 3825123056546413051, 318665857834031151167461]   # strong pseudoprimes to bases 2, 3, 5, 7 (and more)
    semiprimes = [(2 ** 127 - 1) * ((1 << 255) - 19), (2 ** 89 - 1) * (2 ** 107 - 1)]
    composites = [c for c in carmichael + strong_pseudo + semiprimes if c > 20000]
    randoms = [rng.getrandbits(256) | 1 | (1 << 255) for _ in range(24)] + [rng.getrandbits(700) | 1 | (1 << 699) for _ in range(6)]
    return {"known_primes": [H(c) for c in primes], "known_composites": [H(c) for c in composites], "random": [H(c) for c in randoms],
            "is_prime": [bool(util.is_prime(c)) for c in primes + composites + randoms]}


def main():
    # the reference's own known answers (phe/tests/paillier_test.py:128-149, util_test.py:31-44)
    kat = {"n": 126869, "p": 293, "q": 433, "m": 10100, "r": 74384, "c": 935906717,
           "encrypt_1_r_1": 126870, "psquare": 85849, "qsquare": 187489, "p_inverse": 300, "hp": 203, "hq": 133,
           "powmod": [[5, 3, 3, 2], [2, 10, 1000, 24]],
           "invert_mod_101": [util.invert(a, 101) for a in range(1, 101)]}
    pk = paillier.PaillierPublicKey(126869)
    sk = paillier.PaillierPrivateKey(pk, 293, 433)
    assert pk.raw_encrypt(10100, 74384) == 935906717 and sk.raw_decrypt(935906717) == 10100
    assert (sk.psquare, sk.qsquare, sk.p_inverse, sk.hp, sk.hq) == (85849, 187489, 300, 203, 133)
    json.dump(kat, open(os.path.join(HERE, "kat_reference_tests.json"), "w"), indent=1)
    json.dump(make_is_prime(), open(os.path.join(HERE, "is_prime_reference.json"), "w"), indent=0)

    for kb, nvec in [(64, 32), (256, 32), (512, 32), (1024, 48), (2048, 32), (3072, 16), (4096, 8)]:
        fx, pk, sk = make_key_fixture(kb, nvec, seed=1000 + kb)
        json.dump(fx, open(os.path.join(HERE, "vectors_%d.json" % kb), "w"), indent=0)
        print("key", kb, "done", flush=True)
        if kb == 1024:
            json.dump(make_config1(pk, sk), open(os.path.join(HERE, "config1_1024.json"), "w"), indent=0)
            json.dump(make_api_fixture(pk, sk, 77), open(os.path.join(HERE, "api_1024.json"), "w"), indent=0)


if __name__ == "__main__":
    main()
