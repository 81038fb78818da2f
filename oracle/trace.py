"""Call traces of the reference's public API (TEST INFRASTRUCTURE).

tests/golden/make_upstream_traces.py records, while the reference's own unit tests run on the reference, every call
the test code makes into the phe API and every call phe makes into its bigint seam, with arguments and results.  The
tests replay those calls on this package (or through integration/phe_b200_backend.py) and compare the results.
Values are stored by what they hold, not by class, so that one encoding serves both packages."""


class Unsupported(Exception):
    """A value the trace format does not hold (the call is left out of the trace)."""


def _hx(v):
    return "-" + hex(-v) if v < 0 else hex(v)


def _int(s):
    return -int(s[1:], 16) if s.startswith("-") else int(s, 16)


def _kind(x):
    names = {c.__name__ for c in type(x).__mro__}
    for k in ("EncryptedNumber", "EncodedNumber", "PaillierPublicKey", "PaillierPrivateKey"):
        if k in names:
            return k
    return None


def dump(x):
    """A value -> JSON-able list."""
    if x is None:
        return ["none"]
    if isinstance(x, bool):
        return ["bool", x]
    if isinstance(x, int):
        return ["int", _hx(x)]
    if isinstance(x, float) or type(x).__name__ in ("float64", "float32"):
        return ["float", repr(float(x))]
    if isinstance(x, str):
        return ["str", x]
    if isinstance(x, bytes):
        return ["bytes", x.hex()]
    if isinstance(x, type) and "EncodedNumber" in {c.__name__ for c in x.__mro__}:
        return ["encoded_cls", x.BASE]
    k = _kind(x)
    if k == "EncryptedNumber":
        return ["encrypted", _hx(x.public_key.n), _hx(x.ciphertext(be_secure=False)), x.exponent]
    if k == "EncodedNumber":
        return ["encoded", _hx(x.public_key.n), _hx(x.encoding), x.exponent, type(x).BASE]
    if k == "PaillierPublicKey":
        return ["pk", _hx(x.n)]
    if k == "PaillierPrivateKey":
        return ["sk", _hx(x.public_key.n)]
    raise Unsupported(type(x).__name__)


class Loader:
    """JSON-able lists -> objects of a package with the phe API (`pkg.PaillierPublicKey`, `pkg.EncodedNumber`, ...);
    `keys` maps hex(n) to (hex(p), hex(q))."""

    def __init__(self, pkg, keys):
        self.pkg, self.keys, self.pks, self.sks, self.classes = pkg, keys, {}, {}, {}

    def pk(self, n):
        if n not in self.pks:
            self.pks[n] = self.pkg.PaillierPublicKey(_int(n))
        return self.pks[n]

    def sk(self, n):
        if n not in self.sks:
            p, q = self.keys[n]
            self.sks[n] = self.pkg.PaillierPrivateKey(self.pk(n), _int(p), _int(q))
        return self.sks[n]

    def encoded_cls(self, base):
        import math
        if base == self.pkg.EncodedNumber.BASE:
            return self.pkg.EncodedNumber
        if base not in self.classes:
            self.classes[base] = type("EncodedNumberBase%d" % base, (self.pkg.EncodedNumber,),
                                      {"BASE": base, "LOG2_BASE": math.log(base, 2)})
        return self.classes[base]

    def load(self, v):
        t = v[0]
        if t == "none":
            return None
        if t in ("bool", "str"):
            return v[1]
        if t == "int":
            return _int(v[1])
        if t == "float":
            return float(v[1])
        if t == "bytes":
            return bytes.fromhex(v[1])
        if t == "encoded_cls":
            return self.encoded_cls(v[1])
        if t == "encrypted":
            return self.pkg.EncryptedNumber(self.pk(v[1]), _int(v[2]), v[3])
        if t == "encoded":
            return self.encoded_cls(v[4])(self.pk(v[1]), _int(v[2]), v[3])
        if t == "pk":
            return self.pk(v[1])
        if t == "sk":
            return self.sk(v[1])
        raise ValueError(t)
