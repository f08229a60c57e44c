"""Cases and reference for the field-arithmetic conformance tests (test_field_conformance.py).

The device probe (csrc/field_probe.cuh: sso_test_field_op on the GPU, emul_field_op_raw in tests/emul) takes and returns raw
little-endian Montgomery words.  Here a raw word string x stands for the value x R^-1 mod p (R = 2^(32 L)), so unreduced operands
(x >= p) are other representatives of the same value.  Every output is checked two ways: its value against oracle.fields, and its
representation — every coefficient below p — which the byte interface (from_mont rounds anything below 2 p) cannot observe.

The module also restates, in Python, the predicate each data-dependent conditional of the device code takes (the final
subtractions, the quotient estimate of reduce_small, the exit of the binary inversion, the branches of the square roots), so that
the tests can assert that every side of each is reached on every field instead of hoping random operands reach it.
"""
from __future__ import annotations

import random
from dataclasses import dataclass

from oracle.curves import get_curve

# field ids of the probe (also the emulator's emul_field_op ids)
FIELDS = {0: ("bls12_377", "Fr"), 1: ("bls12_377", "Fq"), 2: ("bw6_761", "Fq"), 3: ("mnt4_753", "Fq"), 4: ("mnt6_753", "Fq"),
          5: ("bls12_377", "g2"), 6: ("mnt4_753", "g2"), 7: ("mnt6_753", "g2"),
          8: ("bls12_377", "g2"), 9: ("mnt4_753", "g2"), 10: ("mnt6_753", "g2")}
COOP = {8: 5, 9: 6, 10: 7}                                   # cooperative field -> the one-thread-per-element field

OPS = {"mul": 0, "add": 1, "sub": 2, "sqr": 3, "neg": 4, "inv": 5, "sqr_dedicated": 6, "lex_is_neg": 7, "sqrt": 8,
       "reduce_small": 9, "mad_small_lazy": 10, "conj": 11, "mul_base": 12, "mul_u2": 13, "frob_w": 14}
RC_UNSUPPORTED = 0xFFFFFFFF
_COMMON = {"mul", "add", "sub", "sqr", "neg", "inv", "sqr_dedicated"}
# the (field, op) pairs the probe implements; every other pair must answer RC_UNSUPPORTED
SUPPORTED = {0: _COMMON | {"lex_is_neg", "sqrt"},
             **{f: _COMMON | {"lex_is_neg", "sqrt", "reduce_small", "mad_small_lazy"} for f in (1, 2, 3, 4)},
             5: _COMMON | {"lex_is_neg", "sqrt", "conj", "mul_base"}, 6: _COMMON | {"lex_is_neg", "sqrt", "conj", "mul_base"},
             7: _COMMON | {"lex_is_neg", "sqrt", "mul_base", "mul_u2", "frob_w"},
             8: _COMMON | {"conj", "mul_base"}, 9: _COMMON | {"conj", "mul_base"}, 10: _COMMON | {"mul_base", "mul_u2", "frob_w"}}
UNARY = {"sqr", "neg", "inv", "sqr_dedicated", "lex_is_neg", "sqrt", "reduce_small", "conj", "mul_u2", "frob_w"}

# Unreduced-operand contracts as the code states them (coefficients below A p and B p):
#   base mont_mul: A B p < R (the table of test_emul_device_code.py::test_unreduced_operands_at_their_bounds)
#   dedicated squaring: A^2 p < R
#   Fq2 over the 377-bit field (u^2 = -5): mul 4 A B p < R (A B <= 38), sqr A <= 3 (ext.cuh: 6 p * 23 p = 138 p^2 < p R)
#   Fq2 over the 753-bit field (u^2 = 13), plain and cooperative: A B <= 58 (mul), A <= 29 (sqr)
#   Fq3 (u^3 = 11), plain and cooperative: A, B <= 8
# The cooperative BLS12-377 Fq2 (negative non-residue) takes canonical operands only.
BASE_MUL_BOUNDS = {1: [(6, 23), (4, 6), (3, 3), (2, 12)], 2: [(3, 3), (4, 4), (4, 2), (15, 15)],
                   3: [(58, 406), (29, 26), (14, 14), (125, 2), (192, 192)], 4: [(58, 406), (29, 26), (14, 14), (125, 2), (192, 192)]}
EXT_MUL_BOUNDS = {5: [(3, 12), (12, 3), (3, 3)], 6: [(29, 2), (2, 29), (7, 8)], 7: [(8, 8), (8, 1)],
                  9: [(29, 2), (2, 29), (7, 8)], 10: [(8, 8), (8, 1)]}
EXT_SQR_BOUND = {5: 3, 6: 29, 7: 8, 9: 29, 10: 8}
MAD_SMALL_KS = (2, 5, 11, 13, 26)                            # the factors the code passes (a, NR, coop rows, a' = 26)


@dataclass
class Field:
    fid: int
    F: object                                                # oracle field (Fp or ExtField)
    p: int
    deg: int
    L: int                                                   # limbs per coefficient
    coop: bool

    def __post_init__(self):
        self.R = 1 << (32 * self.L)
        self.Rinv = pow(self.R, -1, self.p)
        self.pinv = pow(self.p, -1, self.R)

    @property
    def words(self):
        return self.deg * self.L

    def val(self, x):
        """value of raw coefficients (tuple) -> oracle element"""
        v = tuple(c * self.Rinv % self.p for c in x)
        return v[0] if self.deg == 1 else v

    def raw(self, v):
        """oracle element -> canonical raw coefficients"""
        cs = (v,) if self.deg == 1 else v
        return tuple(c * self.R % self.p for c in cs)


def field(fid) -> Field:
    name, which = FIELDS[fid]
    c = get_curve(name)
    F = c.g2.F if which == "g2" else getattr(c, which)
    base = F if F.deg == 1 else F.base
    return Field(fid, F, base.p, F.deg, (base.bits + 31) // 32, fid in COOP)


@dataclass
class Case:
    op: str
    a: tuple
    b: tuple
    k: int = 0
    tag: str = ""


# ---------------------------------------------------------------------------------------------------------------------------
# restated device predicates
# ---------------------------------------------------------------------------------------------------------------------------
def mont_u(fd: Field, a: int, b: int) -> int:
    """CIOS / dedicated-squaring value before the final conditional subtraction: (a b + m p) / R, m = -a b p^-1 mod R"""
    R, p = fd.R, fd.p
    m = (-a * b * fd.pinv) % R
    u = a * b + m * p
    assert u % R == 0
    return u // R


def reduce_small_short(fd: Field, y: int) -> bool:
    """reduce_small: the top-limb quotient estimate is one short (the final subtraction is taken)"""
    sh = 32 * (fd.L - 1)
    q = (y >> sh) // ((fd.p >> sh) + 1)
    d = y - q * fd.p
    assert 0 <= d < 2 * fd.p
    return d >= fd.p


def inv_ends_through_u(fd: Field, a: int) -> bool:
    """Fp::inv (binary extended Euclid on the raw residue): does the loop end with u = 1 (else v = 1)?"""
    u, v = a, fd.p
    while u != 1 and v != 1:
        while u % 2 == 0:
            u //= 2
        while v % 2 == 0:
            v //= 2
        if u >= v:
            u -= v
        else:
            v -= u
    return u == 1


def ts_first_k(Fb, a: int) -> int:
    """Tonelli-Shanks on a residue a != 0: log2 of the order of b = a^t, the depth of the first outer iteration"""
    b, k = pow(a, Fb.t_odd, Fb.p), 0
    while b != 1:
        b, k = b * b % Fb.p, k + 1
    return k


def fp2_sqrt(fd: Field, a):
    """ext.cuh Fp2::sqrt restated on values with the base field's Tonelli-Shanks (the device's z = smallest non-residue ^ t, as
    oracle.fields): (branch, root or None).  branch: c1=0/residue, c1=0/non-residue, delta, delta-fallback, norm-non-residue."""
    Fb, nr = fd.F.base, fd.F.nr
    p = fd.p
    a0, a1 = a
    if a1 == 0:
        r = Fb.sqrt(a0)
        if r is not None:
            return "c1=0/residue", (r, 0)
        r = Fb.sqrt(a0 * pow(nr, -1, p) % p)
        return "c1=0/non-residue", (None if r is None else (0, r))
    norm = (a0 * a0 - nr * a1 * a1) % p
    s = Fb.sqrt(norm)
    if s is None:
        return "norm-non-residue", None
    h = pow(2, -1, p)
    branch = "delta"
    c0 = Fb.sqrt((a0 + s) * h % p)
    if c0 is None:
        branch = "delta-fallback"
        c0 = Fb.sqrt((a0 - s) * h % p)
        assert c0 is not None
    return branch, (c0, a1 * pow(2 * c0, -1, p) % p)


def predicates(fd: Field, cs) -> dict:
    """{predicate: {side: count}} over the cases of one field, for the conditionals of the device code"""
    hit = {}

    def mark(name, side):
        hit.setdefault(name, {}).setdefault(side, 0)
        hit[name][side] += 1

    p = fd.p
    for c in cs:
        if fd.deg == 1:
            a, b = c.a[0], c.b[0]
            if c.op == "add":
                s = a + b
                mark("add: s >= p", "s = p" if s == p else ("s > p" if s > p else "s < p"))
            elif c.op == "sub":
                mark("sub: borrow", "a = b" if a == b else ("borrow" if a < b else "no borrow"))
            elif c.op == "neg":
                mark("neg: zero", "zero" if a == 0 else "non-zero")
            elif c.op in ("mul", "sqr_dedicated"):
                u = mont_u(fd, a, b if c.op == "mul" else a)
                mark(c.op + ": u >= p", "u = p" if u == p else ("u > p" if u > p else "u < p"))
            elif c.op == "reduce_small":
                mark("reduce_small: estimate", "one short" if reduce_small_short(fd, a) else "exact")
            elif c.op == "inv" and a % p:
                mark("inv: exit", "u = 1" if inv_ends_through_u(fd, a) else "v = 1")
            elif c.op == "sqrt" and fd.F.two_adicity > 1:
                v = fd.val(c.a)
                if v and fd.F.legendre(v) == 1:
                    mark("sqrt: first Tonelli-Shanks depth", ts_first_k(fd.F, v))
        elif fd.deg == 2 and c.op == "sqrt":
            mark("Fp2::sqrt", fp2_sqrt(fd, fd.val(c.a))[0])
    return hit


def required_sides(fd: Field) -> dict:
    req = {}
    if fd.deg == 1:
        req = {"add: s >= p": {"s = p", "s > p", "s < p"}, "sub: borrow": {"a = b", "borrow", "no borrow"},
               "neg: zero": {"zero", "non-zero"}, "mul: u >= p": {"u = p", "u > p", "u < p"},
               "sqr_dedicated: u >= p": {"u = p", "u > p", "u < p"}, "inv: exit": {"u = 1", "v = 1"}}
        if "reduce_small" in SUPPORTED[fd.fid]:
            req["reduce_small: estimate"] = {"one short", "exact"}
        if fd.F.two_adicity > 1:
            req["sqrt: first Tonelli-Shanks depth"] = set(range(fd.F.two_adicity))
    elif fd.deg == 2 and not fd.coop:
        req["Fp2::sqrt"] = {"c1=0/residue", "c1=0/non-residue", "delta", "delta-fallback", "norm-non-residue"}
    return req


# ---------------------------------------------------------------------------------------------------------------------------
# reference
# ---------------------------------------------------------------------------------------------------------------------------
def frob_consts(fd: Field):
    w1 = pow(fd.F.nr, (fd.p - 1) // 3, fd.p)
    return w1, w1 * w1 % fd.p


def check(fd: Field, c: Case, out: tuple, rc: int):
    """None if the probe's (out, rc) is right for case c, else a description of what is wrong"""
    F, p = fd.F, fd.p
    if c.op not in SUPPORTED[fd.fid]:
        return None if rc == RC_UNSUPPORTED else "rc %#x for an unsupported op" % rc
    if c.op == "reduce_small":
        return None if out == (c.a[0] % p,) else "value"
    if c.op == "mad_small_lazy":
        return None if out == (c.a[0] + c.k * c.b[0],) else "value"
    x, y = fd.val(c.a), fd.val(c.b)
    want_rc = 0
    if c.op == "lex_is_neg":
        return None if rc == (1 if F.gt(x, F.neg(x)) else 0) and out == c.a else "rc %d / out" % rc
    if c.op == "sqrt":
        leg = F.legendre(x)
        if rc != (0 if leg == -1 else 1):
            return "verdict %d for Legendre symbol %d" % (rc, leg)
        if rc == 0:
            return None
        if any(w >= p for w in out):
            return "root not canonical"
        if F.sqr(fd.val(out)) != x:
            return "root squared differs"
        want = F.sqrt(x) if fd.deg == 1 else (fp2_sqrt(fd, x)[1] if fd.deg == 2 else None)
        if want is not None and fd.raw(want) != out:
            return "not the restated root"
        return None
    if c.op in ("mul",):
        v = F.mul(x, y)
    elif c.op == "add":
        v = F.add(x, y)
    elif c.op == "sub":
        v = F.sub(x, y)
    elif c.op in ("sqr", "sqr_dedicated"):
        v = F.sqr(x)
    elif c.op == "neg":
        v = F.neg(x)
    elif c.op == "inv":
        v = F.zero if F.is_zero(x) else F.inv(x)          # inv(0) = 0 on the device
    elif c.op == "conj":
        v = (x[0], (-x[1]) % p)
    elif c.op == "mul_base":
        k = c.b[0] * fd.Rinv % p
        v = tuple(e * k % p for e in x)
    elif c.op == "mul_u2":
        v = F.mul(x, (0, 0, 1))
    elif c.op == "frob_w":
        w1, w2 = frob_consts(fd)
        v = (x[0], x[1] * w1 % p, x[2] * w2 % p)
    else:
        raise AssertionError(c.op)
    if rc != want_rc:
        return "rc %d" % rc
    want = fd.raw(v)
    if tuple(w % p for w in out) != want:
        return "value"
    if out != want:
        return "representation: coefficient >= p"
    return None


# ---------------------------------------------------------------------------------------------------------------------------
# operands
# ---------------------------------------------------------------------------------------------------------------------------
def base_edges(fd: Field, rnd) -> list:
    """edge residues, as raw Montgomery words (all below p)"""
    p, L, R = fd.p, fd.L, fd.R
    top = p >> (32 * (L - 1))
    e = [0, 1, 2, p - 1, p - 2, (p - 1) // 2, (p + 1) // 2, R % p, R * R % p, (top << (32 * (L - 1))) - 1]
    for i in range(1, L):
        e += [1 << (32 * i), (1 << (32 * i)) - 1, p - (1 << (32 * i))]
    ones = (1 << (32 * L)) - 1
    for j in (1, 2, L // 2, L - 1):                           # runs of 0xffffffff limbs, at the bottom and below the top limb
        e += [(1 << (32 * j)) - 1, ((1 << (32 * j)) - 1) << (32 * (L - 1 - j))]
    alt = sum(0xFFFFFFFF << (64 * i) for i in range(L // 2))
    e += [alt & ((1 << (p.bit_length() - 1)) - 1), (alt << 32) & ((1 << (p.bit_length() - 1)) - 1), ones % p]
    e += [rnd.randrange(p) for _ in range(4)]
    out = []
    for x in e:
        if 0 <= x < p and x not in out:
            out.append(x)
    return out


def elem_edges(fd: Field, rnd) -> list:
    """edge elements (tuples of raw coefficients)"""
    be = base_edges(fd, rnd)
    if fd.deg == 1:
        return [(x,) for x in be]
    p = fd.p
    coef = [0, p - 1, fd.R % p, None]                       # None: random
    out = []
    for m in range(len(coef) ** fd.deg):
        t, cs = m, []
        for _ in range(fd.deg):
            c = coef[t % len(coef)]
            cs.append(rnd.randrange(p) if c is None else c)
            t //= len(coef)
        out.append(tuple(cs))
    out += [tuple(rnd.choice(be) for _ in range(fd.deg)) for _ in range(8)]
    return out


def relem(fd: Field, rnd):
    return tuple(rnd.randrange(fd.p) for _ in range(fd.deg))


def sqrt_cases(fd: Field, rnd, n_random: int) -> list:
    F, p = fd.F, fd.p
    cs = []
    if fd.deg == 1:
        s = F.two_adicity
        if s > 1:
            z = pow(F._nonresidue(), F.t_odd, p)              # order 2^s
            for j in range(1, s + 1):                         # a = (g w)^2, g of order 2^j, w of odd order: first depth j - 1
                g = pow(z, 1 << (s - j), p)
                w = pow(rnd.randrange(1, p), 1 << s, p)
                cs.append(F.sqr(g * w % p))
        nq = F._nonresidue()
        cs += [0, 1, p - 1, nq, nq * nq % p] + [rnd.randrange(p) for _ in range(n_random)]
        return [Case("sqrt", fd.raw(v), (0,), tag="sqrt") for v in cs]
    Fb = F.base
    qr = [x for x in (rnd.randrange(1, p) for _ in range(40)) if Fb.legendre(x) == 1][:3]
    nq = [x for x in (rnd.randrange(1, p) for _ in range(40)) if Fb.legendre(x) == -1][:3]
    els = [F.zero, F.one] + [(x,) + (0,) * (fd.deg - 1) for x in qr + nq]
    els += [F.sqr(relem(fd, rnd)) for _ in range(n_random)] + [relem(fd, rnd) for _ in range(n_random)]
    if fd.deg == 2:
        # enough squares with c1 != 0 that both delta branches appear, and non-squares for the norm branch
        br = {}
        while len(br) < 5 or min(br.values()) < 2:
            v = relem(fd, rnd) if rnd.random() < 0.5 else F.sqr(relem(fd, rnd))
            if rnd.random() < 0.2:
                v = (v[0], 0)
            b = fp2_sqrt(fd, v)[0]
            if br.get(b, 0) < 2:
                els.append(v)
            br[b] = br.get(b, 0) + 1
    return [Case("sqrt", fd.raw(v), (0,) * fd.deg, tag="sqrt") for v in els]


def cases(fid: int, volume: str = "emul", seed: int = 0) -> list:
    """the cases of one field; volume "emul" keeps the CPU run short, "gpu" adds >= 2^16 random products and squarings and
    several thousand cases per op"""
    fd = field(fid)
    rnd = random.Random(1000 * fid + seed)
    p, deg, R = fd.p, fd.deg, fd.R
    big = volume == "gpu"
    E = elem_edges(fd, rnd)
    zero = (0,) * deg
    out = []
    ops = sorted(SUPPORTED[fid] - {"sqrt", "reduce_small", "mad_small_lazy"})
    # every supported op on every edge operand, against every edge (binary ops) or a random partner
    Eb = E if big or deg == 1 and fd.L <= 12 else E[:: max(1, len(E) // 24)]
    for op in ops:
        if op in UNARY:
            out += [Case(op, a, relem(fd, rnd), tag="edge") for a in E]
        else:
            out += [Case(op, a, b, tag="edge") for a in E for b in Eb]
    nr = 4096 if big else 24
    for op in ops:
        out += [Case(op, relem(fd, rnd), relem(fd, rnd), tag="random") for _ in range(nr)]
    if big:
        out += [Case(op, relem(fd, rnd), relem(fd, rnd), tag="random block") for op in ("mul", "sqr") for _ in range(1 << 16)]
    if deg == 1:
        # constructed: mont_mul / squaring with a pre-subtraction value u > p (u = p + t, t small), and u = p - 1
        for t in range(1, 6):
            b = rnd.randrange(p // 2, p)
            a = t * R * pow(b, -1, p) % p
            out.append(Case("mul", (a,), (b,), tag="u > p"))
            for _ in range(64):
                s = rnd.randrange(1, p)
                r = fd.F.sqrt(t * R * pow(s * s, -1, p) % p)
                if r is not None:
                    out.append(Case("sqr_dedicated", (r * s % p,), zero, tag="u > p"))
                    break
        out.append(Case("mul", (-(-R // p) * p - R,), (1,), tag="u = p - 1"))
        out.append(Case("mul", (1,), (-(-R // p) * p - R,), tag="u = p - 1"))
        # unreduced zeros p, 2 p, ... where unreduced operands are admitted: the pre-subtraction value is exactly p
        ratio = R // p
        for kz in range(1, min(ratio, 8)):
            if (kz + 1) * p < R and (kz + 1) <= ratio:
                out += [Case("mul", (kz * p,), (1,), tag="unreduced zero"), Case("mul", (rnd.randrange(p),), (kz * p,), tag="unreduced zero")]
            if (kz + 1) ** 2 <= ratio:
                out.append(Case("sqr_dedicated", (kz * p,), zero, tag="unreduced zero"))
        # binary inversion exits: make sure both appear (a = 1 ends through u at once; p - 1 reaches v = 1 first on these primes)
        out += [Case("inv", (a,), zero, tag="inv exit") for a in (1, 2, p - 1, (p + 1) // 2, R % p)]
        out += [Case("add", (1,), (p - 1,), tag="s = p"), Case("add", ((p + 1) // 2,), ((p - 1) // 2,), tag="s = p")]
        out += [Case("sub", (a,), (a,), tag="a = b") for a in (0, 1, p - 1)]
    if fid in BASE_MUL_BOUNDS:
        for A, B in BASE_MUL_BOUNDS[fid]:
            assert A * B * p < R
            prs = [(A * p - 1, B * p - 1), ((A - 1) * p + rnd.randrange(p), (B - 1) * p + rnd.randrange(p)), (A * p - 1, 1),
                   (0, B * p - 1), ((A - 1) * p, B * p - 1), (A * p - 1, (B - 1) * p),
                   (min(A * p - 1, (1 << (A * p).bit_length() - 1) - 1), min(B * p - 1, (1 << (B * p).bit_length() - 1) - 1))]
            out += [Case("mul", (a,), (b,), tag="unreduced %dp x %dp" % (A, B)) for a, b in prs]
        for A in (2, 3, 4):
            assert A * A * p < R
            out += [Case("sqr_dedicated", (a,), zero, tag="unreduced %dp" % A) for a in (A * p - 1, (A - 1) * p + rnd.randrange(p), (A - 1) * p)]
    if "reduce_small" in SUPPORTED[fid]:
        ys = [k * p + d for k in range(17) for d in (-1, 0, 1) if 0 <= k * p + d < 16 * p]
        ys += [rnd.randrange(16 * p) for _ in range(200 if big else 20)]
        out += [Case("reduce_small", (y,), zero, tag="reduce_small") for y in ys]
        for k in MAD_SMALL_KS:
            assert (k + 1) * p < R
            for c, x in ((p - 1, p - 1), (0, p - 1), (p, p), (rnd.randrange(p), rnd.randrange(p)), (p - 1, 0), (0, p)):
                out.append(Case("mad_small_lazy", (c,), (x,), k, tag="mad_small_lazy k=%d" % k))
    if fid in EXT_MUL_BOUNDS:
        def coef_below(A):
            return [A * p - 1, (A - 1) * p + rnd.randrange(p), (A - 1) * p, rnd.randrange(A * p)]
        for A, B in EXT_MUL_BOUNDS[fid]:
            for _ in range(6 if big else 3):
                a = tuple(rnd.choice(coef_below(A)) for _ in range(deg))
                b = tuple(rnd.choice(coef_below(B)) for _ in range(deg))
                out.append(Case("mul", a, b, tag="unreduced %dp x %dp" % (A, B)))
            out.append(Case("mul", (A * p - 1,) * deg, (B * p - 1,) * deg, tag="unreduced %dp x %dp" % (A, B)))
            out.append(Case("mul", ((A - 1) * p,) * deg, (B * p - 1,) * deg, tag="unreduced zero"))
        A = EXT_SQR_BOUND[fid]
        for a in [(A * p - 1,) * deg, ((A - 1) * p,) * deg] + [tuple(rnd.choice(coef_below(A)) for _ in range(deg)) for _ in range(6)]:
            out += [Case("sqr", a, zero, tag="unreduced %dp" % A), Case("sqr_dedicated", a, zero, tag="unreduced %dp" % A)]
    if "sqrt" in SUPPORTED[fid]:
        out += sqrt_cases(fd, rnd, 8 if not big else 64)
    out += named_regressions(fid)
    return out


def named_regressions(fid: int) -> list:
    """inputs of bugs this suite has found, kept by name"""
    return []


def unsupported_cases(fid: int) -> list:
    fd = field(fid)
    one = (1,) + (0,) * (fd.deg - 1)
    return [Case(op, one, one, 1, tag="unsupported") for op in sorted(set(OPS) - SUPPORTED[fid])]


# ---------------------------------------------------------------------------------------------------------------------------
# packing for the probe
# ---------------------------------------------------------------------------------------------------------------------------
def pack(fd: Field, cs):
    """(ops, a, b, k) as lists of uint32"""
    L = fd.L
    ops, a, b, k = [], [], [], []
    for c in cs:
        ops.append(OPS[c.op])
        k.append(c.k)
        for src, dst in ((c.a, a), (c.b, b)):
            src = tuple(src) + (0,) * (fd.deg - len(src))
            for x in src:
                dst += [(x >> (32 * i)) & 0xFFFFFFFF for i in range(L)]
    return ops, a, b, k


def unpack(fd: Field, words, n):
    L = fd.L
    res = []
    for i in range(n):
        e = words[i * fd.words:(i + 1) * fd.words]
        res.append(tuple(sum(int(e[j * L + w]) << (32 * w) for w in range(L)) for j in range(fd.deg)))
    return res
