"""phase2_cli::prepare_phase2 restated for the tests: the radix-2 evaluation domain of ark-poly, a plain recursive group FFT over
oracle points, the Groth16Params container and the transform of a Full-mode accumulator.  Scalar multiplications go through the
C++ leg of the oracle (oracle/cport.py); additions, negations and the bookkeeping are the Python group law.

[UP] as recalled, isolated in snark-setup-operator_b200/csrc/p2prep.cuh: w = GENERATOR^((r - 1) / m) with ark-ff's generator
constants below, the output order of setup_utils::Groth16Params, uncompressed without length prefixes."""
from __future__ import annotations

from dataclasses import dataclass

from oracle import cport, serialize as ser
from oracle.curves import Curve

FR_GENERATOR = {"bls12_377": 22, "bw6_761": 15, "mnt4_753": 17, "mnt6_753": 17}


def two_adicity(curve: Curve) -> int:
    s, t = 0, curve.Fr.p - 1
    while t % 2 == 0:
        s, t = s + 1, t // 2
    return s


def domain_generator(curve: Curve, m: int) -> int:
    """ark-poly Radix2EvaluationDomain::new(m).group_gen for a power of two m <= 2^s."""
    r = curve.Fr.p
    assert m & (m - 1) == 0 and (r - 1) % m == 0
    return pow(FR_GENERATOR[curve.name], (r - 1) // m, r)


def mul(curve: Curve, group: int, P, k: int):
    G = (curve.g1, curve.g2)[group]
    k %= curve.Fr.p
    if P is None or k == 0:
        return None
    if k == 1:
        return P
    out = cport.batch_exp(curve, group, ser.point_to_bytes(G, P, False), 1, 0, 1, k, mode=1, out_compressed=False)
    return ser.point_from_bytes(G, out, False)


def group_fft(curve: Curve, group: int, pts, omega: int):
    """out_i = sum_j omega^(ij) pts_j (recursive radix-2 decimation in time)."""
    G = (curve.g1, curve.g2)[group]
    n = len(pts)
    if n == 1:
        return list(pts)
    r = curve.Fr.p
    even = group_fft(curve, group, pts[0::2], omega * omega % r)
    odd = group_fft(curve, group, pts[1::2], omega * omega % r)
    out = [None] * n
    w = 1
    for k in range(n // 2):
        t = mul(curve, group, odd[k], w)
        out[k] = G.add(even[k], t)
        out[k + n // 2] = G.add(even[k], G.neg(t))
        w = w * omega % r
    return out


def group_ifft(curve: Curve, group: int, pts):
    """IFFT(x)_i = m^-1 sum_j w^(-ij) x_j over the size-m domain."""
    m, r = len(pts), curve.Fr.p
    y = group_fft(curve, group, pts, pow(domain_generator(curve, m), -1, r))
    minv = pow(m, -1, r)
    return [mul(curve, group, P, minv) for P in y]


def lagrange_at(curve: Curve, s: int, m: int):
    """L_i(s) = w^i (s^m - 1) / (m (s - w^i)) over the size-m domain; L_i(w^k) = [i = k] at a domain point."""
    r = curve.Fr.p
    w = domain_generator(curve, m)
    pts = [pow(w, i, r) for i in range(m)]
    s %= r
    if s in pts:
        return [int(x == s) for x in pts]
    return [x * (pow(s, m, r) - 1) * pow(m * (s - x), -1, r) % r for x in pts]


@dataclass
class Groth16Params:
    alpha_g1: object
    beta_g1: object
    beta_g2: object
    coeffs_g1: list
    coeffs_g2: list
    alpha_coeffs_g1: list
    beta_coeffs_g1: list
    h_g1: list

    def to_bytes(self, curve: Curve) -> bytes:
        g1, g2 = curve.g1, curve.g2
        return (ser.point_to_bytes(g1, self.alpha_g1, False) + ser.point_to_bytes(g1, self.beta_g1, False)
                + ser.point_to_bytes(g2, self.beta_g2, False) + ser.points_to_bytes(g1, self.coeffs_g1, False)
                + ser.points_to_bytes(g2, self.coeffs_g2, False) + ser.points_to_bytes(g1, self.alpha_coeffs_g1, False)
                + ser.points_to_bytes(g1, self.beta_coeffs_g1, False) + ser.points_to_bytes(g1, self.h_g1, False))

    @staticmethod
    def from_bytes(curve: Curve, buf: bytes, m: int) -> "Groth16Params":
        s1, s2 = ser.point_size(curve.g1, False), ser.point_size(curve.g2, False)
        o = [0]

        def take(G, sz, n):
            v = ser.points_from_bytes(G, buf[o[0]:o[0] + n * sz], False)
            o[0] += n * sz
            return v
        a, b = take(curve.g1, s1, 2)
        (b2,) = take(curve.g2, s2, 1)
        out = Groth16Params(a, b, b2, take(curve.g1, s1, m), take(curve.g2, s2, m), take(curve.g1, s1, m), take(curve.g1, s1, m),
                            take(curve.g1, s1, m - 1))
        assert o[0] == len(buf), "malformed Groth16Params"
        return out


def read_accumulator(curve: Curve, power: int, acc: bytes):
    """Full-mode accumulator (uncompressed) -> (tauG1, tauG2, alphaTauG1, betaTauG1, betaG2)."""
    s1, s2 = ser.point_size(curve.g1, False), ser.point_size(curve.g2, False)
    n1, n = (1 << (power + 1)) - 1, 1 << power
    o = 64
    out = []
    for G, sz, cnt in ((curve.g1, s1, n1), (curve.g2, s2, n), (curve.g1, s1, n), (curve.g1, s1, n), (curve.g2, s2, 1)):
        out.append(ser.points_from_bytes(G, acc[o:o + cnt * sz], False))
        o += cnt * sz
    assert o == len(acc)
    return out


def prepare_phase2(curve: Curve, power: int, accumulator: bytes, m: int) -> bytes:
    tg1, tg2, ag1, bg1, bg2 = read_accumulator(curve, power, accumulator)
    g1 = curve.g1
    h = [g1.add(tg1[i + m], g1.neg(tg1[i])) for i in range(m - 1)]
    return Groth16Params(ag1[0], bg1[0], bg2[0], group_ifft(curve, 0, tg1[:m]), group_ifft(curve, 1, tg2[:m]), group_ifft(curve, 0, ag1[:m]),
                         group_ifft(curve, 0, bg1[:m]), h).to_bytes(curve)


def synthetic_accumulator(curve: Curve, power: int, s: int, a: int, b: int) -> bytes:
    """Full-mode accumulator of a ceremony with tau = s, alpha = a, beta = b (hash slot zero)."""
    r = curve.Fr.p
    n1, n = (1 << (power + 1)) - 1, 1 << power
    gen1 = ser.point_to_bytes(curve.g1, curve.g1.gen, False)
    gen2 = ser.point_to_bytes(curve.g2, curve.g2.gen, False)
    be = lambda g, gb, cnt, coeff: cport.batch_exp(curve, g, gb * cnt, cnt, 0, s % r, coeff, out_compressed=False)
    return (bytes(64) + be(0, gen1, n1, None) + be(1, gen2, n, None) + be(0, gen1, n, a) + be(0, gen1, n, b)
            + cport.batch_exp(curve, 1, gen2, 1, 0, 1, b, mode=1, out_compressed=False))


def closed_form(curve: Curve, m: int, s: int, a: int, b: int) -> bytes:
    """prepare_phase2 of synthetic_accumulator(curve, p, s, a, b) from the Lagrange polynomials at s."""
    r = curve.Fr.p
    L = lagrange_at(curve, s, m)
    G1, G2 = curve.g1.gen, curve.g2.gen
    sm1 = (pow(s, m, r) - 1) % r
    return Groth16Params(mul(curve, 0, G1, a), mul(curve, 0, G1, b), mul(curve, 1, G2, b), [mul(curve, 0, G1, x) for x in L],
                         [mul(curve, 1, G2, x) for x in L], [mul(curve, 0, G1, a * x) for x in L], [mul(curve, 0, G1, b * x) for x in L],
                         [mul(curve, 0, G1, pow(s, i, r) * sm1) for i in range(m - 1)]).to_bytes(curve)
