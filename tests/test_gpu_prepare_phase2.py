"""prepare_phase2 on the GPU (sso_group_fft_dev, sso_p2_prepare_buf / _file) against the restated transform
(tests/prepare_phase2_ref.py: plain group FFT and the Lagrange closed form), at toy sizes bit for bit and at 2^14 / 2^16 by
sampled one-point multiplications, the sum of the Lagrange basis and the forward transform back to the powers of tau."""
import os
import random

import pytest

import snark_setup_operator_b200 as sso
from oracle import serialize as ser
from oracle.curves import CURVE_NAMES, get_curve
from snark_setup_operator_b200 import phase2 as p2

import prepare_phase2_ref as R

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

REF_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")


def _scalars(c, seed):
    rnd = random.Random(seed)
    return [rnd.randrange(2, c.Fr.p) for _ in range(3)]


def _dev(b: bytes):
    return torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()


def _device_accumulator(name, power, s, a, b):
    """Full-mode accumulator with tau = s, alpha = a, beta = b, built from generator copies by the device batch_exp."""
    c = get_curve(name)
    n1, n = (1 << (power + 1)) - 1, 1 << power
    g1 = ser.point_to_bytes(c.g1, c.g1.gen, False)
    g2 = ser.point_to_bytes(c.g2, c.g2.gen, False)

    def powers(group, gb, cnt, coeff):
        d_in = _dev(gb * cnt)
        d_out = torch.empty_like(d_in)
        sso.batch_exp(name, group, d_in, cnt, 0, s, coeff, d_out, out_compressed=False)
        return d_out.cpu().numpy().tobytes()
    return (bytes(64) + powers(0, g1, n1, None) + powers(1, g2, n, None) + powers(0, g1, n, a) + powers(0, g1, n, b)
            + ser.point_to_bytes(c.g2, R.mul(c, 1, c.g2.gen, b), False))


@pytest.mark.parametrize("name", CURVE_NAMES)
def test_prepare_bytes_against_oracle(name):
    c = get_curve(name)
    s, a, b = _scalars(c, 1)
    acc = R.synthetic_accumulator(c, 5, s, a, b)
    p = sso.Phase1Parameters.new_full(name, 5, 4)
    for m in (1, 2, 8, 32):
        out = p2.prepare_phase2_buf(p, acc, m)
        assert out == R.closed_form(c, m, s, a, b), m
        if m <= 8:
            assert out == R.prepare_phase2(c, 5, acc, m), m


@pytest.mark.parametrize("name", ["bls12_377", "mnt4_753"])
def test_fresh_accumulator(tmp_path, name):
    """tau = 1: every butterfly adds equal points; coeffs = [G, O, ..., O] and h_g1 is all infinity."""
    c = get_curve(name)
    p = sso.Phase1Parameters.new_full(name, 5, 4)
    fn = str(tmp_path / "challenge")
    sso.new_challenge(fn, fn + ".hash", p)
    acc = open(fn, "rb").read()
    m = 16
    out = R.Groth16Params.from_bytes(c, p2.prepare_phase2_buf(p, acc, m), m)
    assert c.g1.eq(out.coeffs_g1[0], c.g1.gen) and all(P is None for P in out.coeffs_g1[1:])
    assert c.g2.eq(out.coeffs_g2[0], c.g2.gen) and all(P is None for P in out.coeffs_g2[1:])
    assert all(P is None for P in out.h_g1)


def _random_points(name, group, n, seed):
    c = get_curve(name)
    G = (c.g1, c.g2)[group]
    s = random.Random(seed).randrange(2, c.Fr.p)
    d_in = _dev(ser.point_to_bytes(G, G.gen, False) * n)
    d_out = torch.empty_like(d_in)
    sso.batch_exp(name, group, d_in, n, 0, s, None, d_out, out_compressed=False)
    return d_out


@pytest.mark.parametrize("name,group", [("bls12_377", 0), ("bls12_377", 1), ("mnt4_753", 1)])
@pytest.mark.parametrize("compressed", [False, True])
def test_group_fft_round_trip(name, group, compressed):
    c = get_curve(name)
    G = (c.g1, c.g2)[group]
    lg, n = 12, 1 << 12
    x = _random_points(name, group, n, 3)
    if compressed:
        xc = torch.empty(n * G.F.nbytes, dtype=torch.uint8, device="cuda")
        sso.reencode(name, group, x, n, xc, in_compressed=False, out_compressed=True)
        x = xc
    y = torch.empty(n * 2 * G.F.nbytes, dtype=torch.uint8, device="cuda")
    back = torch.empty_like(x)
    p2.group_fft(name, group, x, lg, y, inverse=True, in_compressed=compressed)
    p2.group_fft(name, group, y, lg, back, inverse=False, out_compressed=compressed)
    assert torch.equal(back, x)


@pytest.mark.parametrize("name,group", [("bls12_377", 0), ("bw6_761", 1), ("mnt4_753", 1), ("mnt6_753", 1)])
def test_group_fft_edge_inputs(name, group):
    """Infinity, repeated and opposite points: the butterflies double and cancel."""
    c = get_curve(name)
    G = (c.g1, c.g2)[group]
    lg, n = 6, 64
    pts = ser.points_from_bytes(G, _random_points(name, group, n, 5).cpu().numpy().tobytes(), False)
    pts[0] = pts[32] = None
    pts[1] = pts[33]
    pts[2] = G.neg(pts[34])
    pts[3] = pts[35] = pts[4]
    pts[40] = None
    d_x = _dev(ser.points_to_bytes(G, pts, False))
    d_y = torch.empty_like(d_x)
    for inverse in (False, True):
        p2.group_fft(name, group, d_x, lg, d_y, inverse=inverse)
        got = d_y.cpu().numpy().tobytes()
        want = R.group_ifft(c, group, pts) if inverse else R.group_fft(c, group, pts, R.domain_generator(c, n))
        assert got == ser.points_to_bytes(G, want, False), inverse
    # d_out may be d_in
    p2.group_fft(name, group, d_x, lg, d_x, inverse=True)
    assert d_x.cpu().numpy().tobytes() == ser.points_to_bytes(G, R.group_ifft(c, group, pts), False)


@pytest.mark.parametrize("name,power", [("bls12_377", 16), ("mnt4_753", 14)])
def test_prepare_at_size(name, power):
    c = get_curve(name)
    r = c.Fr.p
    s, a, b = _scalars(c, 7)
    m = 1 << power
    acc = _device_accumulator(name, power, s, a, b)
    p = sso.Phase1Parameters.new_full(name, power, 4)
    out = p2.prepare_phase2_buf(p, acc, m)
    s1, s2 = ser.point_size(c.g1, False), ser.point_size(c.g2, False)
    o_c1 = 2 * s1 + s2
    o_c2 = o_c1 + m * s1
    o_a = o_c2 + m * s2
    o_b = o_a + m * s1
    o_h = o_b + m * s1
    assert len(out) == o_h + (m - 1) * s1
    w = R.domain_generator(c, m)
    sm1 = (pow(s, m, r) - 1) % r
    for i in random.Random(2).sample(range(m - 1), 6) + [0, m - 2]:
        wi = pow(w, i, r)
        li = wi * sm1 * pow(m * (s - wi), -1, r) % r
        at = lambda off, sz, k: out[off + k * sz:off + (k + 1) * sz]
        assert at(o_c1, s1, i) == ser.point_to_bytes(c.g1, R.mul(c, 0, c.g1.gen, li), False)
        assert at(o_c2, s2, i) == ser.point_to_bytes(c.g2, R.mul(c, 1, c.g2.gen, li), False)
        assert at(o_a, s1, i) == ser.point_to_bytes(c.g1, R.mul(c, 0, c.g1.gen, a * li), False)
        assert at(o_b, s1, i) == ser.point_to_bytes(c.g1, R.mul(c, 0, c.g1.gen, b * li), False)
        assert at(o_h, s1, i) == ser.point_to_bytes(c.g1, R.mul(c, 0, c.g1.gen, pow(s, i, r) * sm1), False)
    coeffs = out[o_c1:o_c2]
    # sum_i L_i(tau) = 1
    assert p2.points_sum(name, 0, coeffs, m) == ser.point_to_bytes(c.g1, c.g1.gen, False)
    # the forward transform gives back the powers of tau
    d_c = _dev(coeffs)
    d_t = torch.empty_like(d_c)
    p2.group_fft(name, 0, d_c, power, d_t, inverse=False)
    assert d_t.cpu().numpy().tobytes() == acc[64:64 + m * s1]


def test_rejections(tmp_path):
    name = "bls12_377"
    c = get_curve(name)
    s, a, b = _scalars(c, 9)
    acc = R.synthetic_accumulator(c, 3, s, a, b)
    p = sso.Phase1Parameters.new_full(name, 3, 4)

    def code(fn):
        with pytest.raises(sso.SsoError) as e:
            fn()
        return e.value.code
    assert code(lambda: p2.prepare_phase2_buf(p, acc, 16)) == -1               # m > 2^p
    assert code(lambda: p2.prepare_phase2_buf(p, acc, 6)) == -1                # not a power of two
    assert code(lambda: p2.prepare_phase2_buf(p, acc + b"\0", 8)) == -1        # wrong buffer length
    chunked = sso.Phase1Parameters.new_chunk(name, 0, 4, 3, 4)
    assert code(lambda: p2.prepare_phase2_buf(chunked, acc, 8)) == -1
    m6 = sso.Phase1Parameters.new_full("mnt6_753", 16, 4)
    assert code(lambda: p2.prepare_phase2_buf(m6, b"", 1 << 16)) == -1        # beyond the radix-2 domain, checked before the buffer
    # a point of the curve outside the prime-order subgroup in the tauG2 prefix
    G2 = c.g2
    rnd = random.Random(4)
    while True:
        P = G2.point_from_x(tuple(rnd.randrange(G2.F.p) for _ in range(G2.F.deg)), True)
        if P is not None and not G2.in_subgroup(P):
            break
    s1, s2 = ser.point_size(c.g1, False), ser.point_size(c.g2, False)
    off = 64 + 15 * s1 + 1 * s2
    bad = acc[:off] + ser.point_to_bytes(G2, P, False) + acc[off + s2:]
    assert code(lambda: p2.prepare_phase2_buf(p, bad, 4)) == -3
    # files: an existing output and a rejected input leave nothing behind
    fin, fout = str(tmp_path / "response"), str(tmp_path / "phase2")
    open(fin, "wb").write(bad)
    assert code(lambda: p2.prepare_phase2(fout, fin, 4, p)) == -3
    assert not os.path.exists(fout) and not os.path.exists(fout + ".sso-partial")
    assert code(lambda: p2.prepare_phase2(fout, fin, 6, p)) == -1
    assert not os.path.exists(fout)
    open(fout, "wb").write(b"x")
    open(fin, "wb").write(acc)
    assert code(lambda: p2.prepare_phase2(fout, fin, 4, p)) == -5
    assert open(fout, "rb").read() == b"x" and not os.path.exists(fout + ".sso-partial")


@pytest.mark.parametrize("name", ["bls12_377", "mnt6_753"])
def test_file_call(tmp_path, name):
    c = get_curve(name)
    s, a, b = _scalars(c, 11)
    acc = R.synthetic_accumulator(c, 4, s, a, b)
    p = sso.Phase1Parameters.new_full(name, 4, 4)
    fin, fout = str(tmp_path / "response"), str(tmp_path / "phase2")
    open(fin, "wb").write(acc)
    p2.prepare_phase2(fout, fin, 8, p)                                          # (phase2_filename, response_filename, phase2_size, parameters)
    assert open(fout, "rb").read() == p2.prepare_phase2_buf(p, acc, 8) == R.closed_form(c, 8, s, a, b)


def test_reference_file():
    """Consumes the file the Rust reference writes (tests/golden/PREPARE_PHASE2_RECIPE.md) when present."""
    acc_fn = os.path.join(REF_DIR, "p2prep_bls12_377_p5.accumulator.bin")
    out_fn = os.path.join(REF_DIR, "p2prep_bls12_377_p5_m16.phase2.bin")
    if not (os.path.exists(acc_fn) and os.path.exists(out_fn)):
        pytest.skip("reference prepare_phase2 output not generated yet (tests/golden/PREPARE_PHASE2_RECIPE.md)")
    p = sso.Phase1Parameters.new_full("bls12_377", 5, 4)
    assert p2.prepare_phase2_buf(p, open(acc_fn, "rb").read(), 16) == open(out_fn, "rb").read()
