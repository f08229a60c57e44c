"""The group FFT in parts on the GPU (sso_group_fft_parts_buf, sso_p2_prepare_devices_buf / _file) against the transform in one
piece (sso_group_fft_dev, sso_p2_prepare_buf / _file) byte for byte, against the Lagrange closed form, past 2^24 points against
sampled closed-form outputs, and its input checks in every part of every vector."""
import os
import random
from concurrent.futures import ThreadPoolExecutor

import pytest

import snark_setup_operator_b200 as sso
from oracle import serialize as ser
from oracle.curves import CURVE_NAMES, get_curve
from snark_setup_operator_b200 import phase2 as p2

import prepare_phase2_ref as R

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _dev(b: bytes):
    return torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()


def _points(name, group, n, seed, edges):
    """n uncompressed points k_j G; with edges: infinity, a repeated point and its negation at indices of different residues mod 2, 4, 8."""
    c = get_curve(name)
    G = (c.g1, c.g2)[group]
    s = random.Random(seed).randrange(2, c.Fr.p)
    d_in = _dev(ser.point_to_bytes(G, G.gen, False) * n)
    d_out = torch.empty_like(d_in)
    sso.batch_exp(name, group, d_in, n, 0, s, None, d_out, out_compressed=False)
    raw = d_out.cpu().numpy().tobytes()
    if not edges or n < 8:
        return raw
    pts = ser.points_from_bytes(G, raw, False)
    pts[0] = pts[n - 1] = None
    pts[n - 3] = pts[1]
    pts[n // 2 + 2] = G.neg(pts[1])
    return ser.points_to_bytes(G, pts, False)


def _fft_dev(name, group, x, log_n, inverse):
    d_x = _dev(x)
    d_y = torch.empty_like(d_x)
    p2.group_fft(name, group, d_x, log_n, d_y, inverse=inverse)
    return d_y.cpu().numpy().tobytes()


@pytest.mark.parametrize("name", CURVE_NAMES)
@pytest.mark.parametrize("group", [0, 1])
def test_group_fft_parts_equals_group_fft_dev(name, group):
    cases = [(lg, 1 << lp) for lg in (0, 1, 3, 7) for lp in range(lg + 1)] + [(12, 1), (12, 4), (12, 64)]
    for log_n in sorted({lg for lg, _ in cases}):
        x = _points(name, group, 1 << log_n, 10 * log_n + group, edges=True)
        for inverse in (False, True):
            want = _fft_dev(name, group, x, log_n, inverse)
            for parts in [p for lg, p in cases if lg == log_n]:
                got = p2.group_fft_parts(name, group, x, log_n, parts, inverse=inverse)
                assert got == want, (log_n, parts, inverse)


def _scalars(c, seed):
    rnd = random.Random(seed)
    return [rnd.randrange(2, c.Fr.p) for _ in range(3)]


@pytest.mark.parametrize("name", CURVE_NAMES)
def test_prepare_devices_equals_prepare_buf(name):
    c = get_curve(name)
    s, a, b = _scalars(c, 21)
    acc = R.synthetic_accumulator(c, 5, s, a, b)
    p = sso.Phase1Parameters.new_full(name, 5, 4)
    for m in (1, 2, 8, 32):
        want = p2.prepare_phase2_buf(p, acc, m)
        assert want == R.closed_form(c, m, s, a, b), m
        for devices in ([0], [0, 0], [0] * 4, [0] * 8):
            assert p2.prepare_phase2_buf(p, acc, m, devices=devices) == want, (m, devices)


@pytest.mark.parametrize("name,power", [("bls12_377", 16), ("mnt4_753", 14)])
def test_prepare_devices_at_size(tmp_path, name, power):
    from test_gpu_prepare_phase2 import _device_accumulator
    c = get_curve(name)
    s, a, b = _scalars(c, 23)
    m = 1 << power
    acc = _device_accumulator(name, power, s, a, b)
    p = sso.Phase1Parameters.new_full(name, power, 4)
    want = p2.prepare_phase2_buf(p, acc, m)
    for devices in ([0], [0, 0], [0] * 8):
        assert p2.prepare_phase2_buf(p, acc, m, devices=devices) == want, devices
    fin = str(tmp_path / "response")
    open(fin, "wb").write(acc)
    p2.prepare_phase2(str(tmp_path / "one"), fin, m, p)
    p2.prepare_phase2(str(tmp_path / "parts"), fin, m, p, devices=[0] * 4)
    assert open(tmp_path / "parts", "rb").read() == open(tmp_path / "one", "rb").read() == want
    assert sorted(os.listdir(tmp_path)) == ["one", "parts", "response"]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_prepare_devices_on_several_gpus():
    name = "bls12_377"
    c = get_curve(name)
    s, a, b = _scalars(c, 25)
    acc = R.synthetic_accumulator(c, 5, s, a, b)
    p = sso.Phase1Parameters.new_full(name, 5, 4)
    want = p2.prepare_phase2_buf(p, acc, 32)
    assert p2.prepare_phase2_buf(p, acc, 32, devices=[0, 1]) == want
    assert p2.prepare_phase2_buf(p, acc, 32, devices=-1) == want
    x = _points(name, 1, 1 << 7, 3, edges=True)
    assert p2.group_fft_parts(name, 1, x, 7, 8, inverse=True, devices=-1) == _fft_dev(name, 1, x, 7, True)


def test_past_2_24():
    """BLS12-377 G1, 2^25 points x_j = tau^j G in two parts: outputs L_i(tau) G, summing to G; the transform in one piece refuses."""
    name, log_n = "bls12_377", 25
    c = get_curve(name)
    r, n = c.Fr.p, 1 << log_n
    sz = ser.point_size(c.g1, False)
    tau = random.Random(27).randrange(2, r)
    d_gen = _dev(ser.point_to_bytes(c.g1, c.g1.gen, False)).repeat(n)
    d_in = torch.empty_like(d_gen)
    sso.batch_exp(name, 0, d_gen, n, 0, tau, None, d_in, out_compressed=False)
    x = d_in.cpu().numpy().tobytes()
    with pytest.raises(sso.SsoError) as e:
        p2.group_fft(name, 0, d_in, log_n, d_gen, inverse=True)
    assert e.value.code == -1
    del d_gen, d_in
    torch.cuda.empty_cache()
    out = p2.group_fft_parts(name, 0, x, log_n, 2, inverse=True)
    del x
    w = R.domain_generator(c, n)
    tn1 = (pow(tau, n, r) - 1) % r
    samples = [0, (1 << 24) - 1, 1 << 24, n - 1] + random.Random(28).sample(range(n), 60)
    for i in samples:
        wi = pow(w, i, r)
        li = wi * tn1 * pow(n * (tau - wi), -1, r) % r
        assert out[i * sz:(i + 1) * sz] == ser.point_to_bytes(c.g1, R.mul(c, 0, c.g1.gen, li), False), i
    # sum_i L_i(tau) = 1: 2^10 partial sums side by side (one thread each), then their sum
    k = 1 << 10
    chunk = n // k
    with ThreadPoolExecutor(64) as ex:
        partial = list(ex.map(lambda j: p2.points_sum(name, 0, out[j * chunk * sz:(j + 1) * chunk * sz], chunk), range(k)))
    assert p2.points_sum(name, 0, b"".join(partial), k) == ser.point_to_bytes(c.g1, c.g1.gen, False)


def _off_subgroup(G, seed):
    rnd = random.Random(seed)
    while True:
        F = G.F
        P = G.point_from_x(F.from_coeffs(tuple(rnd.randrange(F.p) for _ in range(F.deg))) if F.deg > 1 else F.from_int(rnd.randrange(F.p)), True)
        if P is not None and not G.in_subgroup(P):
            return P


def test_rejections(tmp_path):
    """A flipped byte and a point outside the subgroup, in each residue class mod P = 4 of tauG1, in tauG2, alphaTauG1, betaTauG1
    and in the h_g1 tail tauG1[m .. 2m - 1): SSO_E_INPUT, and the file call leaves no output."""
    name, power, m = "bls12_377", 4, 16
    c = get_curve(name)
    s, a, b = _scalars(c, 29)
    acc = R.synthetic_accumulator(c, power, s, a, b)
    p = sso.Phase1Parameters.new_full(name, power, 4)
    s1, s2 = ser.point_size(c.g1, False), ser.point_size(c.g2, False)
    o_t1, o_t2 = 64, 64 + (2 * m - 1) * s1
    o_a, o_b = o_t2 + m * s2, o_t2 + m * s2 + m * s1
    sites = [(o_t1 + (r + 4 * k) * s1, c.g1, s1) for r, k in ((0, 1), (1, 0), (2, 3), (3, 2))]
    sites += [(o_t2 + 5 * s2, c.g2, s2), (o_a + 6 * s1, c.g1, s1), (o_b + 11 * s1, c.g1, s1), (o_t1 + (m + 3) * s1, c.g1, s1)]
    fin, fout = str(tmp_path / "response"), str(tmp_path / "phase2")
    for i, (off, G, sz) in enumerate(sites):
        flipped = acc[:off + 7] + bytes([acc[off + 7] ^ 0x20]) + acc[off + 8:]
        foreign = acc[:off] + ser.point_to_bytes(G, _off_subgroup(G, i), False) + acc[off + sz:]
        for bad in (flipped, foreign):
            with pytest.raises(sso.SsoError) as e:
                p2.prepare_phase2_buf(p, bad, m, devices=[0] * 4)
            assert e.value.code == -3, (i, e.value.message)
        open(fin, "wb").write(foreign)
        with pytest.raises(sso.SsoError) as e:
            p2.prepare_phase2(fout, fin, m, p, devices=[0] * 4)
        assert e.value.code == -3 and sorted(os.listdir(tmp_path)) == ["response"], i
