"""The group FFT in parts without a GPU: the four-step decomposition of csrc/p2prep.cuh (parts_fft) restated over Fr and over
curve points against the direct transform, and the argument checks of the exports that run it (sso_group_fft_parts_buf,
sso_p2_prepare_devices_buf / _file), which need no device; past them every call fails with SSO_E_CUDA at its first device use
and a file call leaves only its inputs behind."""
import ctypes
import os
import random

import pytest

from conftest import ROOT, has_gpu
from oracle.curves import CURVE_NAMES, get_curve

import prepare_phase2_ref as R

LIB = os.path.join(ROOT, "snark-setup-operator_b200", "libsso_b200.so")


def _stockham_rows(rows, root_of, add, sub, mul):
    """The P-point FFT over rows of equal length in Stockham stages, as parts_block runs it: stage s (Ns = 2^s) multiplies upper row
    P/2 + j by w_2Ns^(j mod Ns) (root_of(2 Ns, e)), then row j's butterfly writes rows o = 2 Ns floor(j / Ns) + (j mod Ns) and o + Ns."""
    P = len(rows)
    s = 0
    while (1 << s) < P:
        ns = 1 << s
        x = [list(r) for r in rows]
        for j in range(P // 2):
            if j % ns:
                x[P // 2 + j] = [mul(v, root_of(2 * ns, j % ns)) for v in x[P // 2 + j]]
        out = [None] * P
        for j in range(P // 2):
            o = (j // ns) * 2 * ns + j % ns
            out[o] = [add(a, t) for a, t in zip(x[j], x[P // 2 + j])]
            out[o + ns] = [sub(a, t) for a, t in zip(x[j], x[P // 2 + j])]
        rows = out
        s += 1
    return rows


def _parts(x, P, w, r, scale, dft, add, sub, mul):
    """X = the size-m DFT of x with root w, times scale, in P parts: part FFT of x[j::P], part twiddle scale w^(j c), rows FFT."""
    m = len(x)
    M = m // P
    rows = []
    for j in range(P):
        y = dft(x[j::P], pow(w, P, r))
        rows.append([mul(v, scale * pow(w, j * c, r) % r) for c, v in enumerate(y)])
    # the row FFT's stage root of order 2 Ns is w^(m / (2 Ns))
    rows = _stockham_rows(rows, lambda order, e: pow(w, m // order * e, r), add, sub, mul)
    return [v for row in rows for v in row]


@pytest.mark.parametrize("name", CURVE_NAMES)
@pytest.mark.parametrize("inverse", [False, True])
def test_four_step_over_fr_equals_the_dft(name, inverse):
    c = get_curve(name)
    r = c.Fr.p
    rnd = random.Random(2 * CURVE_NAMES.index(name) + int(inverse))

    def dft(x, w):
        n = len(x)
        return [sum(v * pow(w, i * k % n, r) for i, v in enumerate(x)) % r for k in range(n)]
    for log_m in range(0, 9):
        m = 1 << log_m
        if m > 1 << R.two_adicity(c):
            continue
        x = [rnd.randrange(r) for _ in range(m)]
        w = R.domain_generator(c, m)
        scale = 1
        if inverse:
            w, scale = pow(w, -1, r), pow(m, -1, r)
        want = [v * scale % r for v in dft(x, w)]
        for log_p in range(0, log_m + 1):
            got = _parts(x, 1 << log_p, w, r, scale, dft, lambda a, b: (a + b) % r, lambda a, b: (a - b) % r, lambda a, k: a * k % r)
            assert got == want, (log_m, log_p)


@pytest.mark.parametrize("log_p", [1, 2, 3])
def test_four_step_over_points_equals_prepare_phase2_ref(log_p):
    name, power, m = "bls12_377", 3, 8
    c = get_curve(name)
    r = c.Fr.p
    s, a, b = (random.Random(log_p).randrange(2, r) for _ in range(3))
    acc = R.synthetic_accumulator(c, power, s, a, b)
    tg1, tg2, ag1, bg1, bg2 = R.read_accumulator(c, power, acc)
    w = pow(R.domain_generator(c, m), -1, r)
    minv = pow(m, -1, r)

    def ifft(group, x):
        G = (c.g1, c.g2)[group]
        return _parts(x, 1 << log_p, w, r, minv, lambda v, om: R.group_fft(c, group, v, om), G.add, lambda p, q: G.add(p, G.neg(q)),
                      lambda p, k: R.mul(c, group, p, k))
    h = [c.g1.add(tg1[i + m], c.g1.neg(tg1[i])) for i in range(m - 1)]
    got = R.Groth16Params(ag1[0], bg1[0], bg2[0], ifft(0, tg1[:m]), ifft(1, tg2[:m]), ifft(0, ag1[:m]), ifft(0, bg1[:m]), h).to_bytes(c)
    assert got == R.prepare_phase2(c, power, acc, m)


def _lib():
    import snark_setup_operator_b200 as sso
    from snark_setup_operator_b200._lib import lib
    return sso, lib()


needs_lib = pytest.mark.skipif(not os.path.exists(LIB), reason="libsso_b200.so not built (run __graft_entry__.build())")
no_gpu = pytest.mark.skipif(has_gpu(), reason="only meaningful without a GPU")


@needs_lib
def test_group_fft_parts_argument_checks():
    sso, L = _lib()
    err = ctypes.create_string_buffer(256)

    def rc(curve, group, log_n, parts, n_in=None, n_out=None, same=False):
        sz = 96 if group == 0 else 192
        nb = (1 << log_n) * sz
        src = ctypes.create_string_buffer(nb if n_in is None else n_in)
        dst = src if same else ctypes.create_string_buffer(nb if n_out is None else n_out)
        return L.sso_group_fft_parts_buf(curve, group, src, len(src), log_n, 1, dst, len(dst), parts, None, 0, 0, err, len(err))
    assert rc(0, 0, 3, 3) == -1                    # not a power of two
    assert rc(0, 0, 3, 0) == -1
    assert rc(0, 0, 3, 16) == -1                   # more parts than points
    assert rc(0, 0, 25, 1, 96, 96) == -1           # a part of 2^25 points
    assert b"2^24" in err.value
    assert rc(0, 0, 48, 1 << 24, 96, 96) == -1     # beyond the 2-adicity of BLS12-377 Fr (47)
    assert rc(0, 2, 3, 2) == -1                    # unknown group
    assert rc(9, 0, 3, 2) == -1                    # unknown curve
    assert rc(0, 0, 3, 2, n_in=8 * 96 - 1) == -1   # buffer lengths
    assert rc(0, 1, 3, 2, n_out=8 * 96) == -1
    assert rc(0, 0, 3, 2, same=True) == -1         # in place
    dev = (ctypes.c_int * 1)(-3)
    src, dst = ctypes.create_string_buffer(8 * 96), ctypes.create_string_buffer(8 * 96)
    if not has_gpu():
        for parts in (1, 2, 8):
            assert rc(0, 0, 3, parts) == -2, err.value
        assert L.sso_group_fft_parts_buf(0, 0, src, len(src), 3, 0, dst, len(dst), 2, None, 0, -1, err, len(err)) == -2
    else:
        assert L.sso_group_fft_parts_buf(0, 0, src, len(src), 3, 0, dst, len(dst), 2, dev, 1, 0, err, len(err)) == -1


@needs_lib
def test_prepare_devices_argument_checks():
    sso, L = _lib()
    err = ctypes.create_string_buffer(256)
    n = ctypes.c_size_t(0)
    p = sso.Phase1Parameters.new_full("bls12_377", 2, 4)
    acc = bytes(p.accumulator_size)
    out = ctypes.create_string_buffer(1 << 16)

    def rc(params, a, m, o=out, cap=None):
        return L.sso_p2_prepare_devices_buf(ctypes.byref(params.c_struct()), a, len(a) if a is not None else 0, m, o, len(o) if cap is None else cap,
                                            ctypes.byref(n), None, 0, 0, err, len(err))
    # the size protocol, as sso_p2_prepare_buf
    assert rc(p, acc, 4, None, 0) == -1 and n.value == (2 + 3 * 4 + 3) * 96 + 5 * 192
    assert rc(p, acc, 3) == -1                      # not a power of two
    assert rc(p, acc, 8) == -1                      # beyond 2^power
    assert rc(p, acc[:-1], 4) == -1                 # accumulator length
    chunked = sso.Phase1Parameters.new_chunk("bls12_377", 0, 4, 2, 4)
    assert rc(chunked, acc, 4) == -1
    m6 = sso.Phase1Parameters.new_full("mnt6_753", 16, 4)
    assert rc(m6, None, 1 << 16, None, 0) == -1 and b"2^15" in err.value
    m4 = sso.Phase1Parameters.new_full("mnt4_753", 31, 4)
    assert rc(m4, None, 1 << 31, None, 0) == -1 and b"2^30" in err.value     # beyond the 2-adicity of MNT4-753 Fr
    # past 2^24 the size passes (the missing accumulator is refused next) where sso_p2_prepare_buf refuses the size
    big = sso.Phase1Parameters.new_full("bls12_377", 25, 4)
    assert rc(big, None, 1 << 25, None, 0) == -1 and b"accumulator is 0 bytes" in err.value
    assert L.sso_p2_prepare_buf(ctypes.byref(big.c_struct()), None, 0, 1 << 25, None, 0, ctypes.byref(n), 0, err, len(err)) == -1
    assert b"beyond the radix-2 domain" in err.value
    if not has_gpu():
        assert rc(p, acc, 4) == -2 and b"no CUDA device" in err.value


def _file_case(d):
    import snark_setup_operator_b200 as sso
    from oracle import phase1
    from oracle.params import Phase1Params
    from snark_setup_operator_b200 import phase2 as p2
    full = sso.Phase1Parameters.new_full("bls12_377", 3, 4)
    open(d / "response", "wb").write(phase1.new_challenge(Phase1Params.new_full("bls12_377", 3, 4)))
    return lambda: p2.prepare_phase2(str(d / "phase2"), str(d / "response"), 4, full, devices=[0, 0])


@needs_lib
@no_gpu
def test_file_call_leaves_only_its_inputs(tmp_path):
    import snark_setup_operator_b200 as sso
    call = _file_case(tmp_path)
    with pytest.raises(sso.SsoError) as e:
        call()
    assert e.value.code == -2, e.value.message
    assert sorted(os.listdir(tmp_path)) == ["response"]


@needs_lib
def test_file_call_refuses_an_existing_output(tmp_path):
    import snark_setup_operator_b200 as sso
    call = _file_case(tmp_path)
    open(tmp_path / "phase2", "wb").write(b"keep")
    with pytest.raises(sso.SsoError) as e:
        call()
    assert e.value.code == -5 and "must not exist" in e.value.message, e.value.message
    assert sorted(os.listdir(tmp_path)) == ["phase2", "response"]
    assert open(tmp_path / "phase2", "rb").read() == b"keep"
