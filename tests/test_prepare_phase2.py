"""prepare_phase2 without a GPU: the restated transform (tests/prepare_phase2_ref.py) against the Lagrange closed form, the
radix-2 domain constants of csrc/constants.cuh against their definition, and the new C ABI entries' refusal to run without a
device (no CPU fallback)."""
import ctypes
import os
import random
import re

import pytest

from conftest import ROOT, has_gpu
from oracle import cport, serialize as ser
from oracle.curves import CURVE_NAMES, get_curve

import prepare_phase2_ref as R

CONSTANTS = os.path.join(ROOT, "snark-setup-operator_b200", "csrc", "constants.cuh")
LIB = os.path.join(ROOT, "snark-setup-operator_b200", "libsso_b200.so")


def _powers(c, group, s, m):
    G = (c.g1, c.g2)[group]
    out = cport.batch_exp(c, group, ser.point_to_bytes(G, G.gen, False) * m, m, 0, s, None, out_compressed=False)
    return ser.points_from_bytes(G, out, False)


@pytest.mark.parametrize("name", CURVE_NAMES)
@pytest.mark.parametrize("group", [0, 1])
@pytest.mark.parametrize("m", [1, 2, 4, 16])
def test_oracle_ifft_is_lagrange_basis(name, group, m):
    c = get_curve(name)
    G = (c.g1, c.g2)[group]
    s = random.Random(m * 10 + group).randrange(2, c.Fr.p)
    x = _powers(c, group, s, m)
    y = R.group_ifft(c, group, x)
    want = [R.mul(c, group, G.gen, k) for k in R.lagrange_at(c, s, m)]
    assert all(G.eq(a, b) for a, b in zip(y, want))
    back = R.group_fft(c, group, y, R.domain_generator(c, m))
    assert all(G.eq(a, b) for a, b in zip(back, x))


@pytest.mark.parametrize("name", CURVE_NAMES)
def test_lagrange_basis_at_a_domain_point(name):
    c = get_curve(name)
    w = R.domain_generator(c, 8)
    assert R.lagrange_at(c, 1, 8) == [1] + [0] * 7
    assert R.lagrange_at(c, pow(w, 3, c.Fr.p), 8) == [0, 0, 0, 1, 0, 0, 0, 0]


def _cuh_words(text, name):
    m = re.search(r"static const uint32_t %s\[(\d+)\] = \{([^}]*)\};" % name, text)
    return sum(int(w.strip().rstrip("u"), 16) << (32 * i) for i, w in enumerate(m.group(2).split(",")))


@pytest.mark.parametrize("name", CURVE_NAMES)
def test_generated_domain_constants(name):
    c = get_curve(name)
    r = c.Fr.p
    text = open(CONSTANTS).read()
    s = R.two_adicity(c)
    assert s == {"bls12_377": 47, "bw6_761": 46, "mnt4_753": 30, "mnt6_753": 15}[name]
    blk = re.search(r"struct FFT_%s \{\n  static constexpr int GENERATOR = (\d+); static constexpr int TWO_ADICITY = (\d+);" % name, text)
    assert (int(blk.group(1)), int(blk.group(2))) == (R.FR_GENERATOR[name], s)
    root, root_inv = _cuh_words(text, "h_%s_fr_root" % name), _cuh_words(text, "h_%s_fr_root_inv" % name)
    assert root == R.domain_generator(c, 1 << s) and root * root_inv % r == 1
    # w_m = root^(2^(s - log m)) is the domain generator and has order exactly m, for every m up to 2^s
    w = root
    for lg in range(s, -1, -1):
        m = 1 << lg
        assert w == R.domain_generator(c, m)
        assert pow(w, m, r) == 1 and (m == 1 or pow(w, m // 2, r) == r - 1)
        w = w * w % r


@pytest.mark.skipif(not os.path.exists(LIB), reason="libsso_b200.so not built (run __graft_entry__.build())")
@pytest.mark.skipif(has_gpu(), reason="only meaningful without a GPU")
def test_new_exports_have_no_cpu_fallback():
    import snark_setup_operator_b200 as sso
    from snark_setup_operator_b200._lib import lib
    L = lib()
    err = ctypes.create_string_buffer(256)
    buf = ctypes.create_string_buffer(64)
    assert L.sso_group_fft_dev(0, 0, ctypes.addressof(buf), 0, 2, 1, ctypes.addressof(buf), 0, 0, err, len(err)) == -2
    p = sso.Phase1Parameters.new_full("bls12_377", 2, 4)
    acc = bytes(p.accumulator_size)
    n = ctypes.c_size_t(0)
    out = ctypes.create_string_buffer(1 << 16)
    assert L.sso_p2_prepare_buf(ctypes.byref(p.c_struct()), acc, len(acc), 4, out, len(out), ctypes.byref(n), 0, err, len(err)) == -2
    assert b"no CPU fallback" in err.value
    # the size protocol and the argument checks need no device
    assert L.sso_p2_prepare_buf(ctypes.byref(p.c_struct()), acc, len(acc), 4, None, 0, ctypes.byref(n), 0, err, len(err)) == -1
    assert n.value == (2 + 3 * 4 + 3) * 96 + 5 * 192
    assert L.sso_p2_prepare_buf(ctypes.byref(p.c_struct()), acc, len(acc), 3, out, len(out), ctypes.byref(n), 0, err, len(err)) == -1
    assert L.sso_p2_prepare_buf(ctypes.byref(p.c_struct()), acc, len(acc), 8, out, len(out), ctypes.byref(n), 0, err, len(err)) == -1
    assert L.sso_p2_prepare_buf(ctypes.byref(p.c_struct()), acc[:-1], len(acc) - 1, 4, out, len(out), ctypes.byref(n), 0, err, len(err)) == -1
    assert L.sso_p2_prepare_file(b"/nonexistent/out", b"/nonexistent/in", 4, ctypes.byref(p.c_struct()), 0, err, len(err)) == -5
    m6 = sso.Phase1Parameters.new_full("mnt6_753", 16, 4)
    assert L.sso_p2_prepare_buf(ctypes.byref(m6.c_struct()), None, 0, 1 << 16, None, 0, ctypes.byref(n), 0, err, len(err)) == -1
    assert b"2^15" in err.value
