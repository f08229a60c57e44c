"""Field-arithmetic conformance: every fp / ext / coop operation of the device code on raw Montgomery words, against the
big-integer reference (tests/field_cases.py), on two backends — the CPU emulator (tests/emul, always) and the B200 through
sso_test_field_op (gpu marker).  Outputs are checked for value AND representation (every coefficient below p); the branch
predicates of the device code are asserted to be hit on both sides; on the GPU the device words must equal the emulator's, and
the cooperative fields run with neighbouring lane groups of one warp taking different operations."""
import ctypes
import os
import subprocess
import tempfile

import pytest

import field_cases as fc
from conftest import ROOT

EMUL_DIR = os.path.join(ROOT, "tests", "emul")
CSRC = os.path.join(ROOT, "snark-setup-operator_b200", "csrc")
BACKENDS = ["emul", pytest.param("gpu", marks=pytest.mark.gpu)]
u32p = ctypes.POINTER(ctypes.c_uint32)


def _build_emul(name, defines=()):
    """the emulator library, rebuilt when a device source is newer; beside the sources when that directory is writable, else in a
    temporary directory"""
    srcs = [os.path.join(EMUL_DIR, "emul.cpp")] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    so = os.path.join(EMUL_DIR, name)
    if not os.access(EMUL_DIR, os.W_OK):
        so = os.path.join(tempfile.mkdtemp(prefix="sso_emul_"), name)
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-pthread", *defines, "-o", so,
                               os.path.join(EMUL_DIR, "emul.cpp")])
    lib = ctypes.CDLL(so)
    lib.emul_field_op_raw.argtypes = [ctypes.c_uint32, u32p, u32p, u32p, u32p, u32p, u32p, ctypes.c_uint64]
    return lib


@pytest.fixture(scope="module")
def emul():
    return _build_emul("libsso_emul.so")


def _arr(words):
    return (ctypes.c_uint32 * max(1, len(words)))(*words)


def run_emul(lib, fid, cs):
    fd = fc.field(fid)
    ops, a, b, k = fc.pack(fd, cs)
    out = (ctypes.c_uint32 * max(1, len(cs) * fd.words))()
    rc = (ctypes.c_uint32 * max(1, len(cs)))()
    assert lib.emul_field_op_raw(fid, _arr(ops), _arr(a), _arr(b), _arr(k), out, rc, len(cs)) == 0
    return fc.unpack(fd, out, len(cs)), list(rc)[:len(cs)]


def run_gpu(fid, cs):
    import numpy as np
    import snark_setup_operator_b200 as sso
    fd = fc.field(fid)
    ops, a, b, k = (np.asarray(x, dtype=np.uint32) for x in fc.pack(fd, cs))
    out = np.zeros(len(cs) * fd.words, dtype=np.uint32)
    rc = np.zeros(len(cs), dtype=np.uint32)
    ptr = lambda x: x.ctypes.data_as(ctypes.c_void_p)
    sso._lib.call("sso_test_field_op", fid, ptr(ops), ptr(a), ptr(b), ptr(k), ptr(out), ptr(rc), len(cs), 0)
    return fc.unpack(fd, out.tolist(), len(cs)), rc.tolist()


def run(backend, request, fid, cs):
    if backend == "emul":
        return run_emul(request.getfixturevalue("emul"), fid, cs)
    return run_gpu(fid, cs)


def assert_conform(fid, cs, outs, rcs):
    fd = fc.field(fid)
    bad = []
    for c, o, r in zip(cs, outs, rcs):
        why = fc.check(fd, c, o, r)
        if why:
            bad.append("%s [%s] a=%s b=%s k=%d: %s" % (c.op, c.tag, [hex(x) for x in c.a], [hex(x) for x in c.b], c.k, why))
    assert not bad, "field %d: %d of %d cases wrong, first: %s" % (fid, len(bad), len(cs), "\n".join(bad[:5]))


def assert_branches(fid, cs):
    fd = fc.field(fid)
    hit = fc.predicates(fd, cs)
    for name, sides in fc.required_sides(fd).items():
        missing = sides - set(hit.get(name, {}))
        assert not missing, (fid, name, sorted(missing))


@pytest.mark.parametrize("fid", sorted(fc.FIELDS))
@pytest.mark.parametrize("backend", BACKENDS)
def test_every_supported_op(backend, request, fid):
    """every supported (field, op) pair on edge, random, constructed and unreduced operands: value and canonical representation;
    every other pair answers 'unsupported' instead of being skipped"""
    cs = fc.cases(fid, "gpu" if backend == "gpu" else "emul")
    assert {c.op for c in cs} == fc.SUPPORTED[fid]
    assert_branches(fid, cs)
    outs, rcs = run(backend, request, fid, cs)
    assert_conform(fid, cs, outs, rcs)
    un = fc.unsupported_cases(fid)
    if un:
        _, rcs = run(backend, request, fid, un)
        assert rcs == [fc.RC_UNSUPPORTED] * len(un), [c.op for c, r in zip(un, rcs) if r != fc.RC_UNSUPPORTED]


@pytest.mark.parametrize("fid", sorted(fc.FIELDS))
def test_cases_reach_every_branch(fid):
    """the case lists reach both sides of every data-dependent conditional of the device code (restated in field_cases.py):
    final subtractions of add / mul / dedicated squaring including s = p and u = p, the borrow of sub including a = b, neg of zero,
    the quotient estimate of reduce_small, both exits of the binary inversion, every first Tonelli-Shanks depth up to the
    2-adicity, the five branches of Fp2::sqrt"""
    assert_branches(fid, fc.cases(fid, "emul"))


def test_fq3_square_root_through_the_norm_equals_plain(emul):
    """DESIGN.md §4: Fp3::sqrt_ts_norm forms the same w = a^((t-1)/2) as the plain Tonelli-Shanks in Fq3, hence the same root, bit
    for bit (a build with -DSSO_FQ3_SQRT_PLAIN selects the plain one)"""
    plain = _build_emul("libsso_emul_fq3plain.so", ["-DSSO_FQ3_SQRT_PLAIN"])
    cs = [c for c in fc.cases(7) if c.op == "sqrt"]
    assert len(cs) >= 20
    o1, r1 = run_emul(emul, 7, cs)
    o2, r2 = run_emul(plain, 7, cs)
    assert r1 == r2 and sum(r1) >= 10
    assert o1 == o2
    assert_conform(7, cs, o2, r2)


@pytest.mark.gpu
@pytest.mark.parametrize("fid", sorted(fc.FIELDS))
def test_gpu_words_equal_emulator_words(emul, fid):
    """the hardware carry chains against the emulated carry model: every case is deterministic (the square roots too), so the
    device and the emulator must return the same words, not only the same values"""
    cs = fc.cases(fid, "emul")
    og, rg = run_gpu(fid, cs)
    oe, re_ = run_emul(emul, fid, cs)
    diff = [i for i in range(len(cs)) if og[i] != oe[i] or rg[i] != re_[i]]
    assert not diff, "field %d: %d cases differ, first %s" % (fid, len(diff), cs[diff[0]])


@pytest.mark.gpu
@pytest.mark.parametrize("fid", sorted(fc.COOP))
@pytest.mark.parametrize("n", [1, 63, 331, 1000])
def test_cooperative_groups_of_one_warp_diverge(fid, n):
    """coop.cuh exchanges with group-masked shuffles, claiming that the lane groups of one warp may run different code: here
    neighbouring groups take different ops — inversions of very different loop lengths (1, p - 1, 2^k, random), squarings,
    products, sums, negations — and n is ragged, so the last warp and the last block are partly empty.  Every element must match
    the reference and equal, word for word, the one-thread-per-element field on the same input."""
    import random
    fd = fc.field(fid)
    p, R = fd.p, fd.R
    rnd = random.Random(n * 11 + fid)
    inv_in = [(R % p,) + (0,) * (fd.deg - 1), ((p - 1),) * fd.deg, (1 << rnd.randrange(1, 32),) + (0,) * (fd.deg - 1)]
    cycle = ["inv", "sqr", "mul", "add", "inv", "neg", "sub", "inv", "mul"]
    cs = []
    for i in range(n):
        op = cycle[(i * 7 + i // 5) % len(cycle)]
        a = inv_in[i % 3] if op == "inv" and i % 4 else fc.relem(fd, rnd)
        cs.append(fc.Case(op, a, fc.relem(fd, rnd), tag="divergent"))
    oc, rc = run_gpu(fid, cs)
    assert_conform(fid, cs, oc, rc)
    op_, rp = run_gpu(fc.COOP[fid], cs)
    assert oc == op_ and rc == rp
