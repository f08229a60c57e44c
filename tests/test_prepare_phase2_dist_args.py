"""The argument checks of sso_p2_prepare_dist_file (prepare_phase2 as a cooperative call of a process group), which need neither a
GPU nor a process group: bad arguments, and a call made without a process group, are SSO_E_ARG before any device use, and no
output or partial output is created.  phase2.prepare_phase2(group=True) reaches that export."""
import ctypes
import os

import pytest

from conftest import ROOT

LIB = os.path.join(ROOT, "snark-setup-operator_b200", "libsso_b200.so")
needs_lib = pytest.mark.skipif(not os.path.exists(LIB), reason="libsso_b200.so not built (run __graft_entry__.build())")


def _setup(d):
    import snark_setup_operator_b200 as sso
    from oracle import phase1
    from oracle.params import Phase1Params
    from snark_setup_operator_b200._lib import lib
    open(d / "response", "wb").write(phase1.new_challenge(Phase1Params.new_full("bls12_377", 3, 4)))
    return sso, lib()


@needs_lib
def test_bad_arguments_and_no_process_group(tmp_path):
    sso, L = _setup(tmp_path)
    err = ctypes.create_string_buffer(256)
    full = sso.Phase1Parameters.new_full("bls12_377", 3, 4)
    out, fin = str(tmp_path / "phase2").encode(), str(tmp_path / "response").encode()

    def rc(params, m, parts=0, o=out, i=fin):
        return L.sso_p2_prepare_dist_file(o, i, m, ctypes.byref(params.c_struct()), parts, err, len(err))
    assert rc(full, 4, o=None) == -1 and b"null" in err.value
    assert rc(full, 4, i=None) == -1 and b"null" in err.value
    assert rc(sso.Phase1Parameters.new_chunk("bls12_377", 0, 4, 3, 4), 4) == -1 and b"Full-mode" in err.value
    assert rc(full, 3) == -1 and b"power of two" in err.value
    assert rc(full, 16) == -1                                    # beyond 2^power
    for parts in (3, 6, 8, 1 << 40):                             # not a power of two; more parts than points
        assert rc(full, 4, parts) == -1 and b"parts" in err.value, parts
    big = sso.Phase1Parameters.new_full("bls12_377", 26, 4)
    assert rc(big, 1 << 26, 2) == -1 and b"2^24" in err.value    # parts of 2^25 points
    # valid arguments, no process group
    for parts in (0, 1, 2, 4):
        assert rc(full, 4, parts) == -1 and b"needs a process group" in err.value, parts
    # without a process group even an existing output is not looked at
    open(tmp_path / "phase2", "wb").write(b"keep")
    assert rc(full, 4) == -1 and b"needs a process group" in err.value
    assert open(tmp_path / "phase2", "rb").read() == b"keep"
    os.remove(tmp_path / "phase2")
    assert sorted(os.listdir(tmp_path)) == ["response"]


@needs_lib
def test_python_keyword_reaches_the_export(tmp_path):
    sso, _ = _setup(tmp_path)
    from snark_setup_operator_b200 import phase2 as p2
    full = sso.Phase1Parameters.new_full("bls12_377", 3, 4)
    out, fin = str(tmp_path / "phase2"), str(tmp_path / "response")
    with pytest.raises(sso.SsoError) as e:
        p2.prepare_phase2(out, fin, 4, full, group=True)
    assert e.value.code == -1 and "needs a process group" in e.value.message
    with pytest.raises(sso.SsoError) as e:
        p2.prepare_phase2(out, fin, 4, full, group=True, parts=3)
    assert e.value.code == -1 and "parts" in e.value.message
    with pytest.raises(ValueError):
        p2.prepare_phase2(out, fin, 4, full, group=True, devices=[0])
    with pytest.raises(ValueError):
        p2.prepare_phase2(out, fin, 4, full, parts=2)
    assert sorted(os.listdir(tmp_path)) == ["response"]
