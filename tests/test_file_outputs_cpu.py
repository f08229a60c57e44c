"""Output transaction of the file entry points, checked without a device: every compute entry fails with SSO_E_CUDA at its
first device use, and several file calls have created their outputs (<name>.sso-partial) by then.  A failed call must leave
exactly its inputs behind, and an output that already exists is refused with SSO_E_IO before any device use and left as it
was.  On a GPU these failure points are not reachable this way; tests/test_gpu_flows.py covers the same behaviour there."""
import hashlib
import os

import pytest

from conftest import has_gpu

import snark_setup_operator_b200 as sso
from oracle import phase1, phase2 as o2, synth
from oracle.chacha import ChaChaRng
from oracle.curves import get_curve
from oracle.params import Phase1Params
from snark_setup_operator_b200 import phase2 as p2

pytestmark = pytest.mark.skipif(has_gpu() or not os.path.exists(sso.library_path()),
                                reason="needs the built library and no CUDA device")

NAME, POWER, CS = "bls12_377", 3, 4
SEED = bytes(range(32))


def _p2_challenge(c):
    g1, g2 = c.g1.gen, c.g2.gen
    m = o2.MPCParameters(g1, g2, g2, g2, [g1] * 2, g1, g1, [g1] * 3, [g1] * 3, [g2] * 3, [g1] * 4, [g1] * 2,
                         hashlib.blake2b(b"constraint system", digest_size=64).digest())
    return m.to_bytes(c, False)


def _case(case, d):
    """Writes the inputs of `case` into d and returns (the call, the output file whose existence it checks first)."""
    f = lambda n: str(d / n)
    put = lambda n, b: open(f(n), "wb").write(b)
    full = sso.Phase1Parameters.new_full(NAME, POWER, CS)
    of = Phase1Params.new_full(NAME, POWER, CS)
    if case == "new_challenge":
        p = sso.Phase1Parameters.new_chunk(NAME, 0, CS, POWER, CS)
        return lambda: sso.new_challenge(f("challenge"), f("challenge.hash"), p), "challenge"
    if case in ("contribute_full", "contribute_chunk"):
        if case == "contribute_full":
            p, ch = full, phase1.new_challenge(of)
        else:
            p, ch = sso.Phase1Parameters.new_chunk(NAME, 1, CS, POWER, CS), synth.synthetic_challenge(Phase1Params.new_chunk(NAME, 1, CS, POWER, CS))
        put("challenge", ch)
        return lambda: sso.contribute(f("challenge"), f("challenge.hash"), f("response"), f("response.hash"), sso.CHECK_NONZERO, 0, p, SEED), "response"
    if case == "verify_full":
        ch = phase1.new_challenge(of)
        put("challenge", ch)
        put("response", phase1.contribute(of, ch, ChaChaRng(SEED))[0])
        return (lambda: sso.transform_pok_and_correctness(f("challenge"), f("challenge.hash"), sso.CHECK_NO, f("response"), f("response.hash"),
                                                          sso.CHECK_NONZERO, f("new_challenge"), f("new_challenge.hash"), 0, True, full),
                "new_challenge")
    if case == "combine":
        p0 = sso.Phase1Parameters.new_chunk(NAME, 0, CS, POWER, CS)
        names = []
        for k in range(p0.sizes()["num_chunks"]):
            put("response_%d" % k, bytes(sso.Phase1Parameters.new_chunk(NAME, k, CS, POWER, CS).contribution_size))
            names.append(f("response_%d" % k))
        put("response_list", ("\n".join(names) + "\n").encode())
        return lambda: sso.combine(f("response_list"), f("combined"), p0), "combined"
    c = get_curve(NAME)
    if case == "p2_contribute":
        put("challenge", _p2_challenge(c))
        return lambda: p2.contribute(NAME, f("challenge"), f("challenge.hash"), f("response"), f("response.hash"), sso.CHECK_NO, 0, SEED), "response"
    if case == "p2_verify":
        ch = _p2_challenge(c)
        put("challenge", ch)
        put("response", o2.contribute(c, ch, ChaChaRng(SEED)))
        return (lambda: p2.verify(NAME, f("challenge"), f("challenge.hash"), sso.CHECK_NO, f("response"), f("response.hash"), sso.CHECK_NO,
                                  f("new_challenge"), f("new_challenge.hash"), 0, False),
                "new_challenge")
    assert case == "prepare_phase2"
    put("response", phase1.new_challenge(of))
    return lambda: p2.prepare_phase2(f("phase2"), f("response"), 4, full), "phase2"


CASES = ["new_challenge", "contribute_full", "contribute_chunk", "verify_full", "combine", "p2_contribute", "p2_verify", "prepare_phase2"]


@pytest.mark.parametrize("case", CASES)
def test_failed_call_leaves_only_its_inputs(tmp_path, case):
    call, _ = _case(case, tmp_path)
    inputs = sorted(os.listdir(tmp_path))
    with pytest.raises(sso.SsoError) as e:
        call()
    assert e.value.code == -2, e.value.message
    assert sorted(os.listdir(tmp_path)) == inputs


@pytest.mark.parametrize("case", ["new_challenge", "combine", "p2_contribute", "p2_verify", "prepare_phase2"])
def test_existing_output_is_refused_and_kept(tmp_path, case):
    call, out = _case(case, tmp_path)
    open(tmp_path / out, "wb").write(b"keep")
    before = sorted(os.listdir(tmp_path))
    with pytest.raises(sso.SsoError) as e:
        call()
    assert e.value.code == -5 and "must not exist" in e.value.message, e.value.message
    assert sorted(os.listdir(tmp_path)) == before
    assert open(tmp_path / out, "rb").read() == b"keep"
