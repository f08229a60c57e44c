"""Host-side mirror of the phase-2 path over the C ABI: the delta update of the Groth16 H / L queries
(`phase2_cli::contribute::<P>`, reference src/bin/contribute.rs:826-839) and its same-ratio check
(`phase2_cli::verify::<P>`, src/bin/contribute.rs:989-1008).  Only the scaling / verification cores are
bound as primitives; `contribute` / `verify` are the reference-shaped calls on the parameter container (csrc/p2.cuh)."""
from __future__ import annotations

import ctypes

from ._lib import call
from .phase1 import CHECK_NO, _dptr, curve_id, curve_sizes, scalar_bytes


def scale_queries(curve, queries, n: int, delta_inv: int, in_compressed=False, out_compressed=False, check=CHECK_NO,
                  device=0, out=None):
    """h_query / l_query (n serialized G1 points: bytes, numpy or a pinned torch tensor) -> the same vector multiplied by
    delta^-1; returns bytes, or fills the writable buffer `out` when given."""
    from .phase1 import _host_ptr
    s = curve_sizes(curve)
    in_ptr, in_len, k1 = _host_ptr(queries)
    out_len = n * (s["g1_c"] if out_compressed else s["g1_u"])
    buf = ctypes.create_string_buffer(out_len) if out is None else None
    out_ptr, out_len2, k2 = (ctypes.addressof(buf), out_len, buf) if out is None else _host_ptr(out)
    call("sso_p2_scale_queries_buf", curve_id(curve), in_ptr, in_len, out_ptr, out_len2, n, scalar_bytes(curve, delta_inv),
         int(in_compressed), int(out_compressed), check, device)
    del k1, k2
    return buf.raw if out is None else out


def verify_queries(curve, before: bytes, after: bytes, n: int, delta_g2_before: bytes, delta_g2_after: bytes,
                   before_compressed=False, after_compressed=False, check=CHECK_NO, subgroup_check=False, rlc_seed32=None, device=0):
    """Raises SsoError(code -4) unless same_ratio(merge_pairs(before, after), (delta_g2_after, delta_g2_before))."""
    call("sso_p2_verify_queries_buf", curve_id(curve), before, len(before), after, len(after), n, int(before_compressed),
         int(after_compressed), delta_g2_before, delta_g2_after, check, int(subgroup_check), rlc_seed32, device)


def points_sum(curve, group: int, points: bytes, n: int, device=0) -> bytes:
    """Sum of n uncompressed points (combining all-gathered per-GPU partial MSM results)."""
    s = curve_sizes(curve)
    out = ctypes.create_string_buffer(s["g1_u"] if group == 0 else s["g2_u"])
    call("sso_points_sum", curve_id(curve), group, points, n, out, len(out), device)
    return out.raw


def contribute_buf(curve, challenge: bytes, seed32: bytes, check_input=CHECK_NO, device=0) -> bytes:
    """phase2_cli::contribute on host buffers: challenge container (uncompressed) -> response (compressed, one more contribution)."""
    from ._lib import SsoError, lib
    need = ctypes.c_size_t(0)
    err = ctypes.create_string_buffer(512)
    rc = lib().sso_p2_contribute_buf(curve_id(curve), challenge, len(challenge), None, 0, ctypes.byref(need), seed32, check_input, device, err, len(err))
    if rc != -1 or need.value == 0:
        raise SsoError(rc, err.value.decode("utf-8", "replace"))
    out = ctypes.create_string_buffer(need.value)
    call("sso_p2_contribute_buf", curve_id(curve), challenge, len(challenge), out, len(out), ctypes.byref(need), seed32, check_input, device)
    return out.raw


def verify_buf(curve, challenge: bytes, response: bytes, check_input=CHECK_NO, check_output=CHECK_NO, subgroup_check_mode=0, rlc_seed32=None,
               device=0) -> bytes:
    """phase2_cli::verify on host buffers -> the new challenge (uncompressed); raises SsoError(code -4) on rejection."""
    from ._lib import SsoError, lib
    need = ctypes.c_size_t(0)
    err = ctypes.create_string_buffer(512)
    rc = lib().sso_p2_verify_buf(curve_id(curve), challenge, len(challenge), response, len(response), None, 0, ctypes.byref(need), check_input,
                                 check_output, subgroup_check_mode, rlc_seed32, device, err, len(err))
    if rc != -1 or need.value == 0:
        raise SsoError(rc, err.value.decode("utf-8", "replace"))
    out = ctypes.create_string_buffer(need.value)
    call("sso_p2_verify_buf", curve_id(curve), challenge, len(challenge), response, len(response), out, len(out), ctypes.byref(need), check_input,
         check_output, subgroup_check_mode, rlc_seed32, device)
    return out.raw


def contribute(curve, challenge_filename, challenge_hash_filename, response_filename, response_hash_filename, check_input, batch_exp_mode,
               seed32: bytes, device=0):
    """phase2_cli::contribute::<P>, argument for argument (reference src/bin/contribute.rs:827-838); P -> curve, rng -> its seed."""
    call("sso_p2_contribute_file", curve_id(curve), challenge_filename.encode(), challenge_hash_filename.encode(), response_filename.encode(),
         response_hash_filename.encode(), check_input, batch_exp_mode, seed32, device)


def verify(curve, challenge_filename, challenge_hash_filename, check_input, response_filename, response_hash_filename, check_output,
           new_challenge_filename, new_challenge_hash_filename, subgroup_check_mode, verify_full, device=0):
    """phase2_cli::verify::<P>, argument for argument (reference src/bin/contribute.rs:990-1007)."""
    call("sso_p2_verify_file", curve_id(curve), challenge_filename.encode(), challenge_hash_filename.encode(), check_input, response_filename.encode(),
         response_hash_filename.encode(), check_output, new_challenge_filename.encode(), new_challenge_hash_filename.encode(), subgroup_check_mode,
         int(verify_full), device)


def group_fft(curve, group: int, d_in, log_n: int, d_out, inverse=False, in_compressed=False, out_compressed=False, device=0):
    """Radix-2 group FFT of 2^log_n points (device buffers: torch uint8 CUDA tensors) over the scalar field's two-adic domain:
    inverse=False gives out_i = sum_j w^(ij) in_j, inverse=True out_i = 2^-log_n sum_j w^(-ij) in_j, natural order."""
    call("sso_group_fft_dev", curve_id(curve), group, _dptr(d_in), int(in_compressed), log_n, int(inverse), _dptr(d_out),
         int(out_compressed), device)


def _devices(devices, device):
    """devices=None: (no list, `device`); -1: every visible device; a list: those devices (an entry may repeat: one more worker)."""
    from .phase1 import _devices_arg
    if devices == -1:
        return None, 0, -1
    arr, n = _devices_arg(list(devices))
    return arr, n, device


def group_fft_parts(curve, group: int, data, log_n: int, parts: int, inverse=False, devices=None, device=0) -> bytes:
    """The transform of group_fft on host bytes (2^log_n uncompressed points) as a four-step FFT in `parts` parts (a power of two,
    2^log_n / parts <= 2^24), spread over `devices` (None: `device`; -1: all visible; a list may repeat a device)."""
    from .phase1 import _host_ptr
    s = curve_sizes(curve)
    ptr, n, keep = _host_ptr(data)
    out = ctypes.create_string_buffer((1 << log_n) * (s["g1_u"] if group == 0 else s["g2_u"]))
    arr, nd, dev = _devices([] if devices is None else devices, device)
    call("sso_group_fft_parts_buf", curve_id(curve), group, ptr, n, log_n, int(inverse), out, len(out), parts, arr, nd, dev)
    del keep
    return out.raw


def prepare_phase2_buf(parameters, accumulator, phase2_size: int, device=0, devices=None) -> bytes:
    """phase2_cli::prepare_phase2 on host buffers: a Full-mode accumulator (uncompressed, `parameters` a Phase1Parameters) ->
    the Lagrange-basis Groth16Params of phase2_size points (alpha_g1 | beta_g1 | beta_g2 | coeffs_g1 | coeffs_g2 |
    alpha_coeffs_g1 | beta_coeffs_g1 | h_g1, uncompressed).  devices=None: the transform in one piece on `device` (at most 2^24
    points); a list of devices (an entry may repeat: one more worker) or -1 (all visible): the transform in parts, the same bytes,
    up to the radix-2 domain of the curve."""
    from ._lib import SsoError, lib
    from .phase1 import _host_ptr
    ptr, n, keep = _host_ptr(accumulator)
    need = ctypes.c_size_t(0)
    err = ctypes.create_string_buffer(512)
    p = parameters.c_struct()
    if devices is None:
        fn, tail = "sso_p2_prepare_buf", (device,)
    else:
        fn, tail = "sso_p2_prepare_devices_buf", _devices(devices, device)
    rc = getattr(lib(), fn)(ctypes.byref(p), ptr, n, phase2_size, None, 0, ctypes.byref(need), *tail, err, len(err))
    if rc != -1 or need.value == 0:
        raise SsoError(rc, err.value.decode("utf-8", "replace"))
    out = ctypes.create_string_buffer(need.value)
    call(fn, ctypes.byref(p), ptr, n, phase2_size, out, len(out), ctypes.byref(need), *tail)
    del keep
    return out.raw


def prepare_phase2(phase2_filename, response_filename, phase2_size: int, parameters, device=0, devices=None, group=False, parts=0):
    """phase2_cli::prepare_phase2, argument for argument (reference src/bin/intermediate_transform.rs:213-226).  devices as for
    prepare_phase2_buf.  group=True: a cooperative call of the process group (dist_init_from_torch): every rank makes the same call on the
    same files and computes its share of the transform in parts on its own GPU; `parts` (a power of two; 0: chosen automatically)
    is the number of parts.  All ranks must map the same files: one host, or a file system whose shared mappings are coherent
    between them."""
    if group:
        if devices is not None:
            raise ValueError("group=True runs on the device of each rank; devices does not apply")
        call("sso_p2_prepare_dist_file", phase2_filename.encode(), response_filename.encode(), phase2_size,
             ctypes.byref(parameters.c_struct()), parts)
        return
    if parts:
        raise ValueError("parts applies to group=True")
    if devices is None:
        call("sso_p2_prepare_file", phase2_filename.encode(), response_filename.encode(), phase2_size, ctypes.byref(parameters.c_struct()),
             device)
        return
    call("sso_p2_prepare_devices_file", phase2_filename.encode(), response_filename.encode(), phase2_size,
         ctypes.byref(parameters.c_struct()), *_devices(devices, device))
