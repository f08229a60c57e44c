"""ctypes loader for libsso_b200.so (built in-tree by `make -C snark-setup-operator_b200/csrc`
or `__graft_entry__.build()`).  Import succeeds without the library so that host-only tools
work, but any call raises — the product has no CPU path."""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.environ.get("SSO_B200_LIB") or os.path.join(_HERE, "libsso_b200.so")   # override: kernel A/B experiments
_lib = None


class SsoError(RuntimeError):
    """Non-zero return of an ABI call; mirrors the reference's panic-with-message convention
    (src/bin/contribute.rs:842-856)."""

    def __init__(self, code: int, msg: str):
        super().__init__("sso_b200 error %d: %s" % (code, msg))
        self.code = code
        self.message = msg


class P1Params(ctypes.Structure):
    _fields_ = [("curve", ctypes.c_uint32), ("proving_system", ctypes.c_uint32), ("contribution_mode", ctypes.c_uint32),
                ("power", ctypes.c_uint32), ("chunk_index", ctypes.c_uint64), ("chunk_size", ctypes.c_uint64),
                ("batch_size", ctypes.c_uint64)]


def library_path() -> str:
    return _LIB_PATH


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise SsoError(-2, "libsso_b200.so is not built (%s); run __graft_entry__.build() — there is no CPU fallback" % _LIB_PATH)
        L = ctypes.CDLL(_LIB_PATH)
        L.sso_version.restype = ctypes.c_char_p
        u8p, u32, u64, vp, cp, sz, i32 = (ctypes.c_char_p, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_char_p,
                                          ctypes.c_size_t, ctypes.c_int)
        L.sso_device_count.restype = ctypes.c_int32
        L.sso_device_name.argtypes = [i32, cp, sz]
        L.sso_curve_sizes.argtypes = [u32, ctypes.POINTER(u64)]
        L.sso_p1_sizes.argtypes = [ctypes.POINTER(P1Params), ctypes.POINTER(u64), cp, sz]
        L.sso_blake2b_512.argtypes = [u8p, sz, cp]
        L.sso_batch_exp_dev.argtypes = [u32, u32, vp, u32, u64, u64, u8p, u8p, vp, u32, u32, i32, cp, sz]
        L.sso_batch_mul_dev.argtypes = [u32, u32, vp, u32, u64, u8p, vp, u32, u32, i32, cp, sz]
        L.sso_reencode_dev.argtypes = [u32, u32, vp, u32, u64, vp, u32, u32, u32, i32, cp, sz]
        L.sso_p1_contribute_dev.argtypes = [ctypes.POINTER(P1Params), vp, vp, u8p, u8p, u8p, u32, i32, cp, sz]
        L.sso_p1_contribute_buf.argtypes = [ctypes.POINTER(P1Params), vp, sz, vp, sz, u8p, u8p, u8p, u8p, sz, u32, i32, cp, sz]
        L.sso_power_pairs_dev.argtypes = [u32, u32, vp, u32, u64, u32, u32, u8p, cp, sz, i32, cp, sz]
        L.sso_merge_pairs_dev.argtypes = [u32, u32, vp, vp, u32, u64, u32, u32, u8p, cp, sz, i32, cp, sz]
        L.sso_same_ratio.argtypes = [u32, u8p, u64, ctypes.POINTER(ctypes.c_uint32), i32, cp, sz]
        pp = ctypes.POINTER(P1Params)
        L.sso_p1_keygen.argtypes = [u32, u8p, u8p, cp, sz, cp, sz, i32, cp, sz]
        L.sso_p1_contribute_seeded_buf.argtypes = [pp, vp, sz, vp, sz, u8p, u32, i32, cp, sz]
        L.sso_p1_contribute_file.argtypes = [pp, cp, cp, cp, cp, u32, u32, u8p, i32, cp, sz]
        L.sso_p1_verify_chunk_buf.argtypes = [pp, vp, sz, vp, sz, vp, sz, u32, u32, u32, u32, u8p, i32, cp, sz]
        L.sso_p1_verify_chunk_file.argtypes = [pp, cp, cp, u32, cp, cp, u32, cp, cp, u32, u32, i32, cp, sz]
        L.sso_points_sum.argtypes = [u32, u32, u8p, u64, cp, sz, i32, cp, sz]
        L.sso_p2_scale_queries_buf.argtypes = [u32, vp, sz, vp, sz, u64, u8p, u32, u32, u32, i32, cp, sz]
        L.sso_p2_verify_queries_buf.argtypes = [u32, u8p, sz, u8p, sz, u64, u32, u32, u8p, u8p, u32, u32, u8p, i32, cp, sz]
        L.sso_p1_new_challenge_dev.argtypes = [ctypes.POINTER(P1Params), vp, i32, cp, sz]
        L.sso_p1_contribute_many_buf.argtypes = [pp, sz, ctypes.POINTER(vp), ctypes.POINTER(sz), ctypes.POINTER(vp), ctypes.POINTER(sz),
                                                 u8p, u8p, u8p, u8p, sz, u32, u32, i32, cp, sz]
        L.sso_p1_contribute_seeded_many_buf.argtypes = [pp, sz, ctypes.POINTER(vp), ctypes.POINTER(sz), ctypes.POINTER(vp), ctypes.POINTER(sz),
                                                        u8p, u32, u32, i32, cp, sz]
        L.sso_p1_verify_chunk_many_buf.argtypes = [pp, sz, ctypes.POINTER(vp), ctypes.POINTER(sz), ctypes.POINTER(vp), ctypes.POINTER(sz),
                                                   ctypes.POINTER(vp), ctypes.POINTER(sz), u32, u32, u32, u32, u8p, u32, i32, cp, sz]
        ip = ctypes.POINTER(ctypes.c_int)
        L.sso_p1_new_challenge_file.argtypes = [cp, cp, pp, i32, cp, sz]
        L.sso_p1_set_generators.argtypes = [u32, u8p, sz, u8p, sz, i32, cp, sz]
        L.sso_p1_combine_file.argtypes = [cp, cp, pp, ip, i32, i32, cp, sz]
        L.sso_p1_verify_ratios_file.argtypes = [pp, cp, u32, ip, i32, i32, u8p, cp, sz]
        L.sso_dist_unique_id.argtypes = [cp, cp, sz]
        L.sso_dist_init.argtypes = [ctypes.c_int32, ctypes.c_int32, u8p, i32, cp, sz]
        L.sso_dist_barrier.argtypes = [cp, sz]
        L.sso_dist_stats.argtypes = [ctypes.POINTER(u64)]
        szp = ctypes.POINTER(sz)
        L.sso_p2_contribute_buf.argtypes = [u32, vp, sz, vp, sz, szp, u8p, u32, i32, cp, sz]
        L.sso_p2_contribute_file.argtypes = [u32, cp, cp, cp, cp, u32, u32, u8p, i32, cp, sz]
        L.sso_p2_verify_buf.argtypes = [u32, vp, sz, vp, sz, vp, sz, szp, u32, u32, u32, u8p, i32, cp, sz]
        L.sso_p2_verify_file.argtypes = [u32, cp, cp, u32, cp, cp, u32, cp, cp, u32, u32, i32, cp, sz]
        L.sso_group_fft_dev.argtypes = [u32, u32, vp, u32, u32, u32, vp, u32, i32, cp, sz]
        L.sso_p2_prepare_buf.argtypes = [pp, vp, sz, u64, vp, sz, szp, i32, cp, sz]
        L.sso_p2_prepare_file.argtypes = [cp, cp, u64, pp, i32, cp, sz]
        L.sso_group_fft_parts_buf.argtypes = [u32, u32, vp, sz, u32, u32, vp, sz, u64, ip, i32, i32, cp, sz]
        L.sso_p2_prepare_devices_buf.argtypes = [pp, vp, sz, u64, vp, sz, szp, ip, i32, i32, cp, sz]
        L.sso_p2_prepare_devices_file.argtypes = [cp, cp, u64, pp, ip, i32, i32, cp, sz]
        L.sso_p2_prepare_dist_file.argtypes = [cp, cp, u64, pp, u64, cp, sz]
        L.sso_profile_enable.argtypes = [ctypes.c_int32]
        L.sso_profile_read.argtypes = [ctypes.POINTER(u64), sz]
        L.sso_imad_peak.argtypes = [i32, i32, ctypes.POINTER(ctypes.c_double), cp, sz]
        L.sso_test_field_mul.argtypes = [u32, u8p, u8p, cp, u64, i32, cp, sz]
        L.sso_test_field_op.argtypes = [u32, vp, vp, vp, vp, vp, vp, u64, i32, cp, sz]
        for name in ("sso_device_name", "sso_curve_sizes", "sso_p1_sizes", "sso_blake2b_512", "sso_batch_exp_dev",
                     "sso_batch_mul_dev", "sso_reencode_dev", "sso_p1_contribute_dev", "sso_p1_contribute_buf", "sso_imad_peak",
                     "sso_test_field_mul", "sso_test_field_op", "sso_p1_new_challenge_dev", "sso_profile_enable", "sso_profile_reset",
                     "sso_profile_read", "sso_power_pairs_dev", "sso_merge_pairs_dev", "sso_same_ratio", "sso_p1_keygen",
                     "sso_p1_contribute_seeded_buf", "sso_p1_contribute_file", "sso_p1_verify_chunk_buf", "sso_p1_verify_chunk_file", "sso_points_sum",
                     "sso_p2_scale_queries_buf", "sso_p2_verify_queries_buf", "sso_p1_contribute_many_buf", "sso_p1_verify_chunk_many_buf",
                     "sso_p1_new_challenge_file", "sso_p1_set_generators", "sso_p1_combine_file", "sso_p1_verify_ratios_file",
                     "sso_p2_contribute_buf", "sso_p2_contribute_file", "sso_p2_verify_buf", "sso_p2_verify_file",
                     "sso_dist_unique_id", "sso_dist_init", "sso_dist_barrier", "sso_dist_finalize", "sso_dist_stats", "sso_p1_contribute_seeded_many_buf",
                     "sso_group_fft_dev", "sso_p2_prepare_buf", "sso_p2_prepare_file", "sso_group_fft_parts_buf",
                     "sso_p2_prepare_devices_buf", "sso_p2_prepare_devices_file", "sso_p2_prepare_dist_file"):
            getattr(L, name).restype = ctypes.c_int32
        _lib = L
    return _lib


def call(fn_name: str, *args):
    """Invoke an ABI function whose last two parameters are (err, errcap); raise SsoError on non-zero."""
    err = ctypes.create_string_buffer(512)
    rc = getattr(lib(), fn_name)(*args, err, len(err))
    if rc != 0:
        raise SsoError(rc, err.value.decode("utf-8", "replace"))
    return rc
