#!/usr/bin/env python3
"""prepare_phase2 at ceremony sizes on one GPU: BLS12-377 m = 2^20, BW6-761 2^18, MNT4-753 2^19, MNT6-753 2^15 (the largest
radix-2 domain of its scalar field).

The accumulator (power log2 m) is synthetic: tau / alpha / beta powers made on the device by sso_batch_exp_dev from generator
copies.  Per curve: one untimed warm-up call at m = 2^10 (module load, pool growth), then
  - call_s        host clock around the synchronous sso_p2_prepare_buf (H2D, input checks, the four FFTs, h_g1, D2H)
  - fft_ms        per vector, the summed CUDA-event times of the kernels of one sso_group_fft_dev (inverse), profiling on
  - twiddle_muls  scalar multiplications of that FFT: m (the m^-1 pass) + (m/2)(log2 m - 1) (stage 0 has only the twiddle 1)
  - imad_fraction twiddle_muls x bench.declared_macs_per_point over fft_ms, as a fraction of the live sso_imad_peak
The card name and power limit are read in the same run.  Usage: tools/gpu_prepare_phase2.py [out.json] [--quick]"""
import json
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
import snark_setup_operator_b200 as sso  # noqa: E402
from oracle import serialize as ser  # noqa: E402
from oracle.curves import get_curve  # noqa: E402
from snark_setup_operator_b200 import phase2 as p2  # noqa: E402

SIZES = {"bls12_377": 20, "bw6_761": 18, "mnt4_753": 19, "mnt6_753": 15}
S, A, B = 0x1234567890ABCDEF1234567, 0x7777777777777777777, 0x3141592653589793238462643


def accumulator(name, power):
    c = get_curve(name)
    n1, n = (1 << (power + 1)) - 1, 1 << power
    parts = [bytes(64)]
    for group, cnt, coeff in ((0, n1, None), (1, n, None), (0, n, A), (0, n, B), (1, 1, B)):
        G = (c.g1, c.g2)[group]
        d_in = torch.frombuffer(bytearray(ser.point_to_bytes(G, G.gen, False)), dtype=torch.uint8).cuda().repeat(cnt)
        d_out = torch.empty_like(d_in)
        if cnt == 1:
            sso.batch_mul(name, group, d_in, 1, coeff, d_out, out_compressed=False)
        else:
            sso.batch_exp(name, group, d_in, cnt, 0, S, coeff, d_out, out_compressed=False)
        parts.append(d_out.cpu().numpy().tobytes())
        del d_in, d_out
    return b"".join(parts)


def fft_kernel_ms(name, group, acc, power):
    """Kernel time of one inverse FFT over the tau prefix of `group`, from the library's per-launch CUDA events."""
    c = get_curve(name)
    s1, s2 = ser.point_size(c.g1, False), ser.point_size(c.g2, False)
    m = 1 << power
    off, sz = (64, s1) if group == 0 else (64 + ((1 << (power + 1)) - 1) * s1, s2)
    d_x = torch.frombuffer(bytearray(acc[off:off + m * sz]), dtype=torch.uint8).cuda()
    d_y = torch.empty_like(d_x)
    sso.profile_reset()
    sso.profile_enable(2)
    p2.group_fft(name, group, d_x, power, d_y, inverse=True)
    sso.profile_enable(False)
    prof = sso.profile_read()
    kinds = ("batch_exp_g1", "batch_exp_g2", "normalize_g1", "normalize_g2", "tau_tables", "other")
    return sum(prof[k]["ms"] for k in kinds), {k: round(prof[k]["ms"], 3) for k in kinds if prof[k]["launches"]}


def main():
    out_fn = next((a for a in sys.argv[1:] if not a.startswith("--")), None)
    quick = "--quick" in sys.argv
    dev = 0
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", str(dev)],
                         capture_output=True, text=True).stdout.strip()
    card = {"name": torch.cuda.get_device_name(dev), "nvidia_smi": smi}
    peak = sso.imad_peak(0, dev)
    rows = []
    for name, power in SIZES.items():
        if quick:
            power = min(power, 12)
        m = 1 << power
        warm = min(power, 10)
        wacc = accumulator(name, warm)
        p2.prepare_phase2_buf(sso.Phase1Parameters.new_full(name, warm, 4), wacc, 1 << warm)
        acc = accumulator(name, power)
        p = sso.Phase1Parameters.new_full(name, power, 4)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = p2.prepare_phase2_buf(p, acc, m)
        call_s = time.perf_counter() - t0
        muls = m + (m // 2) * (power - 1)
        vec = {}
        for group in (0, 1):
            ms, by_kind = fft_kernel_ms(name, group, acc, power)
            macs = muls * bench.declared_macs_per_point(name, group)
            vec["g%d" % (group + 1)] = {"fft_ms": round(ms, 2), "by_kind_ms": by_kind, "twiddle_muls": muls,
                                        "imad_fraction": round(macs / (ms * 1e-3) / peak, 4) if ms > 0 else None}
        row = {"curve": name, "m": m, "call_s": round(call_s, 3), "output_bytes": len(out),
               "fft_vectors": {"coeffs_g1, alpha_coeffs_g1, beta_coeffs_g1 (each)": vec["g1"], "coeffs_g2": vec["g2"]},
               "sum_of_vector_fft_s": round((3 * vec["g1"]["fft_ms"] + vec["g2"]["fft_ms"]) / 1e3, 3)}
        print(json.dumps(row), flush=True)
        rows.append(row)
        del acc, out
    res = {"tool": "tools/gpu_prepare_phase2.py", "card": card, "imad_peak_macs_per_s": peak, "warmup": "one untimed call at m = 2^10",
           "accumulator": "synthetic (device batch_exp from generator copies), power = log2 m", "results": rows}
    print(json.dumps({"card": card, "imad_peak_macs_per_s": peak}))
    if out_fn:
        os.makedirs(os.path.dirname(os.path.abspath(out_fn)), exist_ok=True)
        with open(out_fn, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
