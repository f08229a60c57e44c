#!/usr/bin/env python3
"""prepare_phase2 in parts (sso_p2_prepare_devices_buf) against the transform in one piece (sso_p2_prepare_buf), at the sizes of
profiles/prepare_phase2_b200.json (BLS12-377 m = 2^20, BW6-761 2^18, MNT4-753 2^19), and past 2^24 (BLS12-377 2^25).

The accumulator (power log2 m) is synthetic, as in tools/gpu_prepare_phase2.py.  Per curve: one untimed warm-up call of each path at
m = 2^10, then host-clock times of the synchronous calls, alternating one piece / parts on devices [0], twice each, then the parts
with two workers on GPU 0 (devices [0, 0]) once, then on every visible GPU (devices = -1; once on a one-GPU box, where it is [0]).
Both paths' outputs are compared byte for byte.  Past 2^24 only the parts on every GPU run (the one-piece path refuses the size);
add --big-bw6 for BW6-761 2^26 (64 GB accumulator and 64 GB output in host memory).
The card name, power limit and GPU count are read in the same run.  Usage: tools/gpu_prepare_phase2_devices.py [out.json] [--quick]"""
import json
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

import snark_setup_operator_b200 as sso  # noqa: E402
from gpu_prepare_phase2 import accumulator  # noqa: E402
from snark_setup_operator_b200 import phase2 as p2  # noqa: E402

SIZES = {"bls12_377": 20, "bw6_761": 18, "mnt4_753": 19}


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    return out, round(time.perf_counter() - t0, 3)


def main():
    out_fn = next((a for a in sys.argv[1:] if not a.startswith("--")), None)
    quick = "--quick" in sys.argv
    reps = 2
    ngpu = torch.cuda.device_count()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    card = {"name": torch.cuda.get_device_name(0), "gpu_count": ngpu, "nvidia_smi": smi}
    print(json.dumps(card), flush=True)
    rows = []
    for name, power in SIZES.items():
        if quick:
            power = min(power, 12)
        m = 1 << power
        warm = min(power, 10)
        wp, wacc = sso.Phase1Parameters.new_full(name, warm, 4), accumulator(name, warm)
        p2.prepare_phase2_buf(wp, wacc, 1 << warm)
        p2.prepare_phase2_buf(wp, wacc, 1 << warm, devices=[0])
        p2.prepare_phase2_buf(wp, wacc, 1 << warm, devices=-1)
        acc = accumulator(name, power)
        p = sso.Phase1Parameters.new_full(name, power, 4)
        one, parts1, same = [], [], True
        for _ in range(reps):
            a, t = timed(lambda: p2.prepare_phase2_buf(p, acc, m))
            one.append(t)
            b, t = timed(lambda: p2.prepare_phase2_buf(p, acc, m, devices=[0]))
            parts1.append(t)
            same = same and a == b
        b, t2 = timed(lambda: p2.prepare_phase2_buf(p, acc, m, devices=[0, 0]))
        same = same and a == b
        allg = []
        for _ in range(reps if ngpu > 1 else 1):
            b, t = timed(lambda: p2.prepare_phase2_buf(p, acc, m, devices=-1))
            allg.append(t)
            same = same and a == b
        row = {"curve": name, "m": m, "one_piece_s": one, "parts_1gpu_s": parts1, "parts_2workers_1gpu_s": t2, "parts_all_gpus_s": allg,
               "gpus": ngpu, "same_bytes": same, "one_over_parts_1gpu": round(min(one) / min(parts1), 3),
               "speedup_all_gpus_over_one_piece": round(min(one) / min(allg), 3)}
        print(json.dumps(row), flush=True)
        rows.append(row)
        del acc, a, b
    big = [("bls12_377", 12 if quick else 25)]
    if "--big-bw6" in sys.argv and ngpu >= 8:
        big.append(("bw6_761", 26))
    for name, power in big:
        m = 1 << power
        acc = accumulator(name, power)
        p = sso.Phase1Parameters.new_full(name, power, 4)
        out, t = timed(lambda: p2.prepare_phase2_buf(p, acc, m, devices=-1))
        row = {"curve": name, "m": m, "parts_all_gpus_s": t, "gpus": ngpu, "output_bytes": len(out)}
        print(json.dumps(row), flush=True)
        rows.append(row)
        del acc, out
    res = {"tool": "tools/gpu_prepare_phase2_devices.py", "card": card,
           "warmup": "one untimed call of each path at m = 2^10", "timing": "host clock around each synchronous call, min over reps taken for ratios",
           "accumulator": "synthetic (device batch_exp from generator copies), power = log2 m", "results": rows}
    if out_fn:
        os.makedirs(os.path.dirname(os.path.abspath(out_fn)), exist_ok=True)
        with open(out_fn, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
