#!/usr/bin/env python3
"""prepare_phase2 as a cooperative call of a process group (sso_p2_prepare_dist_file, one process per GPU) next to the same transform
in parts driven by one process over the same GPUs (sso_p2_prepare_devices_file), at BLS12-377 m = 2^20 and MNT4-753 m = 2^19, for
N = 1, 2, 4, 8 GPUs where the box has them.

The accumulator (power log2 m) is synthetic, as in tools/gpu_prepare_phase2.py, and written to a temporary directory.  Per N:
  - dist_s     N ranks spawned by torch.multiprocessing, an NCCL group, dist_init_from_torch; after one untimed call at m = 2^10,
               the host clock of each rank from a barrier to the return of the call; the slowest rank is reported
  - devices_s  in the parent process, one untimed call at m = 2^10 on the same devices, then the host clock around the call on
               devices [0, N)
Both outputs are compared byte for byte.  The card name and power limit are read in the same run.
Usage: tools/gpu_prepare_phase2_dist.py [out.json] [--quick]"""
import json
import os
import subprocess
import sys
import tempfile
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

import snark_setup_operator_b200 as sso  # noqa: E402
from snark_setup_operator_b200 import phase2 as p2  # noqa: E402

SIZES = {"bls12_377": 20, "mnt4_753": 19}
WARM = 10


def _rank(rank, world, port, tmp, name, power):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    sso.dist_init_from_torch(rank)
    f = lambda n: os.path.join(tmp, n)
    p2.prepare_phase2(f("warm_dist"), f("acc_warm"), 1 << WARM, sso.Phase1Parameters.new_full(name, WARM, 4), group=True)
    p = sso.Phase1Parameters.new_full(name, power, 4)
    dist.barrier()
    t0 = time.perf_counter()
    p2.prepare_phase2(f("out_dist"), f("acc"), 1 << power, p, group=True)
    t = time.perf_counter() - t0
    with open(f("time_%d" % rank), "w") as fh:
        fh.write(repr(t))
    sso.dist_finalize()
    dist.destroy_process_group()


def main():
    from gpu_prepare_phase2 import accumulator
    import torch.multiprocessing as mp
    out_fn = next((a for a in sys.argv[1:] if not a.startswith("--")), None)
    quick = "--quick" in sys.argv
    ngpu = torch.cuda.device_count()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    card = {"name": torch.cuda.get_device_name(0), "gpu_count": ngpu, "nvidia_smi": smi}
    print(json.dumps(card), flush=True)
    rows = []
    port = 29700
    with tempfile.TemporaryDirectory() as tmp:
        f = lambda n: os.path.join(tmp, n)
        for name, power in SIZES.items():
            if quick:
                power = min(power, 12)
            m = 1 << power
            with open(f("acc_warm"), "wb") as fh:
                fh.write(accumulator(name, WARM))
            with open(f("acc"), "wb") as fh:
                fh.write(accumulator(name, power))
            torch.cuda.empty_cache()
            p = sso.Phase1Parameters.new_full(name, power, 4)
            for n in (1, 2, 4, 8):
                if n > ngpu:
                    break
                devices = list(range(n))
                port += 1
                mp.spawn(_rank, args=(n, port, tmp, name, power), nprocs=n, join=True)
                dist_s = [float(open(f("time_%d" % r)).read()) for r in range(n)]
                p2.prepare_phase2(f("warm_devices"), f("acc_warm"), 1 << WARM, sso.Phase1Parameters.new_full(name, WARM, 4), devices=devices)
                t0 = time.perf_counter()
                p2.prepare_phase2(f("out_devices"), f("acc"), m, p, devices=devices)
                devices_s = time.perf_counter() - t0
                with open(f("out_dist"), "rb") as a, open(f("out_devices"), "rb") as b:
                    same = a.read() == b.read()
                row = {"curve": name, "m": m, "gpus": n, "dist_s": round(max(dist_s), 3), "dist_s_per_rank": [round(t, 3) for t in dist_s],
                       "devices_s": round(devices_s, 3), "dist_over_devices": round(max(dist_s) / devices_s, 3), "same_bytes": same}
                print(json.dumps(row), flush=True)
                rows.append(row)
                for k in ["warm_dist", "warm_devices", "out_dist", "out_devices"] + ["time_%d" % r for r in range(n)]:
                    os.remove(f(k))
    res = {"tool": "tools/gpu_prepare_phase2_dist.py", "card": card,
           "warmup": "one untimed call of each path at m = 2^10 in the same processes",
           "timing": "host clock: dist from a barrier of the group to the call's return (slowest rank); devices around the call",
           "accumulator": "synthetic (device batch_exp from generator copies), power = log2 m, in a temporary directory",
           "results": rows}
    if out_fn:
        os.makedirs(os.path.dirname(os.path.abspath(out_fn)), exist_ok=True)
        with open(out_fn, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
