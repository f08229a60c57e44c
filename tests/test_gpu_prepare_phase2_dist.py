"""prepare_phase2 as a cooperative call of a process group (sso_p2_prepare_dist_file): one process per GPU joined by
dist_init_from_torch, every rank making the same call on the same files.  The output equals sso_p2_prepare_buf (and
sso_p2_prepare_devices_file) byte for byte for every number of parts; a rejected element in another rank's share, arguments that
differ between the ranks and an existing output fail the call on every rank and leave no file behind.  World sizes 2 and
4 where the box has the GPUs; a group of one rank runs the same export on a one-GPU box."""
import os

import pytest

import snark_setup_operator_b200 as sso

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

NGPU = torch.cuda.device_count() if torch.cuda.is_available() else 0


def _raises(fn):
    try:
        fn()
    except sso.SsoError as e:
        return e
    raise AssertionError("the call did not fail")


def _rank_main(rank, world, port, tmp):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    import faulthandler
    import random
    import sys
    import torch.distributed as dist
    faulthandler.dump_traceback_later(300, exit=True, file=sys.stderr)       # a hang must not hold the GPUs
    from oracle import serialize as ser
    from oracle.curves import CURVE_NAMES, get_curve
    from snark_setup_operator_b200 import phase2 as p2
    import prepare_phase2_ref as R
    from test_gpu_prepare_phase2 import _device_accumulator
    from test_gpu_prepare_phase2_parts import _off_subgroup
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    sso.dist_init_from_torch(rank)
    f = lambda n: os.path.join(tmp, n)

    def leftovers(*names):
        return [n for n in os.listdir(tmp) for k in names if n in (k, k + ".sso-partial")]

    def scalars(c, seed):
        rnd = random.Random(seed)
        return [rnd.randrange(2, c.Fr.p) for _ in range(3)]

    # every curve at power 5: parts 0 (chosen), 2, 4, 8 and 32 = m (one point a part, several parts and blocks a rank)
    power, m = 5, 32
    for name in CURVE_NAMES:
        c = get_curve(name)
        p = sso.Phase1Parameters.new_full(name, power, 4)
        fin = f("acc_" + name)
        if rank == 0:
            open(fin, "wb").write(R.synthetic_accumulator(c, power, *scalars(c, 31)))
        dist.barrier()
        for parts in (0, 2, 4, 8, 32):
            out = f("p2_%s_%d" % (name, parts))
            before = sso.dist_stats()["all_gathers"]
            p2.prepare_phase2(out, fin, m, p, group=True, parts=parts)
            assert sso.dist_stats()["all_gathers"] == before                   # no data collective
            dist.barrier()
            if rank == 0:
                want = p2.prepare_phase2_buf(p, open(fin, "rb").read(), m, device=rank)
                assert open(out, "rb").read() == want, (name, parts)
                assert not os.path.exists(out + ".sso-partial")

    # BLS12-377 at m = 2^16, parts chosen: the bytes of sso_p2_prepare_devices_file on one GPU
    name, power = "bls12_377", 16
    c = get_curve(name)
    p = sso.Phase1Parameters.new_full(name, power, 4)
    fin = f("acc_big")
    if rank == 0:
        open(fin, "wb").write(_device_accumulator(name, power, *scalars(c, 33)))
    dist.barrier()
    p2.prepare_phase2(f("p2_big"), fin, 1 << power, p, group=True)
    dist.barrier()
    if rank == 0:
        p2.prepare_phase2(f("p2_big_devices"), fin, 1 << power, p, devices=[rank])
        assert open(f("p2_big"), "rb").read() == open(f("p2_big_devices"), "rb").read()
        os.remove(fin)

    # rejections with P = 2: tauG1[5] lies in part 1 (dealt to rank 1 of 2, rank 3 of 4), tauG1[m + 18] in the second h_g1 piece
    # (rank 1); either raises on every rank, rank 0 reports the other rank, and no output remains
    name, power, m = "bls12_377", 5, 32
    c = get_curve(name)
    p = sso.Phase1Parameters.new_full(name, power, 4)
    s1 = ser.point_size(c.g1, False)
    good = R.synthetic_accumulator(c, power, *scalars(c, 35))
    for k, idx in enumerate((5, m + 18)):
        fin, out = f("bad%d" % k), f("p2_bad%d" % k)
        if rank == 0:
            off = 64 + idx * s1
            open(fin, "wb").write(good[:off] + ser.point_to_bytes(c.g1, _off_subgroup(c.g1, k), False) + good[off + s1:])
        dist.barrier()
        e = _raises(lambda: p2.prepare_phase2(out, fin, m, p, group=True, parts=2))
        assert e.code in (-3, -4), e.message
        if rank == 0 and world > 1:
            assert "another rank" in e.message, e.message
        dist.barrier()
        assert leftovers(os.path.basename(out)) == []

    # the ranks disagree on parts: SSO_E_ARG everywhere, nothing created
    fin, out = f("acc_args"), f("p2_args")
    if rank == 0:
        open(fin, "wb").write(good)
    dist.barrier()
    if world > 1:
        e = _raises(lambda: p2.prepare_phase2(out, fin, m, p, group=True, parts=2 if rank == 0 else 4))
        assert e.code == -1 and "parts" in e.message, e.message
        dist.barrier()
        assert leftovers(os.path.basename(out)) == []

    # an existing output: SSO_E_IO on every rank, the file untouched
    if rank == 0:
        open(out, "wb").write(b"keep")
    dist.barrier()
    e = _raises(lambda: p2.prepare_phase2(out, fin, m, p, group=True))
    assert e.code == -5 and "must not exist" in e.message, e.message
    dist.barrier()
    assert open(out, "rb").read() == b"keep" and not os.path.exists(out + ".sso-partial")

    sso.dist_finalize()
    dist.destroy_process_group()
    faulthandler.cancel_dump_traceback_later()


@pytest.mark.parametrize("world", [1, 2, 4])
def test_prepare_phase2_one_process_per_gpu(tmp_path, world):
    if world > NGPU:
        pytest.skip("needs %d GPUs" % world)
    import torch.multiprocessing as mp
    mp.spawn(_rank_main, args=(world, 29647 + world, str(tmp_path)), nprocs=world, join=True)
