"""CPU tests of the deterministic mode (the same seed and inputs give bit-identical outputs): the C ABI that carries it,
the switch and the plan keys that hold it, and the rank-ordered GroupNorm reduction of NCCL-mode frame sharding under a
2-rank gloo group."""
import ctypes
import os
import re

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from hi3d_official_b200 import _native, ops
from hi3d_official_b200 import dist as D
from hi3d_official_b200.unet import VideoUNet

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_deterministic_entry_points_are_declared_and_exported():
    """The deterministic mode adds entry points only: hi3d_gemm_params and the ABI version stay as they were."""
    lib = _native.load()
    hdr = open(os.path.join(ROOT, "include", "hi3d_b200.h")).read()
    new = ("hi3d_gemm_det", "hi3d_gemm_tc5_det", "hi3d_groupnorm_silu_det", "hi3d_groupnorm_sums_det",
           "hi3d_groupnorm_group_sums_det", "hi3d_groupnorm_unit_stats_det", "hi3d_groupnorm_partials_floats",
           "hi3d_groupnorm_fold")
    for name in new:
        assert re.search(r"\b" + name + r"\s*\(", hdr) and name in _native.EXPORTS and hasattr(lib, name)
    assert lib.hi3d_abi_version() == 2
    assert re.search(r"int32_t gn_rows;\s*\} hi3d_gemm_params;", hdr)
    assert ctypes.sizeof(_native.GemmParams) == _native.GemmParams.gn_rows.offset + 4


def test_partials_floats_covers_both_producers():
    f = _native.load().hi3d_groupnorm_partials_floats
    # stage-2 level 0: 32 images of 128 x 128, C = 320, unit 10 -> the epilogue slots dominate (512 blocks x 40 octets x 4)
    assert f(32, 128 * 128, 320, 10) == 32 * 512 * 40 * 4
    # the up-conv table covers the four parity classes: output rows per image
    assert f(32, 4 * 64 * 64, 320, 10) == f(32, 128 * 128, 320, 10)
    assert f(0, 1, 8, 1) == 0 and f(1, 1, 12, 1) == 0


class _Net:
    """Just what VideoUNet.plan_key reads (no parameters: the key does not depend on them)."""
    engine = "tc5"
    plan_key = VideoUNet.plan_key


def test_switch_selects_a_distinct_plan_key(monkeypatch):
    net = _Net()
    monkeypatch.delenv("HI3D_DETERMINISTIC", raising=False)
    was = torch.are_deterministic_algorithms_enabled()
    try:
        torch.use_deterministic_algorithms(False)
        assert not ops.deterministic()
        k0, k0s = net.plan_key(32, 64, 64, 16), net.plan_key(16, 64, 64, 8, (0, 2))
        monkeypatch.setenv("HI3D_DETERMINISTIC", "1")
        assert ops.deterministic()
        k1, k1s = net.plan_key(32, 64, 64, 16), net.plan_key(16, 64, 64, 8, (0, 2))
        monkeypatch.setenv("HI3D_DETERMINISTIC", "0")
        assert not ops.deterministic() and net.plan_key(32, 64, 64, 16) == k0
        torch.use_deterministic_algorithms(True)
        assert ops.deterministic() and net.plan_key(32, 64, 64, 16) == k1
    finally:
        torch.use_deterministic_algorithms(was)
    assert k0 != k1 and k0s != k1s and k0[:5] == k1[:5] and k1s[-1] == (0, 2)


def test_fused_sampler_state_follows_the_plan_key():
    """_FusedState (the graph-captured step) is looked up with the plan key, so a toggled switch never replays a stale graph."""
    import inspect

    from hi3d_official_b200 import sampling
    src = inspect.getsource(sampling)
    assert "pkey = unet.plan_key(" in src and "key = (id(unet),) + pkey" in src


def _worker(rank, ws, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(ws))
    dist.init_process_group("gloo", rank=rank, world_size=ws)
    try:
        g = torch.Generator().manual_seed(7)
        parts = [torch.randn(2, 32, 2, generator=g) * 10 ** torch.randint(-3, 4, (2, 32, 2), generator=g) for _ in range(ws)]
        t = parts[rank].clone()
        D.allreduce_sum_(t, deterministic=True)
        ref = parts[0].clone()
        for p in parts[1:]:
            ref += p
        assert torch.equal(t, ref)
        got = [torch.empty_like(t) for _ in range(ws)]
        dist.all_gather(got, t)
        assert all(torch.equal(x, got[0]) for x in got)
        q.put((rank, "ok"))
    except Exception as e:  # noqa: BLE001
        q.put((rank, f"FAIL {type(e).__name__}: {e}"))
    finally:
        dist.destroy_process_group()


def test_two_rank_deterministic_groupnorm_reduction():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert all(r[1] == "ok" for r in res), res
