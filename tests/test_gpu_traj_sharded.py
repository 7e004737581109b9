"""GPU tests of the sharded trajectory driver (run on the B200 box: pytest -m gpu): ShardedBackmapper.backmap_coords with ranks emulated
on one GPU (rank=r, world=W, no process group; each rank fills its own runs and leaves the others NaN) merged over the ranks against
one GPU, and a real two-process run with its gather on rank 0.  A trajectory is never padded and its runs do not depend on the world
size, so with `seed` the fp32 tier must match bit for bit; the f16 tier within its bar, because its MMA tiles sum a row's
neighbours in a layout that depends on the row's place in the plan.  The tests print how many frames came out bit-identical."""
import os
import socket

import pytest
import torch

from codlad_b200 import synthetic, weights
from tests import parity_utils as P

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)

BARS = {"fp32": 0.0, "f16": 1.5e-3}
SEED = 0x5EED_0000_7A5C_0009
VARIANTS = {"ddpm10": ("ddpm", "10", 0.0), "ddim50_eta0": ("ddim", "ddim50", 0.0)}
E = 2

_BMS = {}


def _bm(precision, variant):
    from codlad_b200 import sampler as S
    key = (precision, variant)
    if key not in _BMS:
        sampler, steps, eta = VARIANTS[variant]
        _BMS[key] = S.Backmapper(weights.init_denoiser_state(0), weights.init_vae_decode_state(0), "N6", num_sampling_steps=steps,
                                 precision=precision, sampler=sampler, eta=eta)
    return _BMS[key]


def _job(spec, seed):
    out = []
    for i, (L, n) in enumerate(spec):
        p = synthetic.trajectory(L, n, seed=seed + 17 * i)
        out.append((p.ca_full, p.restype_full, p.info))
    return out


def _emulated(bm, job, world, chunks):
    """backmap_coords of every rank r < world (no process group), merged: each frame must come from exactly one rank."""
    from codlad_b200 import sampler as S
    merged = None
    for r in range(world):
        sb = S.ShardedBackmapper(bm, rank=r, world=world)
        out = sb.backmap_coords(job, num_ensemble=E, chunks=chunks, seed=SEED)
        if merged is None:
            merged = [torch.full_like(o, float("nan")) for o in out]
        for m, o in zip(merged, out):
            mine = ~torch.isnan(o).flatten(1).all(1)
            assert bool(torch.isnan(m[mine]).all()), "a frame came from two ranks"
            assert not bool(torch.isnan(o[mine]).any())
            m[mine] = o[mine]
    for m in merged:
        assert not bool(torch.isnan(m).any()), "a frame came from no rank"
    return merged


def _compare(got, want, precision, label):
    same = total = 0
    worst = 0.0
    for t, (g, w) in enumerate(zip(got, want)):
        assert g.shape == w.shape and g.dtype == torch.float32 and not g.is_cuda
        for f in range(w.shape[0]):
            same += int(torch.equal(g[f], w[f]))
            total += 1
        err = P.rel_err(g, w)
        worst = max(worst, err)
        if precision == "fp32":
            assert torch.equal(g, w), (label, t, err)
        else:
            assert err < BARS[precision], (label, t, err)
    print(f"{label}: worst coordinate rel err {worst:.3e}, bit-identical frames {same}/{total}")


# ---- 1. one trajectory: the sharded driver against Backmapper.backmap_coords ----------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "f16"])
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_one_trajectory_against_backmap_coords(variant, precision):
    """L = 70, 9 frames, 2 members, chunks 4 (runs of 3 / 2 / 2 / 2 frames): world 1 is Backmapper.backmap_coords bit for bit (the
    same plan); worlds 2, 3 and 4, merged over the ranks, match it within the tier's bar."""
    from codlad_b200 import sampler as S
    bm = _bm(precision, variant)
    job = _job([(70, 9)], seed=901)
    ca, restype, info = job[0]
    want = [bm.backmap_coords(ca, restype, info, num_ensemble=E, chunks=4, seed=SEED)]
    one = S.ShardedBackmapper(bm, rank=0, world=1).backmap_coords(job, num_ensemble=E, chunks=4, seed=SEED)
    assert len(one) == 1 and torch.equal(one[0], want[0])
    for world in (2, 3, 4):
        _, parts = S.partition_trajectory_units([9], [70], E, bm.T // 4, bm.T, 4, world)
        print(f"{variant} {precision} world {world}: runs per rank {[[c for _, c in p] for p in parts]}")
        _compare(_emulated(bm, job, world, 4), want, precision, f"{variant} {precision} world {world} vs backmap_coords")


# ---- 2. three trajectories: worlds 2 and 3 against world 1 ----------------------------------------------------------------------
SPEC = [(40, 5), (70, 8), (120, 3)]           # L = 40 runs with K = 40


@pytest.mark.parametrize("precision", ["fp32", "f16"])
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_three_trajectories_against_world_one(variant, precision):
    from codlad_b200 import sampler as S
    bm = _bm(precision, variant)
    job = _job(SPEC, seed=733)
    want = S.ShardedBackmapper(bm, rank=0, world=1).backmap_coords(job, num_ensemble=E, chunks=2, seed=SEED)
    assert [tuple(w.shape) for w in want] == [(n, E, int(info[0].numel()), 3) for (_, n), (_, _, info) in zip(SPEC, job)]
    ca, restype, info = job[1]                  # a trajectory's own frame keys start at its offset: not what it draws alone
    alone = bm.backmap_coords(ca, restype, info, num_ensemble=E, chunks=2, seed=SEED)
    assert not torch.equal(alone, want[1])
    for world in (2, 3):
        _compare(_emulated(bm, job, world, 2), want, precision, f"{variant} {precision} world {world} vs world 1")


# ---- 3. a real two-process run --------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, backend, path):
    import torch.distributed as dist
    from codlad_b200 import sampler as S
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    dev = torch.device("cuda", rank % torch.cuda.device_count())
    torch.cuda.set_device(dev)
    torch.set_grad_enabled(False)
    kw = {"device_id": dev} if backend == "nccl" else {}
    dist.init_process_group(backend, rank=rank, world_size=world, **kw)
    try:
        out = S.ShardedBackmapper(_bm("fp32", "ddim50_eta0")).backmap_coords(_job(SPEC, seed=733), num_ensemble=E, chunks=2,
                                                                              seed=SEED)
        if rank == 0:
            torch.save(out, path)
        else:
            assert out is None
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("backend", ["nccl", "gloo"])
def test_two_processes_gather_on_rank0(backend, tmp_path):
    """Two processes over torch.distributed: rank 0's output equals the world-1 result bit for bit (fp32 tier).  NCCL needs two GPUs
    and sends from the device; gloo sends from the host and runs both ranks on one GPU when there is only one."""
    if backend == "nccl" and torch.cuda.device_count() < 2:
        pytest.skip(f"NCCL needs two GPUs, {torch.cuda.device_count()} present")
    import torch.multiprocessing as mp
    from codlad_b200 import sampler as S
    want = S.ShardedBackmapper(_bm("fp32", "ddim50_eta0"), rank=0, world=1).backmap_coords(_job(SPEC, seed=733), num_ensemble=E,
                                                                                           chunks=2, seed=SEED)
    path = str(tmp_path / "rank0.pt")
    ctx = mp.get_context("spawn")
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, backend, path)) for r in range(2)]
    try:
        for p in procs:
            p.start()
        for p in procs:
            p.join(timeout=600)
            assert p.exitcode == 0, p.exitcode
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join()
    got = torch.load(path)
    _compare(got, want, "fp32", f"two processes ({backend}) vs world 1")
