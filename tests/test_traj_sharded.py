"""CPU tests of the sharded trajectory driver (ShardedBackmapper.backmap_coords): the (trajectory, run) partition, the job-wide frame
keys, the refusals and a world-2 gloo gather whose per-rank compute is replaced by a stand-in (no GPU here).  The compute itself is
covered by tests/test_gpu_traj_sharded.py."""
import math
import os
import random
import socket
import types

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from codlad_b200 import sampler as S
from codlad_b200 import synthetic

T, STEPS = 10, 3
STAND_IN = types.SimpleNamespace(T=T, k_neighbors=64)        # the fields of a Backmapper the host logic reads


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _job(spec, seed=0):
    """[(ca_full, restype, info)] of synthetic trajectories with (L, frames) = spec."""
    out = []
    for i, (L, n) in enumerate(spec):
        p = synthetic.trajectory(L, n, seed=seed + 31 * i + L)
        out.append((p.ca_full, p.restype_full, p.info))
    return out


def _value(t, f, e):
    return float(100000 * t + 100 * f + e)


def _fake_compute(trajectories, units, runs, offsets, num_ensemble, steps, generator, seed=None):
    """Each unit's block holds _value(t, frame, member) in every coordinate."""
    res = {}
    for t, c in units:
        start, n = runs[t][c]
        na = int(trajectories[t][2][0].numel())
        v = torch.tensor([[_value(t, start + i, e) for e in range(num_ensemble)] for i in range(n)])
        res[(t, c)] = v[:, :, None, None].expand(n, num_ensemble, na, 3).contiguous()
    return res


# ---- 1. the partition -----------------------------------------------------------------------------------------------------------
def _cost(L, n_run, E=2, K=64):
    return L * min(K, L) * E * (T + (n_run - 1) * STEPS)


@pytest.mark.parametrize("chunks", [1, 2, 4, 9])
def test_partition_covers_every_run_once_and_runs_ignore_the_world(chunks):
    rnd = random.Random(chunks)
    n_frames = [rnd.randint(1, 40) for _ in range(17)]
    lengths = [rnd.randint(20, 500) for _ in range(17)]
    first = None
    for world in (1, 2, 3, 8):
        runs, parts = S.partition_trajectory_units(n_frames, lengths, 2, STEPS, T, chunks, world)
        if first is None:
            first = runs
        assert runs == first                                          # runs, and so the coherence breaks, do not depend on world
        assert len(parts) == world and all(p == sorted(p) for p in parts)
        units = [(t, c) for t in range(len(runs)) for c in range(len(runs[t]))]
        assert sorted(sum(parts, [])) == units                         # every (t, run) in exactly one share
        costs = {(t, c): _cost(lengths[t], runs[t][c][1]) for t, c in units}
        loads = [sum(costs[u] for u in p) for p in parts]
        assert max(loads) <= sum(loads) / world + max(costs.values()) + 1e-6
    for t, n in enumerate(n_frames):
        assert first[t] == S.trajectory_chunks(n, min(chunks, n))
        assert sum(k for _, k in first[t]) == n


def test_partition_with_more_ranks_than_units():
    runs, parts = S.partition_trajectory_units([3, 1], [50, 40], 1, STEPS, T, 2, 8)
    assert runs == [[(0, 2), (2, 1)], [(0, 1)]]
    assert sorted(sum(parts, [])) == [(0, 0), (0, 1), (1, 0)] and sum(1 for p in parts if not p) == 5
    # a rank with nothing to do neither computes nor fails: its (process-group-less) result is all NaN
    job = _job([(12, 3), (9, 1)])
    called = []

    def compute(*args, **kw):
        called.append(args[1])
        return _fake_compute(*args, **kw)

    idle = [r for r, p in enumerate(parts) if not p]
    out = S.ShardedBackmapper(STAND_IN, rank=idle[0], world=8).backmap_coords(job, chunks=2, steps=STEPS, _compute=compute)
    assert not called and len(out) == 2 and all(bool(torch.isnan(o).all()) for o in out)


def test_partition_cost_is_lpt_over_units():
    """One 100-frame trajectory at L = 300 and chunks 4: four equal runs, one per rank at world 4; the cost follows the formula."""
    runs, parts = S.partition_trajectory_units([100, 7], [300, 30], 3, STEPS, T, 4, 4, k_neighbors=48)
    assert runs[0] == [(0, 25), (25, 25), (50, 25), (75, 25)] and runs[1] == [(0, 2), (2, 2), (4, 2), (6, 1)]
    assert [sum(1 for t, _ in p if t == 0) for p in parts] == [1, 1, 1, 1]
    with pytest.raises(ValueError, match="chunks"):
        S.partition_trajectory_units([5], [30], 1, STEPS, T, 0, 2)
    with pytest.raises(ValueError, match="chunks"):
        S.partition_trajectory_units([5], [30], 1, STEPS, T, True, 2)


# ---- 2. keys ----------------------------------------------------------------------------------------------------------------------
def test_key_offsets_are_the_frames_before():
    assert S.trajectory_key_offsets([5, 8, 3]) == [0, 5, 13]
    assert S.trajectory_key_offsets([7]) == [0]
    assert S.trajectory_key_offsets([2 ** 46, 2 ** 46]) == [0, 2 ** 46]            # last key 2^47 - 1: allowed
    with pytest.raises(ValueError, match=r"job holds 140737488355329 frames in 2 trajectories.*2\^47"):
        S.trajectory_key_offsets([2 ** 46, 2 ** 46 + 1])


def test_compute_gets_the_job_offsets_and_the_seed():
    job = _job([(12, 5), (9, 8), (15, 3)])
    seen = {}

    def compute(trajectories, units, runs, offsets, num_ensemble, steps, generator, seed=None):
        seen.update(units=units, offsets=offsets, steps=steps, seed=seed, generator=generator, E=num_ensemble)
        return _fake_compute(trajectories, units, runs, offsets, num_ensemble, steps, generator)

    out = S.ShardedBackmapper(STAND_IN, rank=0, world=1).backmap_coords(job, num_ensemble=2, chunks=2, seed=77, _compute=compute)
    assert seen == dict(units=[(0, 0), (0, 1), (1, 0), (1, 1), (2, 0), (2, 1)], offsets=[0, 5, 13], steps=T // 4, seed=77,
                        generator=None, E=2)
    for t, (ca, _, info) in enumerate(job):
        assert out[t].shape == (ca.shape[0], 2, info[0].numel(), 3) and out[t].dtype == torch.float32
        want = torch.tensor([[_value(t, f, e) for e in range(2)] for f in range(ca.shape[0])])
        assert torch.equal(out[t][:, :, 0, 0], want) and not bool(torch.isnan(out[t]).any())


def test_a_job_past_the_key_range_is_refused():
    """Two trajectories of 2^46 and 2^46 + 1 frames (stride-0 views, nothing materialised): the last frame key would be 2^47."""
    (ca, restype, info), = _job([(6, 1)])
    big = [(ca.expand(2 ** 46, -1, -1), restype, info), (ca.expand(2 ** 46 + 1, -1, -1), restype, info)]
    sb = S.ShardedBackmapper(STAND_IN, rank=0, world=1)
    with pytest.raises(ValueError, match="job holds 140737488355329 frames"):
        sb.backmap_coords(big, seed=1, _compute=lambda *a, **k: pytest.fail("computed a refused job"))


# ---- 3. refusals ------------------------------------------------------------------------------------------------------------------
def test_refusals():
    sb = S.ShardedBackmapper(STAND_IN, rank=0, world=2)
    job = _job([(12, 4), (9, 3)])
    ca, restype, info = job[1]
    never = lambda *a, **k: pytest.fail("computed a refused job")
    cases = [
        ([], {}, "no trajectory"),
        (job, {"seed": 1, "generator": torch.Generator()}, "excludes generator"),
        (job, {"chunks": 0}, "chunks"),
        (job, {"chunks": 2.0}, "chunks"),
        (job[:1] + [(ca.double(), restype, info)], {}, "trajectory 1: ca_full"),
        (job[:1] + [(ca[:, :, :2], restype, info)], {}, "trajectory 1: ca_full"),
        (job[:1] + [(ca[:0], restype, info)], {}, "trajectory 1: ca_full"),
        (job[:1] + [(ca, restype[1:], info)], {}, "trajectory 1: restype"),
        (job[:1] + [(ca, restype.float(), info)], {}, "trajectory 1: restype"),
        (job[:1] + [(ca, restype)], {}, "trajectory 1: it must be a tuple"),
        ([ca], {}, "trajectory 0: it must be a tuple"),
        (job, {"num_ensemble": 0}, "trajectory 0: num_ensemble"),
        (job, {"steps": T + 1}, r"trajectory 0: steps must be in \[1, 10\]"),
        (job, {"steps": 0}, "trajectory 0: steps"),
    ]
    for trajectories, kw, msg in cases:
        with pytest.raises(ValueError, match=msg):
            sb.backmap_coords(trajectories, _compute=never, **kw)
    # chunks above a trajectory's frame count is allowed (min(chunks, n) runs), unlike Backmapper.backmap_coords
    out = S.ShardedBackmapper(STAND_IN, rank=0, world=1).backmap_coords(job, chunks=6, _compute=_fake_compute)
    assert [o.shape[0] for o in out] == [4, 3]


# ---- 4. world-2 gather over gloo ------------------------------------------------------------------------------------------------
SPEC = [(12, 5), (20, 8), (9, 3)]          # three trajectories of different Na and frame counts


def _gloo_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    job = _job(SPEC)
    sb = S.ShardedBackmapper(STAND_IN, rank, world)
    out = sb.backmap_coords(job, num_ensemble=3, steps=STEPS, chunks=2, seed=5, _compute=_fake_compute)
    # a job with fewer units than ranks: rank 1 has nothing to send
    small = sb.backmap_coords(_job([(11, 1)]), num_ensemble=2, chunks=2, _compute=_fake_compute)
    if rank == 0:
        q.put((out, small))
    else:
        assert out is None and small is None
    dist.barrier()
    dist.destroy_process_group()


def test_world2_gloo_gathers_every_frame_on_rank0():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    out, small = q.get(timeout=180)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    runs, parts = S.partition_trajectory_units([n for _, n in SPEC], [L for L, _ in SPEC], 3, STEPS, T, 2, world)
    assert all(parts) and {t for t, _ in parts[1]}                 # both ranks busy: some blocks did travel
    job = _job(SPEC)
    assert len(out) == 3
    for t, (ca, _, info) in enumerate(job):
        n, na = ca.shape[0], int(info[0].numel())
        assert out[t].shape == (n, 3, na, 3) and out[t].dtype == torch.float32
        want = torch.tensor([[_value(t, f, e) for e in range(3)] for f in range(n)])
        assert torch.equal(out[t], want[:, :, None, None].expand(n, 3, na, 3)), t
    assert len(small) == 1 and small[0].shape == (1, 2, int(_job([(11, 1)])[0][2][0].numel()), 3)
    assert torch.equal(small[0][:, :, 0, 0], torch.tensor([[_value(0, 0, 0), _value(0, 0, 1)]]))
    assert not math.isnan(float(small[0].sum()))
