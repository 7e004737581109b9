"""CPU tests of the keyed sampling noise: the Philox4x32-10 restatement (tests/noise_oracle.py) against Random123's known-answer
vectors, the restatement's own invariances, sampler.member_keys, and the argument checks of engine.keyed_normal and of the seeded
Backmapper entry points (which refuse before touching a device)."""
import numpy as np
import pytest
import torch

from codlad_b200 import engine, sampler, synthetic
from tests import noise_oracle as O

KAT = [  # Random123 kat_vectors, philox4x32 with 10 rounds: counter, key -> output
    ([0, 0, 0, 0], [0, 0], [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]),
    ([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2, [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]),
    ([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0], [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]),
]


@pytest.mark.parametrize("case", range(len(KAT)))
def test_philox_known_answers(case):
    ctr, key, want = KAT[case]
    got = O.philox4x32_10(np.array(ctr, dtype=np.uint32), np.array(key, dtype=np.uint32))
    assert got.tolist() == want


def test_philox_vectorised_equals_scalar():
    rng = np.random.default_rng(0)
    ctr = rng.integers(0, 2 ** 32, size=(64, 4), dtype=np.uint64).astype(np.uint32)
    key = rng.integers(0, 2 ** 32, size=(64, 2), dtype=np.uint64).astype(np.uint32)
    batch = O.philox4x32_10(ctr, key)
    for r in range(64):
        assert O.philox4x32_10(ctr[r], key[r]).tolist() == batch[r].tolist()


def test_uniform_is_in_half_open_unit_interval():
    w = np.array([0, 255, 256, 0x7FFFFFFF, 0x80000000, 0xFFFFFEFF, 0xFFFFFFFF], dtype=np.uint32)
    u = O.uniform01(w)
    assert u.dtype == np.float32
    assert u[0] == u[1] == np.float32(2.0 ** -25)            # the smallest value: log never sees 0
    assert u[2] == np.float32(1.5 * 2.0 ** -24)
    assert bool((u > 0).all()) and bool((u <= 1).all())
    assert u[4] == np.float32(0.5)                           # above 2^23 the + 0.5 rounds to even ...
    assert u[6] == np.float32(1.0)                           # ... and the largest word gives u = 1: the range is (0, 1]


def test_restatement_counter_layout():
    """Channel values come from counter (key lo, key hi, draw, (slice << 21) | i) with key (seed lo, seed hi)."""
    seed, key, draw, s, i = 0x0123456789ABCDEF, (7 << 16) + 3, 5, 9, 17
    w = O.philox4x32_10(np.array([key & 0xFFFFFFFF, key >> 32, draw, (s << 21) | i], dtype=np.uint32),
                        np.array([seed & 0xFFFFFFFF, seed >> 32], dtype=np.uint32))
    u = O.uniform01(w).astype(np.float64)
    want = [np.sqrt(-2 * np.log(u[0])) * np.cos(2 * np.pi * u[1]), np.sqrt(-2 * np.log(u[0])) * np.sin(2 * np.pi * u[1]),
            np.sqrt(-2 * np.log(u[2])) * np.cos(2 * np.pi * u[3])]
    got = O.keyed_normal(seed, [key], 20, draw, s, 1)[0, 0, i]
    assert np.array_equal(got, np.array(want))


def test_restatement_partial_fill_and_padding():
    keys = [0, 1, (3 << 16) + 2, 2 ** 62 + 5]
    full = O.keyed_normal(11, keys, 12, 3, 0, 20)
    assert np.array_equal(O.keyed_normal(11, keys, 12, 3, 5, 7), full[5:12])
    assert np.array_equal(O.keyed_normal(11, keys, 40, 3, 0, 20)[:, :, :12], full)
    assert np.array_equal(O.keyed_normal(11, keys[2:3], 12, 3, 0, 20)[:, 0], full[:, 2])
    assert not np.array_equal(O.keyed_normal(11, keys, 12, 4, 0, 20), full)
    assert not np.array_equal(O.keyed_normal(12, keys, 12, 3, 0, 20), full)


# ---- member keys -------------------------------------------------------------------------------------------------------------------
def _fs(lengths=(20, 15, 9), num_ensemble=1, frame_of=None):
    proteins = [synthetic.make_protein(n, 1, seed=40 + n) for n in lengths]
    return sampler.frames_from_batch(synthetic.collate_many(proteins, 0), [p.info for p in proteins], num_ensemble, frame_of=frame_of)


def test_member_keys_ensemble_major():
    fs = _fs(num_ensemble=4)
    keys = sampler.member_keys(fs)
    assert keys.dtype == torch.int64 and keys.shape == (12,) and not keys.is_cuda
    want = [f * 65536 + e for e in range(4) for f in range(3)]             # b = e * F + f
    assert keys.tolist() == want


def test_member_keys_explicit_members_and_frame_keys():
    fs = _fs(frame_of=[2, 0, 2, 1, 0, 2])
    assert sampler.member_keys(fs).tolist() == [2 * 65536, 0, 2 * 65536 + 1, 65536, 1, 2 * 65536 + 2]
    got = sampler.member_keys(fs, frame_keys=torch.tensor([100, 7, 2 ** 47 - 1]))
    assert got.tolist() == [(2 ** 47 - 1) * 65536, 100 * 65536, (2 ** 47 - 1) * 65536 + 1, 7 * 65536, 100 * 65536 + 1,
                            (2 ** 47 - 1) * 65536 + 2]
    assert sampler.member_keys(fs, frame_keys=[100, 7, 3]).tolist() == sampler.member_keys(fs, np.array([100, 7, 3])).tolist()


def test_member_keys_refusals():
    fs = _fs(frame_of=[0, 1, 2])
    for bad in ([0, 1], [0, 1, -1], [0, 1, 2 ** 47], torch.tensor([0.0, 1.0, 2.0]), torch.tensor([True, False, True])):
        with pytest.raises(ValueError):
            sampler.member_keys(fs, frame_keys=bad)
    big = _fs(lengths=(4,), frame_of=[0] * 65536)
    assert sampler.member_keys(big)[-1] == 65535
    with pytest.raises(ValueError, match="2\\^16"):
        sampler.member_keys(_fs(lengths=(4,), frame_of=[0] * 65537))


def test_unit_keys_match_member_keys_of_the_whole_job():
    fs = _fs(num_ensemble=3)                                               # b = e * 3 + f
    units = [(f, e) for e in range(3) for f in range(3)]
    assert sampler.unit_keys(units).tolist() == sampler.member_keys(fs).tolist()
    assert sampler.unit_keys([(2, 1), (0, 65535), (2 ** 47 - 1, 0)]).tolist() == [2 * 65536 + 1, 65535, (2 ** 47 - 1) * 65536]
    assert sampler.unit_keys([]).shape == (0,)
    for bad in ([(0, 65536)], [(2 ** 47, 0)], [(-1, 0)], [(0, -1)]):
        with pytest.raises(ValueError):
            sampler.unit_keys(bad)


def test_sharded_backmap_hands_the_seed_to_the_compute_hook():
    sb = sampler.ShardedBackmapper(None, rank=0, world=1)
    prot = synthetic.make_protein(12, 1, seed=3)
    batches, infos = [synthetic.collate(prot)], [prot.info]
    seen = []

    def with_seed(batches, infos, units, lengths, generator, seed=None):
        seen.append(seed)
        return {u: torch.zeros(prot.num_atoms, 3) for u in units}

    sb.backmap(batches, infos, 2, _compute=with_seed, seed=17)
    sb.backmap(batches, infos, 2, _compute=with_seed)
    assert seen == [17, None]

    def without_seed(batches, infos, units, lengths, generator):
        return {u: torch.zeros(prot.num_atoms, 3) for u in units}

    sb.backmap(batches, infos, 2, _compute=without_seed)
    with pytest.raises(TypeError):                                         # a hook that cannot take the seed never drops it silently
        sb.backmap(batches, infos, 2, _compute=without_seed, seed=17)


# ---- argument checks ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bad", [
    dict(seed=-1), dict(seed=2 ** 64), dict(seed=1.0), dict(seed=True), dict(draw=-1), dict(draw=2 ** 32), dict(L=0), dict(L=2 ** 21),
    dict(first_slice=-1), dict(n_slices=0), dict(first_slice=2000, n_slices=49), dict(first_slice=2048), dict(n_slices=1.0)])
def test_keyed_normal_scalar_refusals(bad):
    args = dict(seed=1, L=10, draw=0, first_slice=0, n_slices=3)
    args.update(bad)
    with pytest.raises(ValueError):
        engine.check_keyed_normal_args(**args)


def test_keyed_normal_scalar_limits_accepted():
    engine.check_keyed_normal_args(2 ** 64 - 1, 2 ** 21 - 1, 2 ** 32 - 1, 2047, 1)
    engine.check_keyed_normal_args(0, 1, 0, 0, 2048)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_keyed_normal_has_no_cpu_fallback():
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        engine.keyed_normal(1, torch.zeros(2, dtype=torch.int64), 4, 0, 0, 1)


def test_seeded_entry_points_refuse_mixed_noise_sources():
    fs = _fs(num_ensemble=2)
    check = sampler.Backmapper._check_noise_args
    check(fs, None, None, None, None, None, 0)                              # today's path
    check(fs, torch.zeros(1), torch.zeros(1), torch.Generator(), None, None, 0)
    check(fs, None, None, None, 5, None, 7)
    check(fs, None, None, None, 5, torch.zeros(fs.NB, dtype=torch.int64), 0)
    with pytest.raises(ValueError, match="excludes"):
        check(fs, None, None, torch.Generator(), 5, None, 0)
    with pytest.raises(ValueError, match="excludes"):
        check(fs, torch.zeros(1), None, None, 5, None, 0)
    with pytest.raises(ValueError, match="excludes"):
        check(fs, None, torch.zeros(1), None, 5, None, 0)
    with pytest.raises(ValueError, match="need a seed"):
        check(fs, None, None, None, None, torch.zeros(fs.NB, dtype=torch.int64), 0)
    with pytest.raises(ValueError, match="need a seed"):
        check(fs, None, None, None, None, None, 1)
    for keys in (torch.zeros(fs.NB, dtype=torch.int32), torch.zeros(fs.NB + 1, dtype=torch.int64), [0] * fs.NB):
        with pytest.raises(ValueError, match="keys"):
            check(fs, None, None, None, 5, keys, 0)
    for seed, draw in ((-1, 0), (2 ** 64, 0), (1, -1), (1, 2 ** 32)):
        with pytest.raises(ValueError):
            check(fs, None, None, None, seed, None, draw)
