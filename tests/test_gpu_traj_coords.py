"""GPU tests of trajectory backmapping from a coordinate array (run on the B200 box: pytest -m gpu): the device radius graph
(engine.radius_graph) against the host CSR form, Plan.set_coords / Backmapper.update_coords against a fresh host upload of the same
coordinates, Backmapper.backmap_coords against Backmapper.backmap_trajectory, and the refusals of set_coords.  Every comparison is
exact."""
import numpy as np
import pytest
import torch

from codlad_b200 import batching, synthetic, topology, weights

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)


@pytest.fixture(scope="module")
def eng():
    from codlad_b200 import engine
    return engine


_BMS = {}


def _bm(precision="f16", sampler="ddpm", eta=0.0, steps=10):
    from codlad_b200 import sampler as S
    key = (precision, sampler, eta, steps)
    if key not in _BMS:
        _BMS[key] = S.Backmapper(weights.init_denoiser_state(0), weights.init_vae_decode_state(0), "N6", num_sampling_steps=steps,
                                 precision=precision, sampler=sampler, eta=eta)
    return _BMS[key]


def _fs_of(proteins, frame, num_ensemble=1):
    from codlad_b200 import sampler as S
    return S.frames_from_batch(synthetic.collate_many(proteins, frame), [p.info for p in proteins], num_ensemble)


# ---- 1. the radius graph ----------------------------------------------------------------------------------------------------------
def _planted():
    """Pairs at exactly 21 A and one ulp either side, on the axes so that every difference and square is exact or rounds the same on
    both sides: residue 0 at the origin, 1 at +21 x, 2 at -(21 - ulp) y, 3 at +(21 + ulp) z (the others are > 29 A apart)."""
    up, down = np.nextafter(np.float32(21), np.float32(30)), np.nextafter(np.float32(21), np.float32(0))
    X = torch.tensor([[0, 0, 0], [21, 0, 0], [0, -float(down), 0], [0, 0, float(up)]], dtype=torch.float32)
    ca = torch.cat([X[:1] - 3.8, X, X[-1:] + 3.8])[None]                                   # termini are not in the graph
    restype = torch.tensor([0, 3, 5, 7, 9, 0])
    return synthetic.SyntheticProtein(restype, ca, topology.build_info(restype[1:-1]))


def _radius_case(case):
    """(X [F,L,3], lengths [F], host row_ptr, host col) of batching.batch_csr(synthetic.radius_graph(...))."""
    if case == "planted":
        prot = _planted()
        batch = synthetic.collate(prot)
        L = prot.L
        X, _ = batching.pad_frames(batch["CG_nxyz"], batch["num_CGs"], L)
        row, col = batching.batch_csr(batch["CG_nbr_list"], batch["num_CGs"], L)
        return X, batch["num_CGs"].to(torch.int32), row, col
    if case == "ragged":
        proteins = [synthetic.make_protein(n, 1, seed=300 + n) for n in (80, 70, 33)]
    elif case == "compact":
        proteins = [synthetic.make_protein(1000, 1, seed=5, compact=0.0015)]
    elif case == "one":
        proteins = [synthetic.make_protein(1, 1, seed=9)]
    else:
        L = int(case[1:])
        prot = synthetic.make_protein(L, 2, seed=L)
        from codlad_b200 import sampler as S
        fs = S.frames_from_batch(synthetic.collate(prot), prot.info)
        return fs.X, fs.lengths, fs.csr_row, fs.csr_col
    fs = _fs_of(proteins, 0)
    return fs.X, fs.lengths, fs.csr_row, fs.csr_col


@pytest.mark.parametrize("case", ["L40", "L300", "L2000", "compact", "ragged", "one", "planted"])
def test_radius_graph_equals_the_host_csr(eng, case):
    X, lengths, row, col = _radius_case(case)
    got_row, got_col = eng.radius_graph(X.cuda(), lengths.cuda())
    F, L = X.shape[:2]
    print(f"radius graph {case}: F={F} L={L}, {col.numel()} edges, {col.numel() / max(1, int(lengths.sum())):.1f} per residue")
    assert got_row.dtype == torch.int32 and got_col.dtype == torch.int32 and got_row.is_cuda
    assert torch.equal(got_row.cpu(), row) and torch.equal(got_col.cpu(), col)
    if case == "compact":
        assert col.numel() / L > 150
    if case == "one":
        assert col.numel() == 0
    if case == "planted":
        assert got_col.cpu().tolist() == [1, 2, 0, 0]          # 0-1 at 21, 0-2 at 21 - ulp; 0-3 at 21 + ulp is out


def test_radius_graph_is_symmetric_and_deterministic(eng):
    prot = synthetic.make_protein(700, 3, seed=17, compact=0.002)
    X = prot.ca_full[:, 1:-1].contiguous().cuda()
    lengths = torch.tensor([700, 650, 1], dtype=torch.int32)
    row, col = eng.radius_graph(X, lengths)
    row2, col2 = eng.radius_graph(X, lengths)
    assert torch.equal(row, row2) and torch.equal(col, col2)
    row, col = row.cpu().long(), col.cpu().long()
    src = torch.repeat_interleave(torch.arange(3 * 700), row[1:] - row[:-1])
    f, i = src // 700, src % 700
    key = (f * 700 + i) * 700 + col
    back = (f * 700 + col) * 700 + i
    assert torch.equal(torch.sort(key).values, torch.sort(back).values)
    assert int(col.max()) < 700 and bool((col[f == 1] < 650).all()) and int((f == 2).sum()) == 0


# ---- 2. plan update against a fresh host upload -----------------------------------------------------------------------------------
def _scaled(proteins, scale):
    """The same proteins with every frame-0 trace scaled about its centroid (fewer edges above 1, more below)."""
    out = []
    for p in proteins:
        ca = p.ca_full[:1]
        c = ca.mean(1, keepdim=True)
        out.append(synthetic.SyntheticProtein(p.restype_full, (c + (ca - c) * scale).contiguous(), p.info))
    return out


def _fresh(bm, fs):
    """A plan of fs's geometry uploaded on the host path (set_frames + set_topology with the host CSR), not shared with bm's cache."""
    from codlad_b200.engine import Plan
    plan = Plan(bm.denoiser, fs.F, fs.NB, fs.L, bm.precision)
    plan.set_frames(fs.X, fs.lengths, fs.cg_z, fs.frame_of)
    plan.set_topology(bm.vae, fs.ca_full, fs.csr_row, fs.csr_col, fs.orders, fs.slot_atom, fs.out_off)
    return plan


def _state(bm, plan, fs, latent):
    out = {name: plan.buffer(name).cpu() for name in ("nbr_idx", "nbr_dist", "hE0")}
    idx, zq, ic, xyz = plan.decode(bm.vae, latent, denorm=True, num_atoms_total=fs.total_atoms)
    out.update(idx=idx.cpu(), zq=zq.cpu(), ic_recon=ic.cpu(), xyz=xyz.cpu())
    return out


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_update_coords_equals_a_fresh_upload(precision):
    """Upload frame set A (ragged 80 / 70 / 33, two members each: NB > F), then move the plan through four coordinate sets whose edge
    count goes down, then up past the first capacity, then back: after every update the k-NN graph, h_E0 and the decode of a fixed
    latent equal those of a plan uploaded from the same coordinates on the host, bit for bit.  The step loop still replays."""
    from codlad_b200 import sampler as S
    bm = _bm(precision)
    base = [synthetic.make_protein(n, 1, seed=400 + n) for n in (80, 70, 33)]
    fs_a = _fs_of(base, 0, 2)
    plan = bm.upload(fs_a)
    latent = synthetic.latent_noise((fs_a.NB, fs_a.L, 3), 5).cuda()
    x = synthetic.latent_noise((fs_a.NB, fs_a.L, 3), 6).cuda()
    bm.sample(plan, fs_a, z=x)
    edges = [int(fs_a.csr_col.numel())]
    for scale in (1.4, 0.55, 0.8, 1.0):
        target = _fs_of(_scaled(base, scale), 0, 2)
        edges.append(int(target.csr_col.numel()))
        bm.update_coords(plan, fs_a, target.ca_full.cuda())
        got = _state(bm, plan, fs_a, latent)
        ref_plan = _fresh(bm, target)
        want = _state(bm, ref_plan, target, latent)
        ref_plan.close()
        for k in want:
            assert torch.equal(got[k], want[k]), (scale, k)
    print(f"update_coords {precision}: edge counts {edges}")
    assert edges[1] < edges[0] < edges[2] and edges[2] > 1.5 * edges[0]
    # the captured step loop is still valid and samples over the new geometry: equal to the fresh plan's pass
    got = bm.sample(plan, fs_a, z=x, step_noise=synthetic.latent_noise((10, fs_a.NB, fs_a.L, 3), 7))["xyz"].cpu()
    bm2 = S.Backmapper(weights.init_denoiser_state(0), weights.init_vae_decode_state(0), "N6", num_sampling_steps=10, precision=precision)
    target = _fs_of(_scaled(base, 1.0), 0, 2)
    want = bm2.sample(bm2.upload(target), target, z=x, step_noise=synthetic.latent_noise((10, fs_a.NB, fs_a.L, 3), 7))["xyz"].cpu()
    assert torch.equal(got, want)


# ---- 3. backmap_coords against backmap_trajectory ---------------------------------------------------------------------------------
VARIANTS = {"ddpm": ("ddpm", 0.0), "ddim_eta0": ("ddim", 0.0), "ddim_eta1": ("ddim", 1.0)}


@pytest.mark.parametrize("precision", ["fp32", "f16"])
@pytest.mark.parametrize("num_ensemble", [1, 3])
@pytest.mark.parametrize("chunks", [1, 3])
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_backmap_coords_equals_backmap_trajectory(variant, chunks, num_ensemble, precision):
    """The same 7-frame trajectory (L = 40) through backmap_trajectory (batch dicts with the host radius graph) and backmap_coords
    (the coordinate array; every graph built on the device), with the same seeded generator: identical host output.  10 steps,
    refinement start 3.  The coordinates go in on the host for one chunk and on the device for three."""
    sampler, eta = VARIANTS[variant]
    prot = synthetic.trajectory(40, 7, seed=61)
    X = prot.ca_full[:, 1:-1].double()
    d = torch.cdist(X, X)
    assert float((d - 21.0).abs().min()) > 1e-4          # no pair where the host graph and the device rule may legitimately differ
    batches = [synthetic.collate(prot, [f]) for f in range(7)]
    bm = _bm(precision, sampler, eta)
    want = bm.backmap_trajectory(batches, prot.info, num_ensemble=num_ensemble, steps=3, chunks=chunks,
                                 generator=torch.Generator(device="cuda").manual_seed(99))
    ca = prot.ca_full if chunks == 1 else prot.ca_full.cuda()
    got = bm.backmap_coords(ca, prot.restype_full, prot.info, num_ensemble=num_ensemble, steps=3, chunks=chunks,
                            generator=torch.Generator(device="cuda").manual_seed(99))
    assert got.shape == want.shape == (7, num_ensemble, prot.num_atoms, 3) and not got.is_cuda
    assert torch.equal(got, want)


# ---- 4. refusals ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_set_coords_refusals(precision):
    from codlad_b200 import _native as N
    from codlad_b200.engine import Plan
    bm = _bm(precision)
    prot = synthetic.make_protein(30, 1, seed=3)
    fs = _fs_of([prot], 0, 2)
    plan = Plan(bm.denoiser, fs.F, fs.NB, fs.L, precision)
    plan.set_frames(fs.X, fs.lengths, fs.cg_z, fs.frame_of)
    ca = fs.ca_full.cuda()
    with pytest.raises(RuntimeError, match="cb2_plan_set_topology has not been called"):
        plan.set_coords(bm.vae, ca)
    plan.set_topology(bm.vae, fs.ca_full, fs.csr_row, fs.csr_col, fs.orders, fs.slot_atom, fs.out_off)
    plan.set_coords(bm.vae, ca)
    with pytest.raises(ValueError, match="shape"):
        plan.set_coords(bm.vae, ca[:, :-1])
    with pytest.raises(ValueError, match="on cuda"):
        plan.set_coords(bm.vae, fs.ca_full)
    with pytest.raises(ValueError, match="shape"):
        bm.update_coords(plan, fs, ca[:, 1:])
    assert N.lib().cb2_plan_set_coords(plan.handle, bm.vae.handle, None, None) != 0
    assert b"null argument" in N.lib().cb2_last_error()
    plan.close()
