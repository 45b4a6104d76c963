"""Slab layout (me_set_layout, ME_LAYOUT_SLAB): every rank of a multi-GPU job lays out and evaluates only the voxel layers it
owns.  One context per rank on ONE device stands in for the ranks; the all-reduces of the job (SUM / MAX over the accumulator
block, MAX over the W table of the voxel stage) are done here with torch on that device.  The reduced results must reproduce
the world = 1 pass: counts bit-exact, sums to summation order."""
import numpy as np
import pytest

from cloud_map_evaluation_b200 import _abi as A
from cloud_map_evaluation_b200 import dist as mdist
from cloud_map_evaluation_b200 import synth

pytestmark = pytest.mark.gpu

EST, GT = A.ME_CLOUD_EST, A.ME_CLOUD_GT


@pytest.fixture(scope="module")
def api():
    from cloud_map_evaluation_b200 import api as _api
    return _api


def _view(ptr, n):
    import torch
    return torch.as_tensor(mdist._DeviceBlock(ptr, n), device="cuda:0")


def _reference(api, est, gt, p, radius, vox, min_points, gt_mme=True, **kw):
    with api.MapEvalB200(vmd_voxel_size=vox, **kw) as ctx:
        ctx.set_cloud(EST, est)
        ctx.set_cloud(GT, gt)
        m_e = ctx.eval_mme_accum(EST, radius, 10)
        ent_e = ctx.get_entropies(EST)
        m_g = ctx.eval_mme_accum(GT, radius, 5) if gt_mme else None
        e, g = ctx.eval_nn_accum(p)
        nn_e, nn_g = ctx.get_nn(EST), ctx.get_nn(GT)
        awd = ctx.calculateVMD(vox, min_points, 5)
    return dict(m_e=m_e, m_g=m_g, e=e, g=g, awd=awd, ent_e=ent_e, nn_e=nn_e, nn_g=nn_g)


def _slab_job(api, est, gt, p, radius, vox, min_points, world, gt_mme=True, per_point=True, **kw):
    """the pass of bench.py on `world` ranks, all of them contexts on cuda:0"""
    import torch
    ctxs = []
    out = {}
    try:
        for r in range(world):
            c = api.MapEvalB200(rank=r, world=world, vmd_voxel_size=vox, **kw)
            c.set_layout(A.ME_LAYOUT_SLAB)
            c.set_cloud(EST, est)
            c.set_cloud(GT, gt)
            ctxs.append(c)
        ents, nns_e, nns_g = [], [], []
        for c in ctxs:
            c.accum_reset()
            c.eval_mme_accum_device(EST, radius, 10)
            if per_point:
                ents.append(c.get_entropies(EST))
            if gt_mme:
                c.eval_mme_accum_device(GT, radius, 5)
            c.eval_nn_accum_device(p)
            if per_point:
                nns_e.append(c.get_nn(EST))
                nns_g.append(c.get_nn(GT))
            c.voxel_begin(vox, min_points)
            c.synchronize()
        out["layouts"] = [c.layout_active() for c in ctxs]
        slab = all(l["layout"] == A.ME_LAYOUT_SLAB for l in out["layouts"])
        assert slab or all(l["layout"] == A.ME_LAYOUT_REPLICATED for l in out["layouts"]), "ranks disagree on the layout"
        out["slab"] = slab
        if slab:
            tabs = [_view(*c.voxel_w_table()) for c in ctxs]
            assert len({t.numel() for t in tabs}) == 1
            owners = torch.stack([(t >= 0).to(torch.int32) for t in tabs]).sum(0)
            assert int(owners.max()) <= 1, "a voxel pair computed by two ranks"
            m = torch.stack(tabs).max(0).values
            for t in tabs:
                t.copy_(m)
            torch.cuda.synchronize()
        for c in ctxs:
            c.voxel_finish_accum_device(5)
            c.synchronize()
        blocks = []
        for c in ctxs:
            ptr, n_sum, n_max = c.accum_block()
            blocks.append(_view(ptr, n_sum + n_max))
        allb = torch.stack(blocks)
        red = torch.cat([allb[:, :n_sum].sum(0), allb[:, n_sum:].max(0).values])
        out["blocks"] = allb.cpu().numpy()
        blocks[0].copy_(red)
        torch.cuda.synchronize()
        e, g, mm = ctxs[0].accum_fetch(want_mme=(True, gt_mme))
        out.update(e=e, g=g, m_e=mm[0], m_g=mm[1] if gt_mme else None, awd=ctxs[0].accum_fetch_awd(), ents=ents, nns_e=nns_e,
                   nns_g=nns_g)
    finally:
        for c in ctxs:
            c.close()
    return out


def _cmp_acc(a, b):
    da, db = A.struct_to_dict(a), A.struct_to_dict(b)
    for k in ("n_query", "n_corr", "n_inlier", "n_ub"):
        assert da[k] == db[k], k
    for k in ("sum_d", "sum_d2", "sum_d_all", "sum_d2_all", "sum_nn_dist"):
        np.testing.assert_allclose(da[k], db[k], rtol=1e-11, err_msg=k)


def _cmp_job(job, ref, n_est, n_gt, world):
    assert job["slab"], job["layouts"]
    lay = job["layouts"]
    # every point has exactly one owner, and no rank lays out the whole cloud
    assert sum(l["n_owned"][0] for l in lay) == n_est and sum(l["n_owned"][1] for l in lay) == n_gt
    assert max(l["n_laid_out"][0] for l in lay) < n_est
    _cmp_acc(job["e"], ref["e"])
    _cmp_acc(job["g"], ref["g"])
    assert job["e"].n_query == n_est and job["g"].n_query == n_gt
    for m, r in ((job["m_e"], ref["m_e"]), (job["m_g"], ref["m_g"])):
        if r is None:
            continue
        assert (m.n_query, m.n_valid) == (r.n_query, r.n_valid)
        np.testing.assert_allclose(m.sum_entropy, r.sum_entropy, rtol=1e-11)
        assert (m.min_entropy, m.max_entropy) == (r.min_entropy, r.max_entropy)
    a, r = job["awd"], ref["awd"]
    for k in ("n_pairs", "n_scs", "n_voxels_est", "n_voxels_gt", "n_active", "n_new", "n_old"):
        assert getattr(a, k) == getattr(r, k), k
    np.testing.assert_allclose([a.awd, a.scs], [r.awd, r.scs], rtol=1e-11, equal_nan=True)
    if job["ents"]:
        # per-point outputs: a rank reports the points it owns (0 / NaN elsewhere); together they are the world = 1 arrays
        np.testing.assert_allclose(np.sum(job["ents"], axis=0), ref["ent_e"], rtol=1e-9, atol=1e-12)
        for got, exp in ((job["nns_e"], ref["nn_e"]), (job["nns_g"], ref["nn_g"])):
            d2 = np.stack([g[1] for g in got])
            idx = np.stack([g[0] for g in got])
            evaluated = ~np.isnan(d2)
            assert np.all(evaluated.sum(0) == 1)
            sel = evaluated.argmax(0)
            cols = np.arange(d2.shape[1])
            np.testing.assert_array_equal(d2[sel, cols], exp[1])
            np.testing.assert_array_equal(idx[sel, cols], exp[0])


# Surface scenes refine to cell edges whose dense table exceeds the budget and get the sparse cell table, which is laid out whole
# (-> replicated layout).  A caller-fixed cell edge of 0.5 m keeps this scaled-down scene on the dense table.
OUTDOOR = dict(nn_cell_size=0.5)


@pytest.mark.parametrize("world", [3, 8])
def test_flat_outdoor_scene_is_cut_along_y(api, world):
    """200 m x 200 m of ground, walls and trunks: 67 voxel layers along y, 5 along z (most points in two of them)."""
    est, gt, cfg = synth.make_pair("C4", scale=0.004)
    p = A.make_nn_params(cfg["tau"], 1.0)
    ref = _reference(api, est, gt, p, cfg["nn_radius"], cfg["vmd_voxel_size"], 8, **OUTDOOR)
    job = _slab_job(api, est, gt, p, cfg["nn_radius"], cfg["vmd_voxel_size"], 8, world, **OUTDOOR)
    _cmp_job(job, ref, len(est), len(gt), world)
    assert {l["axis"] for l in job["layouts"]} == {1}
    assert ref["awd"].n_pairs > 50 and ref["awd"].n_scs > 0
    # the busiest rank lays out about 1 / world of the cloud (+ halo, + the granularity of 3 m voxel layers)
    assert max(l["n_laid_out"][0] for l in job["layouts"]) < 1.7 * len(est) / world


@pytest.mark.parametrize("world", [2, 3])
def test_c3_box_at_small_scale(api, world):
    est, gt, cfg = synth.make_pair("C3", scale=0.02)
    p = A.make_nn_params(cfg["tau"], 1.0)
    ref = _reference(api, est, gt, p, cfg["nn_radius"], cfg["vmd_voxel_size"], 20)
    job = _slab_job(api, est, gt, p, cfg["nn_radius"], cfg["vmd_voxel_size"], 20, world)
    _cmp_job(job, ref, len(est), len(gt), world)
    assert len({l["axis"] for l in job["layouts"]}) == 1
    assert ref["awd"].n_pairs > 50 and ref["awd"].n_scs > 0


@pytest.mark.parametrize("world", [2, 4])
def test_uniform_box(api, world):
    est, gt, cfg = synth.make_pair("C1", scale=0.5)
    vox = cfg["side"] / 16.0
    p = A.make_nn_params(cfg["tau"], 1.0, pairing=A.ME_PAIRING_AS_WRITTEN)
    ref = _reference(api, est, gt, p, 0.1, vox, 5)
    job = _slab_job(api, est, gt, p, 0.1, vox, 5, world)
    _cmp_job(job, ref, len(est), len(gt), world)
    assert ref["awd"].n_pairs > 100


@pytest.mark.parametrize("world", [2, 5])
def test_indoor_rooms_small_radius(api, world):
    est, gt, cfg = synth.make_pair("C5", scale=0.001)
    p = A.make_nn_params(cfg["tau"], 1.0)
    ref = _reference(api, est, gt, p, cfg["nn_radius"], cfg["vmd_voxel_size"], 10, gt_mme=False)
    job = _slab_job(api, est, gt, p, cfg["nn_radius"], cfg["vmd_voxel_size"], 10, world, gt_mme=False)
    _cmp_job(job, ref, len(est), len(gt), world)


@pytest.mark.parametrize("world", [2, 4])
def test_neighbours_on_other_ranks_slabs(api, world):
    """The ground truth covers only the south half of the scene, the estimate all of it (plus isolated points): the nearest
    neighbour of most northern points lies tens of metres away, on another rank's slab — found by the exact finish over the
    whole cloud; full Chamfer and the per-point outputs see them."""
    est, gt, cfg = synth.make_pair("C4", scale=0.004)
    gt = np.ascontiguousarray(gt[gt[:, 1] < 90.0])
    rs = np.random.RandomState(5)
    out = np.column_stack([rs.uniform(1, 199, 300), rs.uniform(1, 199, 300), rs.uniform(0.5, 6, 300)])      # inside the scene's box
    est = np.ascontiguousarray(np.vstack([est, out.astype(np.float32).astype(np.float64)]))
    assert 0.3 * len(est) < np.count_nonzero(est[:, 1] > 100.0)
    p = A.make_nn_params(cfg["tau"], 1.0)
    ref = _reference(api, est, gt, p, cfg["nn_radius"], cfg["vmd_voxel_size"], 8, **OUTDOOR)
    job = _slab_job(api, est, gt, p, cfg["nn_radius"], cfg["vmd_voxel_size"], 8, world, **OUTDOOR)
    _cmp_job(job, ref, len(est), len(gt), world)
    assert ref["e"].n_far > 1000


def test_scene_that_cannot_be_cut_stays_replicated(api):
    """Too few voxel layers for the world size: the slab request is ignored, the replicated path runs as before."""
    est, gt, cfg = synth.make_pair("C1", scale=0.05)
    p = A.make_nn_params(cfg["tau"], 1.0)
    with api.MapEvalB200(vmd_voxel_size=cfg["side"]) as ctx:
        ctx.set_cloud(EST, est)
        ctx.set_cloud(GT, gt)
        e_ref, g_ref = ctx.eval_nn_accum(p)
    tot = None
    for r in range(4):
        with api.MapEvalB200(rank=r, world=4, vmd_voxel_size=cfg["side"]) as ctx:
            ctx.set_layout(A.ME_LAYOUT_SLAB)
            ctx.set_cloud(EST, est)
            ctx.set_cloud(GT, gt)
            e, g = ctx.eval_nn_accum(p)
            lay = ctx.layout_active()
            assert lay["layout"] == A.ME_LAYOUT_REPLICATED and lay["n_laid_out"] == [len(est), len(gt)]
            awd = ctx.calculateVMD(cfg["side"], 5, 5)      # the one-call voxel stage is available on a replicated layout
            assert awd.n_voxels_est >= 1
        tot = [e.n_query, list(e.n_inlier)] if tot is None else [tot[0] + e.n_query, [a + b for a, b in zip(tot[1], e.n_inlier)]]
    assert tot[0] == len(est) and tot[1] == list(e_ref.n_inlier)


def test_one_call_voxel_stage_refuses_an_active_slab_layout(api):
    est, gt, cfg = synth.make_pair("C5", scale=0.001)
    with api.MapEvalB200(rank=1, world=2, vmd_voxel_size=cfg["vmd_voxel_size"]) as ctx:
        ctx.set_layout(A.ME_LAYOUT_SLAB)
        ctx.set_cloud(EST, est)
        ctx.set_cloud(GT, gt)
        with pytest.raises(Exception, match="slab layout"):
            ctx.calculateVMD(cfg["vmd_voxel_size"], 20, 5)
        with pytest.raises(Exception, match="replicated layout"):
            ctx.estimate_normals(EST, 10)
        # back to the replicated layout: the same context serves the one-call stage again
        ctx.set_layout(A.ME_LAYOUT_REPLICATED)
        assert ctx.calculateVMD(cfg["vmd_voxel_size"], 20, 5).n_voxels_est > 0


def test_sparse_cell_table_stays_replicated(api):
    """A scene that gets the sparse cell table (laid out whole) ignores the slab request: same results, replicated layout."""
    est, gt, cfg = synth.make_pair("C4", scale=0.004)
    p = A.make_nn_params(cfg["tau"], 1.0)
    sparse = dict(max_grid_cells=1)         # a budget of one cell: this small scene would otherwise get a dense table
    ref = _reference(api, est, gt, p, cfg["nn_radius"], cfg["vmd_voxel_size"], 20, **sparse)
    tot = 0
    for r in range(2):
        with api.MapEvalB200(rank=r, world=2, vmd_voxel_size=cfg["vmd_voxel_size"], **sparse) as ctx:
            ctx.set_layout(A.ME_LAYOUT_SLAB)
            ctx.set_cloud(EST, est)
            ctx.set_cloud(GT, gt)
            e, g = ctx.eval_nn_accum(p)
            assert ctx.layout_active()["layout"] == A.ME_LAYOUT_REPLICATED
            tot += e.n_inlier[0]
    assert tot == ref["e"].n_inlier[0]
