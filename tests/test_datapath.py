"""Segmentation input pipeline (SURVEY.md 8 f1): the numpy restatement against the recorded outputs of the UNMODIFIED reference
functions where they are deterministic (CPU), and the device pipeline against the restatement (GPU)."""
import contextlib

import numpy as np
import pytest
import torch

from oracle import datapath_ref as D
from tests.reference_golden import Reference

REF = Reference("reference_datapath")


def _scan(n, seed):
    """points on room surfaces, 2-3 cm apart: several points per 4 cm voxel, like an S3DIS scan"""
    r = np.random.RandomState(seed)
    p = r.rand(n, 3).astype(np.float32) * np.array([6.0, 4.0, 3.0], dtype=np.float32)
    kind = r.randint(0, 4, n)
    p[kind == 0, 2] = 0.0
    p[kind == 1, 0] = 0.0
    p[kind == 2, 1] = 4.0
    p += (r.randn(n, 3) * 0.004).astype(np.float32)
    feat = (r.rand(n, 3) * 255).astype(np.float32)
    label = r.randint(0, 13, n).astype(np.float32)
    return p, feat, label


@contextlib.contextmanager
def _reference(module):
    """the UNMODIFIED reference module while its outputs are being recorded, None otherwise"""
    if not REF.recording:
        yield None
        return
    from oracle import ref_loader as RL
    with RL.RefTree("seg") as t:
        yield t.imp(module)


def test_restatement_matches_reference_functions():
    """fnv_hash_vec bit for bit; voxelize as SETS of voxels / members (the reference's argsort is unstable, so the member it
    picks inside a voxel is implementation-defined)."""
    coord, _, _ = _scan(50000, 0)
    c0 = coord - coord.min(0)
    disc = np.floor(c0 / np.float32(0.04))
    with _reference("modules.voxelize_utils") as V:
        REF.equal("fnv_hash_vec", D.fnv_hash_vec(disc), lambda: V.fnv_hash_vec(disc))
        ref_count = REF.array("voxelize.count", lambda: V.voxelize(c0, 0.04, mode=1)[1].astype(np.uint16))
        my_sort, my_count = D.voxelize(c0, 0.04, mode=1)
        assert np.array_equal(ref_count, my_count)
        s = np.cumsum(np.insert(ref_count, 0, 0))
        voxels = np.random.RandomState(1).randint(0, len(ref_count), 200)
        # same members per voxel, any order
        members = lambda order: np.concatenate([np.sort(order[s[v]:s[v + 1]]) for v in voxels])
        assert np.array_equal(REF.array("voxelize.members", lambda: members(V.voxelize(c0, 0.04, mode=1)[0])), members(my_sort))
        np.random.seed(3)
        pick = REF.array("voxelize.pick", lambda: V.voxelize(c0, 0.04).astype(np.uint16))
        keys = D.fnv_hash_vec(disc)
        assert len(pick) == len(ref_count) and len(np.unique(keys[pick])) == len(pick)
        # hash_type='ravel': keys bit for bit (also for a cloud that does not start at the origin), same voxel sizes
        for i, c in enumerate((c0, coord - np.float32(1.7))):
            d = np.floor(c / np.float32(0.04))
            REF.equal(f"ravel_hash_vec[{i}]", D.ravel_hash_vec(d), lambda: V.ravel_hash_vec(d))
        rc = REF.array("voxelize_ravel.count", lambda: V.voxelize(c0, 0.04, hash_type='ravel', mode=1)[1].astype(np.uint16))
        ms, mc = D.voxelize(c0, 0.04, hash_type='ravel', mode=1)
        assert np.array_equal(rc, mc) and np.array_equal(np.sort(rc), np.sort(ref_count))


def test_scene_crop_plan_matches_reference_data_process():
    """data_load's voxel parts and data_process's covering crops (segmentation/tool/test_s3dis.py:114-159) against the
    UNMODIFIED reference functions, same numpy seed.  Rows whose fp32 squared distances to a seed tie exactly come out of the
    reference's unstable argsort in either order (seen: a swapped pair in 13 of 117 crops), so crops are compared as row sets plus
    position-wise agreement.  The reference's crop coordinates and features are kept for a sample of crops."""
    import types
    coord, feat, _ = _scan(30000, 4)
    my_parts = D.scene_parts(coord, 0.04)
    with _reference("tool.test_s3dis") as T:
        def ref_parts():
            T.args = types.SimpleNamespace(voxel_size=0.04, voxel_max=3000, data_norm='mean', color_mean=None, color_std=None)
            idx_sort, count = T.voxelize(coord - np.min(coord, 0), 0.04, mode=1)
            return [idx_sort[np.cumsum(np.insert(count, 0, 0)[0:-1]) + i % count] for i in range(count.max())]
        # same voxels in the same order; which MEMBER is i-th in a voxel is the unstable argsort's choice
        assert np.array_equal(REF.array("scene_parts.sizes", lambda: [len(p) for p in ref_parts()]), [len(p) for p in my_parts])
        assert len(my_parts) >= 2
        assert sorted(np.unique(np.concatenate(my_parts))) == list(range(coord.shape[0]))      # every point is in some part

        ref = []

        def ref_process():
            if not ref:
                np.random.seed(9)
                ref.append(T.data_process(coord.copy(), feat.copy(), my_parts))
            return ref[0]
        ro = [int(o) for o in REF.array("data_process.offsets", lambda: ref_process()[3])]
        sample = np.sort(np.random.RandomState(2).choice(len(ro), 4, replace=False))
        cut = np.cumsum([ro[j] for j in sample])[:-1]
        kept = lambda k, dtype: dict(zip(sample, np.split(REF.array(f"data_process.{k}_sample", lambda: np.concatenate(
            [ref_process()[("rows", "coord", "feat").index(k)][j] for j in sample]).astype(dtype)), cut)))
        ri, rc, rf = kept("rows", np.uint16), kept("coord", np.float32), kept("feat", np.float32)
    np.random.seed(9)
    mi, mc, mf, mo = D.data_process(coord, feat, my_parts, 3000)
    assert ro == mo and len(mi) > len(my_parts)
    same = 0
    for j, b in enumerate(mi):
        # the same rows in every crop, crop after crop
        REF.equal(f"data_process.rows_set[{j}]", np.sort(b), lambda: np.sort(ref_process()[0][j]))
        same += REF.same(f"data_process.rows[{j}]", b, lambda: ref_process()[0][j])
        if j in ri:
            a = ri[j]
            eq = a == b
            assert eq.mean() > 0.99                                    # in the same order except inside distance ties
            assert np.array_equal(rc[j][eq], mc[j][eq]) and np.array_equal(rf[j][eq], mf[j][eq])
    assert same >= len(mi) // 2                                      # most crops have no tie at all


@pytest.mark.gpu
@pytest.mark.parametrize("n,seed", [(50000, 0), (400000, 1), (3000, 2)])
def test_device_voxelize_matches_restatement(n, seed):
    from repsurf_b200.seg import datapath as G
    cuda = torch.device("cuda")
    coord, feat, label = _scan(n, seed)
    c0 = coord - coord.min(0)
    dc = torch.from_numpy(c0).to(cuda)
    disc = np.floor(c0 / np.float32(0.04))
    assert np.array_equal(G.fnv_hash_vec(dc, 0.04).cpu().numpy().view(np.uint64), D.fnv_hash_vec(disc))
    idx_sort, count = G.voxelize(dc, 0.04, mode=1)
    w_sort, w_count = D.voxelize(c0, 0.04, mode=1)
    assert np.array_equal(idx_sort.cpu().numpy(), w_sort) and np.array_equal(count.cpu().numpy(), w_count)
    np.random.seed(5)
    got = G.voxelize(dc, 0.04).cpu().numpy()
    np.random.seed(5)
    assert np.array_equal(got, D.voxelize(c0, 0.04))


@pytest.mark.gpu
def test_device_data_prepare_and_collate_match_restatement():
    from repsurf_b200.seg import datapath as G
    from repsurf_b200.seg import pointops as P
    cuda = torch.device("cuda")
    batch, want = [], []
    for i, n in enumerate((300000, 120000)):
        coord, feat, label = _scan(n, 10 + i)
        np.random.seed(20 + i)
        batch.append(G.data_prepare(torch.from_numpy(coord).to(cuda), torch.from_numpy(feat).to(cuda),
                                    torch.from_numpy(label).to(cuda), voxel_size=0.04, voxel_max=20000))
        np.random.seed(20 + i)
        want.append(D.data_prepare(coord, feat, label, 0.04, 20000))
    for (c, f, l), (wc, wf, wl) in zip(batch, want):
        assert c.shape == wc.shape and c.shape[0] <= 20000
        assert np.array_equal(l.cpu().numpy(), wl.astype(np.int64))           # same points, same order
        assert np.array_equal(f.cpu().numpy(), wf.astype(np.float32))
        assert np.abs(c.cpu().numpy() - wc).max() < 1e-5                       # centring: fp64 mean here, fp32 in numpy
    coord, feat, label, offset = G.collate_fn(batch)
    assert coord.shape[0] == sum(b[0].shape[0] for b in batch)
    assert offset.dtype == torch.int32 and offset.tolist() == list(np.cumsum([b[0].shape[0] for b in batch]))
    assert P.host_offsets(offset) == tuple(offset.tolist())
    # the prepared batch feeds the packed model directly
    from repsurf_b200.models import RepSurfSeg
    out = RepSurfSeg().to(cuda).eval()([coord, feat, offset])
    assert out.shape == (coord.shape[0], 13) and torch.isfinite(out).all()


@pytest.mark.gpu
@pytest.mark.parametrize("shift", [0.0, 1.7])
def test_device_ravel_hash_matches_restatement(shift):
    from repsurf_b200.seg import datapath as G
    cuda = torch.device("cuda")
    coord, _, _ = _scan(120000, 6)
    c0 = coord - coord.min(0) if shift == 0.0 else coord - np.float32(shift)
    dc = torch.from_numpy(c0).to(cuda)
    disc = np.floor(c0 / np.float32(0.04))
    assert np.array_equal(G.ravel_hash_vec(dc, 0.04).cpu().numpy().view(np.uint64), D.ravel_hash_vec(disc))
    idx_sort, count = G.voxelize(dc, 0.04, hash_type='ravel', mode=1)
    w_sort, w_count = D.voxelize(c0, 0.04, hash_type='ravel', mode=1)
    assert np.array_equal(idx_sort.cpu().numpy(), w_sort) and np.array_equal(count.cpu().numpy(), w_count)
    np.random.seed(5)
    got = G.voxelize(dc, 0.04, hash_type='ravel').cpu().numpy()
    np.random.seed(5)
    assert np.array_equal(got, D.voxelize(c0, 0.04, hash_type='ravel'))


@pytest.mark.gpu
def test_device_column_extrema_with_negative_zero():
    """-0.0 among negative coordinates: the float atomics must not take its bit pattern (INT_MIN) for the minimum"""
    from repsurf_b200 import _native as N
    cuda = torch.device("cuda")
    c = torch.tensor([[-5.0, 2.0, -0.0], [-0.0, -3.0, -1.0], [4.0, -0.0, -2.0]], device=cuda).repeat(400, 1).contiguous()
    lo = torch.full((3,), float("inf"), device=cuda)
    hi = torch.full((3,), float("-inf"), device=cuda)
    N.call("rsb_coord_min", c.shape[0], c, lo)
    N.call("rsb_coord_max", c.shape[0], c, hi)
    assert lo.tolist() == [-5.0, -3.0, -2.0] and hi.tolist() == [4.0, 2.0, 0.0]
