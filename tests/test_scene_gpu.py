"""Whole-scene inference (SURVEY.md 8 f2): the kNN(32) label median filter on ONE segment of 10^6 points and the vote
accumulation of segmentation/tool/test_s3dis.py, on the sm_100a operators."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
cuda = torch.device("cuda")


def _room(n, seed):
    """points on the surfaces of a 30 x 20 x 3 m room with furniture-like blobs: surface-heavy like S3DIS scans"""
    g = torch.Generator().manual_seed(seed)
    u = torch.rand(n, 3, generator=g)
    kind = torch.randint(0, 6, (n,), generator=g)
    p = u * torch.tensor([30.0, 20.0, 3.0])
    p[kind == 0, 2] = 0.0                                   # floor
    p[kind == 1, 2] = 3.0                                   # ceiling
    p[kind == 2, 0] = 0.0                                   # walls
    p[kind == 3, 1] = 20.0
    blob = kind >= 4                                        # dense clusters
    centres = torch.rand(64, 3, generator=g) * torch.tensor([30.0, 20.0, 1.5])
    which = torch.randint(0, 64, (n,), generator=g)
    p[blob] = centres[which[blob]] + 0.3 * torch.randn(int(blob.sum()), 3, generator=g)
    return (p + 1e-3 * torch.randn(n, 3, generator=g)).contiguous()


def test_grid_knn_k32_on_a_million_point_segment_matches_all_pairs():
    """k = 32 over a single 10^6-point segment: the uniform-grid search against this package's exact all-pairs kernel
    (10^12 candidate pairs), indices and distances bit for bit."""
    from repsurf_b200 import _native as N
    from repsurf_b200.seg import pointops as P
    n, k = 1_000_000, 32
    xyz = _room(n, 0).to(cuda)
    off = torch.tensor([n], dtype=torch.int32, device=cuda)
    idx, dist = P.knnquery(k, xyz, xyz, off, off)                       # grid path (n >= KNN_GRID_MIN_POINTS)
    idx2 = torch.empty_like(idx)
    dist2 = torch.empty_like(dist)
    N.call("rsb_knnquery_packed", 1, n, k, xyz, xyz, off, off, idx2, dist2, 1)
    assert torch.equal(idx, idx2) and torch.equal(dist, dist2)
    assert bool((idx[:, 0] == torch.arange(n, device=cuda, dtype=torch.int32)).float().mean() > 0.999)   # self first (d = 0)


def test_grid_knn_k32_matches_reference_cuda_on_one_large_segment():
    from repsurf_b200.seg import pointops as P
    from tests import refcuda as R
    from tests.reference_golden import Reference, sample_rows
    REF = Reference("reference_cuda")
    n, k = 200_000, 32
    xyz = _room(n, 1).to(cuda)
    off = torch.tensor([n], dtype=torch.int32, device=cuda)
    idx, dist = P.knnquery(k, xyz, xyz, off, off)
    REF.equal("knn_packed_scene.idx", idx, lambda: R.knn_packed(k, xyz, xyz, off, off)[0])
    rows = torch.from_numpy(sample_rows(n, 512)).to(cuda)
    rd2 = torch.from_numpy(REF.array("knn_packed_scene.dist2_rows", lambda: R.knn_packed(k, xyz, xyz, off, off)[1][rows])).to(cuda)
    assert torch.equal(dist[rows], torch.sqrt(rd2)) or float((dist[rows] - torch.sqrt(rd2)).abs().max()) < 1e-6


def test_median_filter_matches_torch_median():
    from repsurf_b200.seg import scene as S
    from repsurf_b200.seg import pointops as P
    n, k = 300_000, 32
    xyz = _room(n, 2).to(cuda)
    g = torch.Generator().manual_seed(3)
    label = torch.randint(0, 13, (n,), generator=g, dtype=torch.int32).to(cuda)
    got = S.pc_median_filter_gpu(xyz, label, k)
    off = torch.tensor([n], dtype=torch.int32, device=cuda)
    idx, _ = P.knnquery(k, xyz, xyz, off, off)
    want = torch.median(label[idx.view(-1).long()].view(n, k), 1)[0].cpu().numpy()     # util/utils.py:242-244
    assert isinstance(got, np.ndarray) and np.array_equal(got, want)
    for kk in (1, 5, 16):                                                                # odd / even sizes
        idx, _ = P.knnquery(kk, xyz, xyz, off, off)
        want = torch.median(label[idx.view(-1).long()].view(n, kk), 1)[0]
        assert torch.equal(S.label_median(xyz, label, kk), want)


def test_vote_accumulation_and_decision():
    from repsurf_b200.seg import scene as S
    g = torch.Generator().manual_seed(4)
    n, nc = 50_000, 13
    votes = S.SceneVotes(n, nc, cuda)
    pred = torch.zeros(n, nc, dtype=torch.float64)
    cnt = torch.zeros(n, dtype=torch.float64)
    for _ in range(3):
        rows = 30_000
        idx = torch.randperm(n, generator=g)[:rows]                    # unique inside a crop batch, as in the reference loop
        buf = torch.randn(rows, 16, generator=g).to(cuda)              # row-padded logits (pitch 16), like the classifier head
        logits = buf[:, :nc]
        votes.add(logits, idx)
        pred[idx] += torch.softmax(logits.cpu().double(), 1)
        cnt[idx] += 1
    assert torch.allclose(votes.pred.cpu().double(), pred, rtol=1e-5, atol=1e-6) and torch.equal(votes.count.cpu().double(), cnt)
    seen = cnt > 0
    got = votes.decide().cpu()
    want = torch.argmax(votes.pred.cpu() / votes.count.cpu()[:, None], 1)
    assert torch.equal(got[seen].long(), want[seen])
    assert bool((got[~seen] == 0).all())                                # never-visited points: NaN rows -> class 0 (numpy.argmax)


def test_scene_inference_loop_runs_eval_model_on_crops():
    from repsurf_b200.models import RepSurfSeg
    from repsurf_b200.seg import scene as S
    from oracle.model_ref import det_fill_
    n = 60_000
    xyz = _room(n, 5)
    g = torch.Generator().manual_seed(6)
    feat = torch.rand(n, 3, generator=g)
    model = det_fill_(RepSurfSeg()).to(cuda)
    crops = []
    for c in range(4):                                                  # nearest-crops of 20 000 points around 4 seeds
        d = ((xyz - xyz[torch.randint(0, n, (1,), generator=g)]) ** 2).sum(1)
        crops.append(torch.argsort(d)[:20_000])
    coords = [(xyz[i] - xyz[i].mean(0)).contiguous() for i in crops]
    feats = [feat[i].contiguous() for i in crops]
    np.random.seed(0)
    lab = S.scene_inference(model, coords, feats, crops, n, 13, batch_size=2, filter_k=32, coord_all=xyz)
    assert lab.shape == (n,) and lab.dtype == torch.int32 and int(lab.min()) >= 0 and int(lab.max()) < 13
    # a second pass reproduces the labels (eval mode: no batch statistics, no dropout; the umbrella flip is seeded)
    np.random.seed(0)
    assert torch.equal(S.scene_inference(model, coords, feats, crops, n, 13, batch_size=2, filter_k=32, coord_all=xyz), lab)


def test_argmin_f64_is_numpy_argmin():
    """first occurrence among equal minima, negative and positive values"""
    from repsurf_b200 import _native as N
    r = np.random.RandomState(0)
    for n, dup in ((1, False), (77, True), (100_003, True), (1_000_000, False)):
        v = r.randn(n) if n != 77 else np.abs(r.randn(n))
        if dup:
            v[[n // 3, n // 2, n - 1]] = v.min() - 1.0              # three equal minima: the first one wins
        work = torch.empty(2, dtype=torch.int64, device=cuda)
        N.call("rsb_argmin_f64", n, torch.from_numpy(v).to(cuda), work)
        assert int(work[1]) == int(np.argmin(v))


def test_scene_parts_and_crop_plan_match_restatement():
    """data_load / data_process of segmentation/tool/test_s3dis.py:114-159 on the device against the numpy restatement (which
    tests/test_datapath.py pins to the unmodified reference functions): same parts, same crops in the same order, same rows."""
    from oracle import datapath_ref as D
    from repsurf_b200.seg import scene as S
    n = 150_000
    xyz = _room(n, 11)
    xyz = (xyz * torch.tensor([0.2, 0.2, 1.0])).contiguous()               # 6 x 4 x 3 m: several points per 4 cm voxel
    feat = (torch.rand(n, 3, generator=torch.Generator().manual_seed(12)) * 255).contiguous()
    c_np, f_np = xyz.numpy(), feat.numpy()
    parts = S.scene_parts(xyz.to(cuda), 0.04)
    want_parts = D.scene_parts(c_np, 0.04)
    assert len(parts) == len(want_parts) >= 2
    for a, b in zip(parts, want_parts):
        assert np.array_equal(a.cpu().numpy(), b)
    np.random.seed(21)
    gi, gc, gf, go = S.data_process(xyz.to(cuda), feat.to(cuda), parts, 20_000)
    np.random.seed(21)
    wi, wc, wf, wo = D.data_process(c_np, f_np, want_parts, 20_000)
    assert go == wo and len(gi) == len(wi) > len(parts) and max(go) == 20_000
    for a, b in zip(gi, wi):
        assert np.array_equal(a.cpu().numpy(), b)                           # scene rows of every crop, in order
    for a, b in zip(gf, wf):
        assert np.array_equal(a.cpu().numpy(), (b).astype(np.float32))
    for a, b in zip(gc, wc):
        assert np.abs(a.cpu().numpy() - b).max() < 5e-5                     # centring: fp64 mean here, fp32 running sum in numpy
    covered = torch.zeros(n, dtype=torch.bool)
    covered[torch.cat([i.cpu() for i in gi])] = True
    assert bool(covered.all())                                              # every scene point receives at least one vote


def test_infer_scene_end_to_end_covers_every_point():
    """parts -> covering crops -> batched eval forward -> votes -> decision -> median filter, one call; every point is voted
    for (no NaN row reaches the decision) and a seeded rerun reproduces the labels (up to vote-order ties)"""
    from repsurf_b200.models import RepSurfSeg
    from repsurf_b200.seg import scene as S
    from oracle.model_ref import det_fill_
    n = 90_000
    xyz = (_room(n, 15) * torch.tensor([0.2, 0.2, 1.0])).contiguous()
    feat = (torch.rand(n, 3, generator=torch.Generator().manual_seed(16)) * 255).contiguous()
    model = det_fill_(RepSurfSeg()).to(cuda)
    np.random.seed(2)
    lab = S.infer_scene(model, xyz, feat, 13, voxel_size=0.04, voxel_max=24_000, batch_size=3, filter_k=32)
    assert lab.shape == (n,) and lab.dtype == torch.int32 and int(lab.min()) >= 0 and int(lab.max()) < 13
    np.random.seed(2)
    votes_before = S.SceneVotes                                           # the vote counts of a second pass: all >= 1
    counts = {}

    class Probe(votes_before):
        def decide(self):
            counts["min"] = float(self.count.min())
            return super().decide()
    S.SceneVotes = Probe
    try:
        again = S.infer_scene(model, xyz, feat, 13, voxel_size=0.04, voxel_max=24_000, batch_size=3, filter_k=32)
    finally:
        S.SceneVotes = votes_before
    assert counts["min"] >= 1.0
    # votes of one batch are accumulated with float atomics: three or more crops of a batch that share a point may add up in a
    # different order, so a class tie at the last ulp may fall the other way
    assert float((again == lab).float().mean()) > 0.999


@pytest.mark.parametrize("rows,nc,ignore", [(50_000, 13, None), (4097, 13, 255), (1000, 20, 3)])
def test_cross_entropy_matches_torch(rows, nc, ignore):
    """seg/loss.CrossEntropyLoss (one kernel: value + gradient) against nn.CrossEntropyLoss in fp64, on the row-padded logits
    view the classifier head produces, with ignored rows."""
    import torch.nn as nn
    from repsurf_b200.seg.loss import CrossEntropyLoss
    g = torch.Generator().manual_seed(rows)
    buf = (torch.randn(rows, (nc + 3) // 4 * 4, generator=g) * 3).to(cuda)
    target = torch.randint(0, nc, (rows,), generator=g).to(cuda)
    if ignore is not None:
        target[torch.rand(rows, generator=g).to(cuda) < 0.2] = ignore
    a = buf.clone().requires_grad_(True)
    b = buf[:, :nc].double().detach().requires_grad_(True)
    kw = {} if ignore is None else {"ignore_index": ignore}
    la = CrossEntropyLoss(**kw)(a[:, :nc], target)
    lb = nn.CrossEntropyLoss(**kw)(b, target)
    assert abs(float(la) - float(lb)) < 1e-5 * max(1.0, abs(float(lb)))
    (la * 1.7).backward()
    (lb * 1.7).backward()
    assert float(a.grad[:, nc:].abs().sum()) == 0.0
    assert float((a.grad[:, :nc].double() - b.grad).abs().max()) < 1e-6 * float(b.grad.abs().max()) + 1e-12
