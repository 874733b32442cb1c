"""GPU parity suite (-m gpu): every CUDA operator, called through the C-ABI, against the CPU oracle on the same
seeded inputs (bit-exact for indices), against the recorded outputs of the reference's own CUDA kernels,
and size-independent properties at the full BASELINE sizes."""
import math
import os

import numpy as np
import pytest
import torch

from oracle import oracle as O

pytestmark = pytest.mark.gpu

cuda = torch.device("cuda")


def _cls():
    from repsurf_b200.cls import pointops as P
    return P


def _seg():
    from repsurf_b200.seg import pointops as P
    return P


def _ulp_equal(a, b, ulps=1):
    """distances that went through sqrt: torch's CUDA sqrt and the CPU's differ by <= 1 ulp on some inputs"""
    a, b = a.detach().cpu().contiguous(), b.detach().cpu().contiguous()
    ia, ib = a.view(torch.int32).long(), b.view(torch.int32).long()
    return bool(((ia - ib).abs() <= ulps).all())


def _cloud(b, n, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(b, n, 3, generator=g) * 2 - 1) * scale


# ------------------------------------------------------------------------------------------- FPS (dense)
@pytest.mark.parametrize("b,n,m", [(1, 128, 32), (4, 1024, 512), (3, 512, 128), (2, 1000, 333), (1, 40960, 1024),
                                   (2, 5000, 700), (1, 20000, 500), (1, 100000, 300), (3, 7, 5), (1, 1, 1), (2, 300, 300)])
def test_fps_dense_matches_oracle(b, n, m):
    xyz = _cloud(b, n, 100 + n)
    want = O.fps_dense(xyz, m)
    got = _cls().furthestsampling(xyz.to(cuda), m).cpu()
    assert torch.equal(got, want)


def test_fps_dense_ties_and_duplicates():
    # duplicated points and exact ties exercise the bit-reversed-thread tie rule (R2)
    g = torch.Generator().manual_seed(5)
    base = torch.randint(-3, 4, (2, 700, 3), generator=g).float() * 0.25      # lattice => many exact ties
    want = O.fps_dense(base, 400)
    got = _cls().furthestsampling(base.to(cuda), 400).cpu()
    assert torch.equal(got, want)
    zeros = torch.zeros(1, 64, 3)
    assert torch.equal(_cls().furthestsampling(zeros.to(cuda), 16).cpu(), O.fps_dense(zeros, 16))


def test_fps_dense_fused_xyz_and_known_answer(golden_dir):
    xyz = torch.from_numpy(np.load(os.path.join(golden_dir, "airplane_xyz_4096.npy")))[None].contiguous()
    idx, new_xyz = _cls().furthestsampling_with_xyz(xyz.to(cuda), 512)
    assert torch.equal(idx.cpu(), O.fps_dense(xyz, 512))
    assert torch.equal(new_xyz.cpu(), xyz[0][idx.cpu()[0].long()][None])


@pytest.mark.parametrize("plan", ["1,64", "1,256", "1,1024", "2,128", "4,256", "8,512", "16,128"])
def test_fps_all_cluster_shapes(plan, monkeypatch):
    monkeypatch.setenv("RSB_FPS_PLAN", plan)
    xyz = _cloud(3, 2048, 77)
    assert torch.equal(_cls().furthestsampling(xyz.to(cuda), 256).cpu(), O.fps_dense(xyz, 256))


# ------------------------------------------------------------------------------------------- FPS (packed)
def _packed(sizes, seed):
    g = torch.Generator().manual_seed(seed)
    xyz = torch.rand(sum(sizes), 3, generator=g) * torch.tensor([8.0, 8.0, 3.0])
    off = torch.tensor(np.cumsum(sizes), dtype=torch.int32)
    return xyz, off


@pytest.mark.parametrize("sizes,stride", [((1000, 500, 2047), 4), ((40960,), 16), ((10240, 10240, 300), 4), ((5, 9), 2),
                                          # a segment beyond the register-resident capacity (16 CTAs x 512 threads x 16 points):
                                          # the streaming plan with the caller's scratch buffer (whole-scene sizes)
                                          ((150000, 3000), 250), ((131072 - 1024, 200), 128), ((131073, 1077), 512)])
def test_fps_packed_matches_oracle(sizes, stride):
    xyz, off = _packed(sizes, 3)
    noff = torch.tensor(np.cumsum([s // stride for s in sizes]), dtype=torch.int32)
    want = O.fps_packed(xyz, off, noff)
    got = _seg().furthestsampling(xyz.to(cuda), off.to(cuda), noff.to(cuda)).cpu()
    assert torch.equal(got, want)


def _edge_safe(xyz, off, num_sectors, min_points=10000, margin=1e-4):
    """Nudge (rotate about z) every point whose azimuth lies within `margin` of an inner sector edge, so that the
    sector membership cannot depend on a last-ulp difference between the CPU and CUDA atan2 / linspace."""
    xyz = xyz.clone()
    for _ in range(8):
        bad_total, start = 0, 0
        for end in off.tolist():
            pts = xyz[start:end]
            if end - start >= min_points:
                ang = torch.atan2(pts[:, 0], pts[:, 1])
                edges = torch.linspace(float(ang.min()), float(ang.max()) + 1e-4, num_sectors + 1)[1:-1]
                bad = ((ang[:, None] - edges[None, :]).abs() < margin).any(1)
                # never move the two extreme points (they define the edges)
                bad[ang.argmin()] = False
                bad[ang.argmax()] = False
                if bad.any():
                    c, s_ = math.cos(3e-4), math.sin(3e-4)
                    x, y = pts[bad, 0].clone(), pts[bad, 1].clone()
                    pts[bad, 0], pts[bad, 1] = c * x - s_ * y, s_ * x + c * y
                    bad_total += int(bad.sum())
            start = end
        if bad_total == 0:
            return xyz
    raise AssertionError("could not move the points off the sector edges")


@pytest.mark.parametrize("skew", [False, True])
def test_sectorized_fps_matches_oracle(skew):
    """skew: 70 % of the first cloud sits in one sector, so its largest sector exceeds the 1.1x-mean capacity of the
    first launch and goes through the follow-up launch of rsb_furthestsampling_packed_bounded."""
    xyz, off = _packed((12000, 3000, 10500), 8)
    xyz = xyz - xyz.mean(0)
    if skew:
        g = torch.Generator().manual_seed(11)
        phi = torch.rand(8400, generator=g) * 1.2 + 0.1             # azimuth atan2(x, y) in a 1.2 rad wedge
        r = torch.rand(8400, generator=g) * 4 + 0.5
        xyz[:8400, 0], xyz[:8400, 1] = r * torch.sin(phi), r * torch.cos(phi)
    xyz = _edge_safe(xyz, off, 4)
    noff = torch.tensor(np.cumsum([3000, 750, 2625]), dtype=torch.int32)
    want = O.sectorized_fps(xyz, off, noff, 4)
    got = _seg().sectorized_fps(xyz.to(cuda), off.to(cuda), noff.to(cuda), 4).cpu()
    assert got.dtype == torch.int64
    assert torch.equal(got, want)


def test_sectorized_fps_small_clouds_use_device_maximum():
    """clouds below min_points are single sectors; with every cloud under 1024 points the reference's block size
    (tie rule) follows the largest one, which only the device knows when sizes come from the sector split."""
    xyz, off = _packed((700, 300, 900), 5)
    noff = torch.tensor(np.cumsum([175, 75, 225]), dtype=torch.int32)
    want = O.sectorized_fps(xyz, off, noff, 4)
    got = _seg().sectorized_fps(xyz.to(cuda), off.to(cuda), noff.to(cuda), 4).cpu()
    assert torch.equal(got, want)


# ------------------------------------------------------------------------------------------- ball query
@pytest.mark.parametrize("b,n,m,r,ns", [(2, 1024, 512, 0.2, 32), (2, 512, 128, 0.4, 64), (1, 4096, 300, 0.1, 16),
                                        (1, 33, 7, 0.5, 8), (1, 2000, 64, 0.05, 32)])
def test_ballquery_matches_oracle(b, n, m, r, ns):
    xyz = _cloud(b, n, 200 + n)
    q = xyz[:, torch.randperm(n, generator=torch.Generator().manual_seed(1))[:m]].contiguous()
    want = O.ballquery(r, ns, xyz, q)
    got = _cls().ballquery(r, ns, xyz.to(cuda), q.to(cuda)).cpu()
    assert torch.equal(got, want)


def test_ballquery_empty_balls_are_zero():
    xyz = _cloud(1, 256, 9)
    q = torch.full((1, 5, 3), 50.0)
    assert int(_cls().ballquery(0.2, 16, xyz.to(cuda), q.to(cuda)).abs().sum()) == 0


# ------------------------------------------------------------------------------------------- kNN
@pytest.mark.parametrize("b,n,m,k", [(2, 1024, 1024, 9), (1, 3000, 500, 32), (1, 700, 700, 3), (2, 100, 37, 64),
                                     (1, 500, 100, 100), (1, 400, 50, 200), (1, 5, 5, 9)])
def test_knn_dense_matches_oracle(b, n, m, k):
    xyz = _cloud(b, n, 300 + n)
    q = xyz[:, :m].contiguous()
    want = O.knn_dense(k, xyz, q)
    got = _cls().knnquery(k, xyz.to(cuda), q.to(cuda)).cpu()
    assert torch.equal(got, want)


def test_knn_dense_lattice_ties_are_stable():
    g = torch.Generator().manual_seed(6)
    xyz = torch.randint(-4, 5, (1, 600, 3), generator=g).float() * 0.5
    want = O.knn_dense(16, xyz, xyz)
    got = _cls().knnquery(16, xyz.to(cuda), xyz.to(cuda)).cpu()
    assert torch.equal(got, want)


@pytest.mark.parametrize("b,n,m,k", [(2, 1024, 256, 16), (1, 300, 300, 100), (1, 50, 10, 64)])
def test_knn_heap_dense_matches_oracle(b, n, m, k):
    xyz = _cloud(b, n, 400 + n)
    q = xyz[:, :m].contiguous()
    want = O.knn_heap_dense(k, xyz, q)
    got = _cls().knnquery_heap(k, xyz.to(cuda), q.to(cuda)).cpu()
    assert torch.equal(got, want)


def test_knn_heap_lattice_ties_replay_exactly():
    g = torch.Generator().manual_seed(7)
    xyz = torch.randint(-3, 4, (1, 500, 3), generator=g).float() * 0.5
    want = O.knn_heap_dense(12, xyz, xyz)
    got = _cls().knnquery_heap(12, xyz.to(cuda), xyz.to(cuda)).cpu()
    assert torch.equal(got, want)


@pytest.mark.parametrize("sizes,msizes,k", [((3000, 1000, 4500), None, 9), ((2048, 2048), (512, 512), 32),
                                            ((700, 20, 1300), (700, 20, 1300), 3), ((40,), (40,), 32)])
def test_knn_packed_matches_oracle(sizes, msizes, k):
    xyz, off = _packed(sizes, 11)
    if msizes is None:
        q, noff = xyz, off
    else:
        parts, start = [], 0
        for s, ms in zip(sizes, msizes):
            parts.append(xyz[start:start + ms])
            start += s
        q = torch.cat(parts).contiguous()
        noff = torch.tensor(np.cumsum(msizes), dtype=torch.int32)
    widx, wdist = O.knn_packed(k, xyz, q, off, noff)
    gidx, gdist = _seg().knnquery(k, xyz.to(cuda), q.to(cuda), off.to(cuda), noff.to(cuda))
    assert torch.equal(gidx.cpu(), widx)
    assert _ulp_equal(gdist, wdist)


def test_knn_packed_lattice_ties_replay_exactly():
    g = torch.Generator().manual_seed(8)
    xyz = torch.randint(-3, 4, (900, 3), generator=g).float() * 0.5
    off = torch.tensor([400, 900], dtype=torch.int32)
    widx, _ = O.knn_packed(9, xyz, xyz, off, off)
    gidx, _ = _seg().knnquery(9, xyz.to(cuda), xyz.to(cuda), off.to(cuda), off.to(cuda))
    assert torch.equal(gidx.cpu(), widx)


def test_nearestneighbor_matches_oracle():
    unk, kn = _cloud(2, 900, 21), _cloud(2, 250, 22)
    wd2, widx = O.nn3(unk, kn)
    gdist, gidx = _cls().nearestneighbor(unk.to(cuda), kn.to(cuda))
    assert torch.equal(gidx.cpu(), widx)
    assert _ulp_equal(gdist, torch.sqrt(wd2))


# ------------------------------------------------------------------------------------------- gathers
def test_dense_gather_group_interp_fwd_bwd():
    P = _cls()
    g = torch.Generator().manual_seed(30)
    f = torch.randn(3, 13, 257, generator=g)
    idx1 = torch.randint(0, 257, (3, 50), generator=g).int()
    idx2 = torch.randint(0, 257, (3, 50, 7), generator=g).int()
    fc = f.to(cuda).requires_grad_(True)
    out1 = P.gathering(fc, idx1.to(cuda))
    assert torch.equal(out1.detach().cpu(), O.gather_fwd(f, idx1))
    go1 = torch.randn(out1.shape, generator=g)
    out1.backward(go1.to(cuda))
    assert torch.allclose(fc.grad.cpu(), O.gather_bwd(go1, idx1, 257), rtol=1e-5, atol=1e-5)
    fc.grad = None
    out2 = P.grouping(fc, idx2.to(cuda))
    assert torch.equal(out2.detach().cpu(), O.group_fwd(f, idx2))
    go2 = torch.randn(out2.shape, generator=g)
    out2.backward(go2.to(cuda))
    assert torch.allclose(fc.grad.cpu(), O.group_bwd(go2, idx2, 257), rtol=1e-5, atol=1e-5)
    fc.grad = None
    idx3 = torch.randint(0, 257, (3, 80, 3), generator=g).int()
    w = torch.rand(3, 80, 3, generator=g)
    out3 = P.interpolation(fc, idx3.to(cuda), w.to(cuda))
    assert torch.equal(out3.detach().cpu(), O.interp_fwd(f, idx3, w))
    go3 = torch.randn(out3.shape, generator=g)
    out3.backward(go3.to(cuda))
    assert torch.allclose(fc.grad.cpu(), O.interp_bwd(go3, idx3, w, 257), rtol=1e-5, atol=1e-5)
    li = torch.randint(0, 1 << 40, (2, 3, 100), generator=g)
    ii = torch.randint(0, 100, (2, 9, 4), generator=g).int()
    got = P.grouping_int(li.to(cuda), ii.to(cuda)).cpu()
    assert torch.equal(got, torch.gather(li[:, :, None].expand(-1, -1, 9, -1), 3, ii.long()[:, None].expand(-1, 3, -1, -1)))


@pytest.mark.parametrize("c", [3, 10, 16, 77])
def test_packed_group_interp_fwd_bwd(c):
    P = _seg()
    g = torch.Generator().manual_seed(31 + c)
    f = torch.randn(500, c, generator=g)
    idx = torch.randint(0, 500, (123, 9), generator=g).int()
    fc = f.to(cuda).requires_grad_(True)
    out = P.grouping(fc, idx.to(cuda))
    assert torch.equal(out.detach().cpu(), O.group_packed_fwd(f, idx))
    go = torch.randn(out.shape, generator=g)
    out.backward(go.to(cuda))
    assert torch.allclose(fc.grad.cpu(), O.group_packed_bwd(go, idx, 500), rtol=1e-5, atol=1e-5)
    fc.grad = None
    idx3 = torch.randint(0, 500, (321, 3), generator=g).int()
    w = torch.rand(321, 3, generator=g)
    out3 = P._InterpApply.apply(fc, idx3.to(cuda), w.to(cuda))
    assert torch.equal(out3.detach().cpu(), O.interp_packed_fwd(f, idx3, w))
    go3 = torch.randn(out3.shape, generator=g)
    out3.backward(go3.to(cuda))
    assert torch.allclose(fc.grad.cpu(), O.interp_packed_bwd(go3, idx3, w, 500), rtol=1e-5, atol=1e-5)


# ------------------------------------------------------------------------------------------- full-size properties
def test_full_size_properties_s3dis_shape():
    """BASELINE config 3 sizes (8 x 40960): properties that need no oracle run."""
    P = _seg()
    B, N = 8, 40960
    g = torch.Generator().manual_seed(99)
    xyz = (torch.rand(B * N, 3, generator=g) * torch.tensor([8.0, 8.0, 3.0])).to(cuda)
    off = P.make_offsets([N * (i + 1) for i in range(B)], cuda)
    noff = P.make_offsets([N // 4 * (i + 1) for i in range(B)], cuda)
    idx = P.furthestsampling(xyz, off, noff).long()
    # every pick lies in its own cloud, is unique, and the first pick is the segment start
    cloud = torch.arange(B, device=cuda).repeat_interleave(N // 4)
    assert torch.equal(idx // N, cloud)
    assert idx.unique().numel() == idx.numel()
    assert torch.equal(idx[:: N // 4], torch.arange(B, device=cuda) * N)
    # FPS is greedy: the running min-distance of successive picks never increases
    first = xyz[idx[:512]].double()
    d = ((first[:, None] - first[None]) ** 2).sum(-1)
    d = d + torch.triu(torch.full_like(d, 1e9))           # only earlier picks
    mins = d[1:].min(dim=1)[0]
    assert (mins[1:] <= mins[:-1] * (1 + 1e-5)).all()
    # kNN: self is the nearest neighbour, distances ascend, indices stay inside the cloud
    nidx, ndist = P.knnquery(9, xyz, xyz, off, off)
    assert torch.equal(nidx[:, 0].long(), torch.arange(B * N, device=cuda))
    assert (ndist[:, 1:] >= ndist[:, :-1]).all()
    assert torch.equal(nidx.long() // N, (torch.arange(B * N, device=cuda) // N)[:, None].expand(-1, 9))
    # against brute force on a slice
    sl = slice(N, N + 256)
    D = torch.cdist(xyz[sl].double(), xyz[N:2 * N].double())
    assert torch.equal(D.topk(9, largest=False)[1] + N, nidx[sl].long())


# ------------------------------------------------------------------------------------------- grid kNN == all-pairs kNN
@pytest.mark.parametrize("sizes,k", [((5000, 3000), 9), ((40960,), 32), ((3000, 9000, 2500), 3), ((2500, 2100), 64)])
def test_knn_grid_equals_allpairs(sizes, k, monkeypatch):
    P = _seg()
    xyz, off = _packed(sizes, 17)
    q = xyz[::3].contiguous()
    msizes = [len(range(a, b, 3)) for a, b in zip([0] + list(np.cumsum(sizes)[:-1]), np.cumsum(sizes))]
    # rows of q must stay grouped per cloud: rebuild per cloud
    parts, start = [], 0
    for sz in sizes:
        parts.append(xyz[start:start + sz][::3])
        start += sz
    q = torch.cat(parts).contiguous()
    noff = torch.tensor(np.cumsum([p.shape[0] for p in parts]), dtype=torch.int32)
    monkeypatch.setattr(P, "KNN_GRID_MIN_POINTS", None)
    bi, bd = P.knnquery(k, xyz.to(cuda), q.to(cuda), off.to(cuda), noff.to(cuda))
    monkeypatch.setattr(P, "KNN_GRID_MIN_POINTS", 1)
    gi, gd = P.knnquery(k, xyz.to(cuda), q.to(cuda), off.to(cuda), noff.to(cuda))
    assert torch.equal(bi, gi) and torch.equal(bd, gd)


def test_knn_grid_lattice_and_degenerate_inputs(monkeypatch):
    P = _seg()
    monkeypatch.setattr(P, "KNN_GRID_MIN_POINTS", 1)
    g = torch.Generator().manual_seed(8)
    lat = torch.randint(-6, 7, (3000, 3), generator=g).float() * 0.5          # many exact ties -> replay path
    off = torch.tensor([1200, 3000], dtype=torch.int32)
    widx, wdist = O.knn_packed(9, lat, lat, off, off)
    gidx, gdist = P.knnquery(9, lat.to(cuda), lat.to(cuda), off.to(cuda), off.to(cuda))
    assert torch.equal(gidx.cpu(), widx) and _ulp_equal(gdist, wdist)
    flat = torch.rand(2000, 3, generator=g) * torch.tensor([5.0, 5.0, 0.0])   # planar cloud (zero extent in z)
    off1 = torch.tensor([2000], dtype=torch.int32)
    widx, _ = O.knn_packed(16, flat, flat, off1, off1)
    gidx, _ = P.knnquery(16, flat.to(cuda), flat.to(cuda), off1.to(cuda), off1.to(cuda))
    assert torch.equal(gidx.cpu(), widx)
    few = torch.rand(5, 3, generator=g)                                        # fewer points than k
    off2 = torch.tensor([5], dtype=torch.int32)
    widx, _ = O.knn_packed(9, few, few, off2, off2)
    gidx, _ = P.knnquery(9, few.to(cuda), few.to(cuda), off2.to(cuda), off2.to(cuda))
    assert torch.equal(gidx.cpu(), widx)


# ------------------------------------------------------------------------------------------- fused umbrella geometry
@pytest.mark.parametrize("order,rotate,skip", [("seg", True, False), ("cls", False, True)])
def test_umbrella_kernel_matches_tensor_formulation(order, rotate, skip):
    """csrc/umbrella.cu vs oracle.geometry_ref.umbrella_features (a vectorised torch restatement, itself pinned to the
    unmodified reference's tensors by tests/test_oracle_cpu.py; the kernel is pinned to them directly in
    tests/test_models_gpu.py).  Points whose neighbour azimuths tie within an ulp may sort differently."""
    from repsurf_b200 import _native as N
    from oracle.geometry_ref import umbrella_features
    P = _seg()
    g = torch.Generator().manual_seed(41)
    n, k = 6000, 9
    xyz = (torch.rand(n, 3, generator=g) * torch.tensor([4.0, 4.0, 2.0])).to(cuda)
    off = torch.tensor([2500, 6000], dtype=torch.int32, device=cuda)
    idx, _ = P.knnquery(k, xyz, xyz, off, off)
    flip = (torch.randint(0, 2, (n,), generator=g).float() * 2 - 1).to(cuda)
    G = k - (1 if skip else 0)
    out = torch.empty(n, G, 10, device=cuda)
    N.call("rsb_umbrella_features", n, k, 1 if skip else 0, 1 if rotate else 0, 1 if order == "seg" else 0, xyz, idx, flip, out, 10, 10)
    nb = idx[:, 1:] if skip else idx
    offsets = xyz[nb.long()] - xyz[:, None]
    want = umbrella_features(offsets, flip.view(-1, 1, 1), rotate_key=rotate, order=order)
    err = (out - want).abs().amax(dim=(1, 2)) / want.abs().max()
    assert (err > 1e-5).float().mean().item() < 2e-3
    assert not torch.isnan(out).any() or torch.isnan(want).any()


# ------------------------------------------------------------------------------------------- fused row builder
@pytest.mark.parametrize("polar,cf", [(True, 0), (True, 64), (False, 32)])
def test_group_rows_matches_gather_composition(polar, cf):
    """csrc/group.cu group_rows_* vs the reference's composition (gathers, subtraction, xyz2sphere, cat:
    segmentation/modules/repsurface_utils.py:36-49): gathers and relative xyz bit-exact, polar columns to an ulp of
    the libdevice functions, backward scatter against an fp64 index_add."""
    from oracle.geometry_ref import xyz2sphere
    from repsurf_b200.mlp import group_rows
    g = torch.Generator().manual_seed(43)
    n, M, ns, cn = 5000, 700, 24, 10
    xyz = torch.rand(n, 3, generator=g).to(cuda)
    new_xyz = xyz[torch.randperm(n, generator=g)[:M].to(cuda)].contiguous()
    idx = torch.randint(0, n, (M, ns), generator=g, dtype=torch.int32).to(cuda)
    idx[:, 0] = torch.arange(M, device=cuda, dtype=torch.int32)          # some zero-length offsets (rho == 0)
    new_xyz[:] = xyz[:M]
    normal = torch.randn(n, cn, generator=g).to(cuda).requires_grad_()
    feat = torch.randn(n, cf, generator=g).to(cuda).requires_grad_() if cf else None
    rows, (P4, F) = group_rows(xyz, new_xyz, idx, normal, feat, ns, polar)
    rel = xyz[idx.long()] - new_xyz[:, None]
    pos = torch.cat([rel, xyz2sphere(rel)], -1) if polar else rel
    P = pos.shape[-1]
    rows3 = rows.view(M, ns, -1)
    assert torch.equal(rows3[..., :3], rel)
    if polar:
        err = (rows3[..., 3:P] - pos[..., 3:]).abs().amax(dim=(0, 1))
        assert (err < 2e-6).all(), err       # torch's CUDA sqrt is not the IEEE one (<= 1 ulp), acos amplifies it
    assert (rows3[..., P:P4] == 0).all() and F == cn + cf
    assert torch.equal(rows3[..., P4:P4 + cn], normal[idx.long()])
    if cf:
        assert torch.equal(rows3[..., P4 + cn:P4 + F], feat[idx.long()])
    assert (rows3[..., P4 + F:] == 0).all()
    w = torch.randn(rows.shape, generator=torch.Generator().manual_seed(1)).to(cuda)
    (rows * w).sum().backward()
    w3 = w.view(M, ns, -1).double()
    want = torch.zeros(n, cn, dtype=torch.float64, device=cuda).index_add_(0, idx.view(-1).long(), w3[..., P4:P4 + cn].reshape(-1, cn))
    assert torch.allclose(normal.grad.double(), want, rtol=1e-5, atol=1e-5)
    if cf:
        want = torch.zeros(n, cf, dtype=torch.float64, device=cuda).index_add_(0, idx.view(-1).long(), w3[..., P4 + cn:P4 + F].reshape(-1, cf))
        assert torch.allclose(feat.grad.double(), want, rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("k", [9, 32])
def test_dense_knn_large_clouds_grid_route_matches_allpairs_and_reference(k):
    """Dense API (cls) on clouds above the grid threshold: the grid route == this package's all-pairs kernels ==
    the reference's CUDA kernels (insertion-order and heap-order semantics), bit for bit."""
    from repsurf_b200 import _native as N
    from repsurf_b200.cls import pointops as P
    from tests import refcuda as R
    from tests.reference_golden import Reference
    g = torch.Generator().manual_seed(77 + k)
    b, n, m = 3, 6000, 1500
    xyz = torch.rand(b, n, 3, generator=g).to(cuda)
    new_xyz = xyz[:, :m].contiguous()
    assert n >= P.KNN_GRID_MIN_POINTS
    got = P.knnquery(k, xyz, new_xyz)
    ap = torch.empty_like(got)
    N.call("rsb_knnquery_dense", b, n, m, k, xyz, new_xyz, ap, None)
    assert torch.equal(got, ap)
    goth = P.knnquery_heap(k, xyz, new_xyz)
    aph = torch.empty_like(goth)
    d2 = torch.empty(b, m, k, device=cuda)
    N.call("rsb_knnquery_heap_dense", b, n, m, k, xyz, new_xyz, aph, d2)
    assert torch.equal(goth, aph)
    REF = Reference("reference_cuda")
    REF.equal(f"knn_dense_large[{k}]", got, lambda: R.knn_dense(k, xyz, new_xyz))
    REF.equal(f"knn_heap_dense_large[{k}]", goth, lambda: R.knn_heap_dense(k, xyz, new_xyz)[0])
