"""The REFERENCE's own CUDA kernels (compiled unmodified into oracle/_ref by oracle/build_ref.sh, their outputs recorded in
tests/golden/reference_cuda.*) versus (a) the CPU oracle — this is what pins the oracle's rounding / tie rules R1-R5 to the
real reference — and (b, GPU) the sm_100a kernels at sizes the CPU oracle would take too long for."""
import numpy as np
import pytest
import torch

from oracle import oracle as O
from tests import refcuda as R
from tests.reference_golden import Reference, sample_rows

REF = Reference("reference_cuda")
cuda = torch.device("cuda")


def _cloud(b, n, seed):
    return torch.rand(b, n, 3, generator=torch.Generator().manual_seed(seed)) * 2 - 1


def _lattice(b, n, seed, lo=-3, hi=4):
    return torch.randint(lo, hi, (b, n, 3), generator=torch.Generator().manual_seed(seed)).float() * 0.5


# ---- (a) oracle == reference CUDA -------------------------------------------------------------------------
@pytest.mark.parametrize("gen,b,n,m", [(_cloud, 3, 1024, 512), (_cloud, 2, 777, 300), (_lattice, 2, 640, 320),
                                       (_cloud, 1, 5000, 600), (_lattice, 1, 96, 50)])
def test_oracle_fps_dense_equals_reference_cuda(gen, b, n, m):
    xyz = gen(b, n, 1 + n)
    REF.equal(f"fps_dense{gen.__name__}[{b},{n},{m}]", O.fps_dense(xyz, m), lambda: R.fps_dense(xyz.to(cuda), m))


def test_oracle_fps_packed_equals_reference_cuda():
    sizes = (900, 3000, 411)
    off = torch.tensor(np.cumsum(sizes), dtype=torch.int32)
    noff = torch.tensor(np.cumsum([s // 4 for s in sizes]), dtype=torch.int32)
    for gen, seed in ((_cloud, 3), (_lattice, 4)):
        xyz = gen(1, sum(sizes), seed)[0].contiguous()
        REF.equal(f"fps_packed{gen.__name__}", O.fps_packed(xyz, off, noff),
                  lambda: R.fps_packed(xyz.to(cuda), off.to(cuda), noff.to(cuda)))


def test_oracle_ballquery_equals_reference_cuda():
    xyz = _cloud(2, 1024, 5)
    q = xyz[:, :300].contiguous()
    for r, ns in ((0.2, 32), (0.4, 64), (0.05, 8)):
        REF.equal(f"ballquery[{r},{ns}]", O.ballquery(r, ns, xyz, q), lambda: R.ballquery(r, ns, xyz.to(cuda), q.to(cuda)))


def test_oracle_knn_equals_reference_cuda():
    for gen in (_cloud, _lattice):
        xyz = gen(2, 800, 6)
        q = xyz[:, :200].contiguous()
        g = gen.__name__
        REF.equal(f"knn_dense{g}", O.knn_dense(9, xyz, q), lambda: R.knn_dense(9, xyz.to(cuda), q.to(cuda)))
        widx, wd2 = O.knn_heap_dense(16, xyz, q, return_dist2=True)
        REF.equal(f"knn_heap_dense{g}.idx", widx, lambda: R.knn_heap_dense(16, xyz.to(cuda), q.to(cuda))[0])
        REF.equal(f"knn_heap_dense{g}.dist2", wd2, lambda: R.knn_heap_dense(16, xyz.to(cuda), q.to(cuda))[1])
        wd, wi = O.nn3(q, xyz)
        REF.equal(f"nn3{g}.idx", wi, lambda: R.nn3(q.to(cuda), xyz.to(cuda))[1])
        REF.equal(f"nn3{g}.dist2", wd, lambda: R.nn3(q.to(cuda), xyz.to(cuda))[0])


def test_oracle_knn_packed_equals_reference_cuda():
    sizes = (1500, 700)
    for gen in (_cloud, _lattice):
        xyz = gen(1, sum(sizes), 7)[0].contiguous()
        off = torch.tensor(np.cumsum(sizes), dtype=torch.int32)
        widx, wd2 = O.knn_packed(12, xyz, xyz, off, off, sqrt=False)
        ref = lambda: R.knn_packed(12, xyz.to(cuda), xyz.to(cuda), off.to(cuda), off.to(cuda))
        REF.equal(f"knn_packed{gen.__name__}.idx", widx, lambda: ref()[0])
        REF.equal(f"knn_packed{gen.__name__}.dist2", wd2, lambda: ref()[1])


# ---- (b) sm_100a kernels == reference CUDA at full size -----------------------------------------------------
@pytest.mark.gpu
def test_fps_full_size_equals_reference_cuda():
    from repsurf_b200.seg import pointops as P
    B, N = 4, 40960
    xyz = (torch.rand(B * N, 3, generator=torch.Generator().manual_seed(8)) * torch.tensor([8.0, 8.0, 3.0])).to(cuda)
    off = P.make_offsets([N * (i + 1) for i in range(B)], cuda)
    noff = P.make_offsets([N // 4 * (i + 1) for i in range(B)], cuda)
    REF.equal("fps_packed_full", P.furthestsampling(xyz, off, noff), lambda: R.fps_packed(xyz, off, noff))


@pytest.mark.gpu
def test_knn_full_size_equals_reference_cuda():
    from repsurf_b200.seg import pointops as P
    B, N = 2, 40960
    xyz = (torch.rand(B * N, 3, generator=torch.Generator().manual_seed(9)) * torch.tensor([8.0, 8.0, 3.0])).to(cuda)
    off = P.make_offsets([N * (i + 1) for i in range(B)], cuda)
    rows = torch.from_numpy(sample_rows(B * N, 512)).to(cuda)
    for k in (9, 32):
        gidx, gdist = P.knnquery(k, xyz, xyz, off, off)
        REF.equal(f"knn_packed_full[{k}].idx", gidx, lambda: R.knn_packed(k, xyz, xyz, off, off)[0])
        rd2 = torch.from_numpy(REF.array(f"knn_packed_full[{k}].dist2_rows", lambda: R.knn_packed(k, xyz, xyz, off, off)[1][rows])).to(cuda)
        assert ((gdist[rows].view(torch.int32).long() - torch.sqrt(rd2).view(torch.int32).long()).abs() <= 1).all()


@pytest.mark.gpu
def test_cls_ops_full_size_equal_reference_cuda():
    from repsurf_b200.cls import pointops as P
    xyz = _cloud(32, 1024, 10).to(cuda)
    fidx = P.furthestsampling(xyz, 512)
    REF.equal("fps_dense_full", fidx, lambda: R.fps_dense(xyz, 512))
    q = torch.gather(xyz, 1, fidx.long()[..., None].expand(-1, -1, 3)).contiguous()
    REF.equal("ballquery_full", P.ballquery(0.2, 32, xyz, q), lambda: R.ballquery(0.2, 32, xyz, q))
    REF.equal("knn_dense_full", P.knnquery(9, xyz, xyz), lambda: R.knn_dense(9, xyz, xyz))
