"""subtraction / aggregation (the PointTransformer operators of the shared pointops package, SURVEY.md 8 f4): the C oracle on
the CPU against plain tensor formulas; the sm_100a kernels against the oracle and against the recorded outputs of the reference's own CUDA kernels."""
import numpy as np
import pytest
import torch

from oracle import oracle as O


def _case(n, ns, c, w_c, seed):
    g = torch.Generator().manual_seed(seed)
    inp = torch.randn(n, c, generator=g)
    in2 = torch.randn(n, c, generator=g)
    pos = torch.randn(n, ns, c, generator=g)
    w = torch.randn(n, ns, w_c, generator=g)
    idx = torch.randint(0, n, (n, ns), generator=g, dtype=torch.int32)
    go3 = torch.randn(n, ns, c, generator=g)
    go2 = torch.randn(n, c, generator=g)
    return inp, in2, pos, w, idx, go3, go2


CASES = [(500, 16, 32, 4, 0), (777, 8, 48, 6, 1), (64, 5, 7, 7, 2), (2000, 16, 64, 8, 3)]


@pytest.mark.parametrize("n,ns,c,w_c,seed", CASES)
def test_oracle_matches_tensor_formulas(n, ns, c, w_c, seed):
    inp, in2, pos, w, idx, go3, go2 = _case(n, ns, c, w_c, seed)
    li = idx.long()
    assert torch.equal(O.subtraction_fwd(inp, in2, idx), inp[:, None, :] - in2[li])
    g1, g2 = O.subtraction_bwd(go3, idx)
    assert torch.allclose(g1, go3.sum(1), rtol=1e-5, atol=1e-5)
    want2 = torch.zeros(n, c).index_add_(0, li.reshape(-1), -go3.reshape(-1, c))
    assert torch.allclose(g2, want2, rtol=1e-5, atol=1e-5)
    wfull = w.repeat(1, 1, c // w_c) if c % w_c == 0 else torch.stack([w[..., ch % w_c] for ch in range(c)], -1)
    want = ((inp[li] + pos).double() * wfull.double()).sum(1)
    assert torch.allclose(O.aggregation_fwd(inp, pos, w, idx).double(), want, rtol=1e-5, atol=1e-5)
    g_in, g_pos, g_w = O.aggregation_bwd(inp, pos, w, idx, go2)
    t = go2[:, None, :] * wfull
    assert torch.equal(g_pos, t)
    assert torch.allclose(g_in, torch.zeros(n, c).index_add_(0, li.reshape(-1), t.reshape(-1, c)), rtol=1e-5, atol=1e-5)
    gw_full = (go2[:, None, :] * (inp[li] + pos)).double()
    want_w = torch.zeros(n, ns, w_c, dtype=torch.float64)
    for ch in range(c):
        want_w[..., ch % w_c] += gw_full[..., ch]
    assert torch.allclose(g_w.double(), want_w, rtol=1e-5, atol=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("n,ns,c,w_c,seed", CASES + [(40960, 16, 64, 8, 4)])
def test_kernels_match_oracle_and_reference_cuda(n, ns, c, w_c, seed):
    from repsurf_b200.seg import pointops as P
    from tests import refcuda as R
    from tests.reference_golden import Reference, sample_rows
    REF = Reference("reference_cuda")
    case = f"[{n},{ns},{c},{w_c},{seed}]"
    cuda = torch.device("cuda")
    inp, in2, pos, w, idx, go3, go2 = [t.to(cuda) for t in _case(n, ns, c, w_c, seed)]
    small = n <= 2000
    rows = torch.from_numpy(sample_rows(n, 128)).to(cuda)        # reference gradients are kept for a sample of rows
    # ---- subtraction
    a = inp.clone().requires_grad_(True)
    b = in2.clone().requires_grad_(True)
    out = P.subtraction(a, b, idx)
    if small:
        assert torch.equal(out.cpu(), O.subtraction_fwd(inp.cpu(), in2.cpu(), idx.cpu()))            # bit-exact
    out.backward(go3)
    REF.equal("subtraction_fwd" + case, out, lambda: R.subtraction_fwd(inp, in2, idx))               # bit-exact vs reference CUDA
    r1 = REF.array("subtraction_bwd.grad1_rows" + case, lambda: R.subtraction_bwd(go3, idx)[0][rows])
    r2 = REF.array("subtraction_bwd.grad2_rows" + case, lambda: R.subtraction_bwd(go3, idx)[1][rows])
    assert torch.allclose(a.grad[rows].cpu(), torch.from_numpy(r1), rtol=1e-5, atol=1e-5)
    assert torch.allclose(b.grad[rows].cpu(), torch.from_numpy(r2), rtol=1e-5, atol=1e-5)
    if small:
        g1, g2 = O.subtraction_bwd(go3.cpu(), idx.cpu())
        assert torch.allclose(a.grad.cpu(), g1, rtol=1e-5, atol=1e-5) and torch.allclose(b.grad.cpu(), g2, rtol=1e-5, atol=1e-5)
    # ---- aggregation
    x = inp.clone().requires_grad_(True)
    p = pos.clone().requires_grad_(True)
    ww = w.clone().requires_grad_(True)
    out = P.aggregation(x, p, ww, idx)
    if small:
        assert torch.equal(out.cpu(), O.aggregation_fwd(inp.cpu(), pos.cpu(), w.cpu(), idx.cpu()))  # bit-exact (same fma chain)
    out.backward(go2)
    REF.equal("aggregation_fwd" + case, out, lambda: R.aggregation_fwd(inp, pos, w, idx))            # bit-exact vs reference CUDA
    REF.equal("aggregation_bwd.grad_pos" + case, p.grad, lambda: R.aggregation_bwd(inp, pos, w, idx, go2)[1])
    r_in = REF.array("aggregation_bwd.grad_in_rows" + case, lambda: R.aggregation_bwd(inp, pos, w, idx, go2)[0][rows])
    r_w = REF.array("aggregation_bwd.grad_w_rows" + case, lambda: R.aggregation_bwd(inp, pos, w, idx, go2)[2][rows])
    assert torch.allclose(x.grad[rows].cpu(), torch.from_numpy(r_in), rtol=1e-5, atol=1e-5)
    assert torch.allclose(ww.grad[rows].cpu(), torch.from_numpy(r_w), rtol=1e-4, atol=1e-4)
    if small:
        g_in, g_pos, g_w = O.aggregation_bwd(inp.cpu(), pos.cpu(), w.cpu(), idx.cpu(), go2.cpu())
        assert torch.equal(p.grad.cpu(), g_pos)
        assert torch.allclose(x.grad.cpu(), g_in, rtol=1e-5, atol=1e-5) and torch.allclose(ww.grad.cpu(), g_w, rtol=1e-4, atol=1e-4)


@pytest.mark.gpu
def test_queryandgroup_and_interpolation2_match_compositions():
    """The thin members of the packed API (pointops.py:165-186, :273-307) against their definitions."""
    from repsurf_b200.seg import pointops as P
    cuda = torch.device("cuda")
    g = torch.Generator().manual_seed(9)
    n, m, c, ns = 3000, 700, 20, 12
    xyz = torch.rand(n, 3, generator=g).to(cuda)
    sel = torch.randperm(n, generator=g)[:m].sort().values.to(cuda)
    new_xyz = xyz[sel].contiguous()
    feat = torch.randn(n, c, generator=g).to(cuda)
    off = torch.tensor([1200, n], dtype=torch.int32, device=cuda)
    noff = torch.tensor([int((sel < 1200).sum()), m], dtype=torch.int32, device=cuda)
    out = P.queryandgroup(ns, xyz, new_xyz, feat, None, off, noff, use_xyz=True)
    idx, _ = P.knnquery(ns, xyz, new_xyz, off, noff)
    want = torch.cat([xyz[idx.long()] - new_xyz[:, None], feat[idx.long()]], -1)
    assert torch.equal(out, want)
    assert torch.equal(P.queryandgroup(ns, xyz, new_xyz, feat, idx, off, noff, use_xyz=False), feat[idx.long()])
    # interpolation2: coarse (new_xyz, m points) -> fine (xyz, n points)
    cf = torch.randn(m, c, generator=g).to(cuda).requires_grad_(True)
    got = P.interpolation2(new_xyz, xyz, cf, noff, off, k=3)
    i3, d3 = P.knnquery(3, new_xyz, xyz, noff, off)
    wgt = 1.0 / (d3 + 1e-8)
    wgt = wgt / wgt.sum(1, keepdim=True)
    want = (cf.detach()[i3.long()].double() * wgt[..., None].double()).sum(1)
    assert torch.allclose(got.double(), want, rtol=1e-5, atol=1e-6)
    go = torch.randn(n, c, generator=g).to(cuda)
    got.backward(go)
    wantg = torch.zeros(m, c, dtype=torch.float64, device=cuda).index_add_(0, i3.reshape(-1).long(),
                                                                         (go[:, None, :].double() * wgt[..., None].double()).reshape(-1, c))
    assert torch.allclose(cf.grad.double(), wantg, rtol=1e-5, atol=1e-5)
    assert torch.equal(P.interpolation(new_xyz, xyz, cf.detach(), noff, off, k=3), got.detach())
