"""The float64 field reference (tests/field_reference.py) against torch's grid_sample, the CPU oracle and autograd, and the
sensitivity of the element-wise bound the GPU field tests use: slightly wrong versions of the reference must fail it."""
import itertools

import pytest
import torch
import torch.nn.functional as F

from oracle import kplanes_oracle as ko
from tests import field_reference as fr


class _Pts:
    """Duck-typed ops.Points (the reference only reads these fields)."""

    def __init__(self, D, pts=None, origins=None, directions=None, starts=None, ends=None, times=None, norm_mode=1,
                 aabb=(0.0,) * 6):
        self.D, self.pts, self.origins, self.directions, self.starts, self.ends, self.times = D, pts, origins, directions, starts, ends, times
        self.S = 1 if starts is None else starts.shape[-1]
        self.norm_mode, self.aabb = norm_mode, aabb


def _planes(gen, c, reso, lo=-1.0, hi=1.0):
    return [torch.empty(1, c, reso[b], reso[a]).uniform_(lo, hi, generator=gen) for a, b in itertools.combinations(range(len(reso)), 2)]


def _edge_points(gen, m, reso):
    """Off-grid points in [-1.2, 1.2], texel centres, exactly +-1 and beyond, mixed per coordinate."""
    d = len(reso)
    pts = torch.rand(m, d, generator=gen) * 2.4 - 1.2
    for j in range(d):
        r = max(reso[j], 2)
        centres = torch.randint(0, r, (m,), generator=gen).float() / (r - 1) * 2.0 - 1.0
        special = torch.tensor([-1.0, 1.0, -1.5, 1.5, 0.0])[torch.randint(0, 5, (m,), generator=gen)]
        pick = torch.randint(0, 3, (m,), generator=gen)
        pts[:, j] = torch.where(pick == 0, centres, torch.where(pick == 1, special, pts[:, j]))
    return pts


@pytest.mark.parametrize("reso", [(5, 7, 4), (9, 1, 6), (1, 1, 3)])
def test_single_plane_interpolant_matches_grid_sample(reso):
    """Each plane alone (use_mask with one bit) is grid_sample(bilinear, border, align_corners) of its two coordinates."""
    gen = torch.Generator().manual_seed(1)
    planes = [p.double() for p in _planes(gen, 4, reso)]
    pts = _edge_points(gen, 500, reso)
    pt = fr.coords(_Pts(3, pts=pts))
    for p, (a, b) in enumerate(itertools.combinations(range(3), 2)):
        mine = fr.gather(pt, [planes], 1 << p, True)
        grid = pts[:, [a, b]].double().view(1, 1, -1, 2)
        ref = F.grid_sample(planes[p], grid, mode="bilinear", padding_mode="border", align_corners=True).view(4, -1).t()
        # fp32 vs fp64 source index: |d ix| <= 3u (R-1) per axis, times the largest texel difference (2 max|v|)
        tol = 12 * fr.U * max(reso) * float(planes[p].abs().max())
        assert float((mine - ref).abs().max()) <= tol, (reso, p)


def test_weights_and_touched_corners_at_grid_edges():
    """x = +-1 and beyond: one corner with weight 1; a texel centre: the second corner has weight 0 and is not touched;
    an axis with R = 1: one texel, weight 1."""
    x = torch.tensor([-1.0, 1.0, -3.0, 2.0, 0.0, 0.5])
    i0, i1, w0, w1 = fr.axis(x, 5)
    assert i0.tolist() == [0, 4, 0, 4, 2, 3] and i1.tolist() == [1, 4, 1, 4, 3, 4]
    assert w0.tolist() == [1.0] * 6 and w1.tolist() == [0.0] * 6
    i0, i1, w0, w1 = fr.axis(x, 1)
    assert (i0 == 0).all() and (i1 == 0).all() and (w0 == 1).all() and (w1 == 0).all()
    plane = [torch.rand(1, 4, 5, 5).double() for _ in range(3)]
    pt = fr.coords(_Pts(3, pts=torch.tensor([[0.0, 0.5, 1.0]])))
    _, n, touched = fr.scatter(pt, [plane], 0x7, True, torch.ones(1, 4), [True] * 3)
    assert [int(t.sum()) for t in touched] == [1, 1, 1] and all(int(c.sum()) == 1 for c in n)


@pytest.mark.parametrize("concat", [True, False])
@pytest.mark.parametrize("d", [3, 4])
def test_gather_matches_oracle_within_the_bound(d, concat):
    """The CPU oracle (fp32 grid_sample, another fp32 implementation of the same sums) meets the bound the GPU tests use;
    frozen time planes (use_mask 0x0B: planes XT, YT, ZT skipped) match the oracle's freeze_time_planes."""
    gen = torch.Generator().manual_seed(2)
    reso = [(6, 5, 7, 4)[:d], (12, 10, 14, 4)[:d]]
    ms = [_planes(gen, 8, r, 0.1, 0.5) for r in reso]
    pts = _edge_points(gen, 2000, reso[1])
    pt = fr.coords(_Pts(d, pts=pts))
    assert fr.gather_ratio(ko.interpolate_kplanes(pts, ms, concat), pt, ms, 0x3F if d == 4 else 0x7, concat) <= 1.0
    if d == 4:
        frozen = ko.interpolate_kplanes(pts, ms, concat, freeze_time_planes=True)
        assert fr.gather_ratio(frozen, pt, ms, 0x0B, concat) <= 1.0


def test_ray_coordinates_follow_the_kernel_op_order():
    """norm_mode 0 / 1 equal the oracle's _normalized on positions o + (d*(s+e))*0.5; norm_mode 2 is the L_inf contraction."""
    gen = torch.Generator().manual_seed(3)
    n, s = 40, 6
    o = torch.randn(n, 3, generator=gen)
    dr = F.normalize(torch.randn(n, 3, generator=gen), dim=-1)
    edges = torch.sort(torch.rand(n, s + 1, generator=gen) * 4.0, dim=-1).values
    st, en = edges[:, :-1].contiguous(), edges[:, 1:].contiguous()
    t = torch.rand(n, generator=gen)
    aabb = torch.tensor([[-1.5, -1.0, -2.0], [1.5, 2.0, 2.0]])
    pos = o[:, None, :] + (dr[:, None, :] * (st + en)[..., None]) * 0.5
    q = ko._normalized(pos, aabb).reshape(-1, 3)
    for mode, want in ((0, q), (1, q * 2.0 - 1.0)):
        pt = fr.coords(_Pts(4, origins=o, directions=dr, starts=st, ends=en, times=t, norm_mode=mode, aabb=tuple(aabb.reshape(-1).tolist())))
        assert torch.equal(pt[:, :3], want) and torch.equal(pt[:, 3], (t * 2.0 - 1.0).repeat_interleave(s))
    pt = fr.coords(_Pts(3, origins=o, directions=dr, starts=st, ends=en, norm_mode=2))
    p64 = pos.reshape(-1, 3).double()
    mag = p64.abs().amax(-1, keepdim=True)
    want = torch.where(mag < 1, p64, (2 - 1 / mag) * p64 / mag) * 0.5
    assert float((pt[:, :3].double() - want).abs().max()) < 1e-6 and (pt[:, 3] == 0).all()


def test_scatter_is_the_gradient_of_the_gather():
    """Scatter == autograd of the float64 gather (sum and concat, a plane without target, frozen time planes)."""
    gen = torch.Generator().manual_seed(4)
    reso = [(5, 6, 7, 3), (9, 11, 13, 1)]
    ms = [[p.double().requires_grad_(True) for p in _planes(gen, 4, r)] for r in reso]
    pt = fr.coords(_Pts(4, pts=_edge_points(gen, 700, reso[1])))
    for concat, mask in ((True, 0x3F), (False, 0x1B)):
        out = fr.gather(pt, ms, mask, concat)
        g = torch.randn(out.shape, generator=gen, dtype=torch.float64)
        auto = torch.autograd.grad((out * g).sum(), [p for s in ms for p in s], allow_unused=True)
        need = [True] * 12
        need[4] = False
        mine, n, touched = fr.scatter(pt, [[p.detach() for p in s] for s in ms], mask, concat, g, need)
        for i, (a, b) in enumerate(zip(auto, mine)):
            if not need[i] or not (mask >> (i % 6)) & 1:
                assert b is None
                continue
            a = fr.texels(a)
            assert torch.allclose(a, b, rtol=0, atol=1e-12 * float(a.abs().max())), (concat, i)
            assert bool((a[~touched[i]] == 0).all())


@pytest.mark.parametrize("relu", [True, False])
def test_density_matches_oracle_and_autograd(relu):
    """Forward: the oracle's density_field (fp32, norm_mode 0 ray form) meets the density bound.  Backward: float64
    autograd of the same forward through trunc_exp."""
    gen = torch.Generator().manual_seed(5)
    n, s = 30, 7
    origins, directions, times, aabb = ko.synthetic_rays(n, gen)
    dp = ko.make_density_params(aabb, [10, 9, 11, 5], 8, gen)
    edges = torch.sort(torch.rand(n, s + 1, generator=gen) * 3.0, dim=-1).values
    st, en = edges[:, :-1].contiguous(), edges[:, 1:].contiguous()
    P = _Pts(4, origins=origins, directions=directions, starts=st, ends=en, times=times.reshape(-1), norm_mode=0,
             aabb=tuple(aabb.reshape(-1).tolist()))
    pt = fr.coords(P)
    w1, w2 = dp.sigma_w
    if relu:
        pos = origins[:, None, :] + (directions[:, None, :] * (st + en)[..., None]) * 0.5
        ref = ko.density_field(dp, pos, times).reshape(-1)
        assert fr.density_ratio(ref, pt, dp.grids, w1, w2, True, 0x3F) <= 1.0
    planes = [p.double().requires_grad_(True) for p in dp.grids]
    W1, W2 = w1.double().requires_grad_(True), w2.double().requires_grad_(True)
    raw, _ = fr.density(pt, planes, W1, W2, relu, 0x3F)
    g = torch.randn(raw.shape, generator=gen, dtype=torch.float64)
    auto = torch.autograd.grad((ko.trunc_exp(raw) * g).sum(), planes + [W1, W2])
    mine, _, gw1, gw2 = fr.density_backward(pt, [p.detach() for p in dp.grids], w1, w2, relu, 0x3F, g, [True] * 6)
    for a, b in zip(auto, mine + [gw1, gw2]):
        a = fr.texels(a) if a.dim() == 4 else a.reshape(b.shape)
        assert torch.allclose(a, b, rtol=0, atol=1e-12 * float(a.abs().max()))


# ---- sensitivity of the bound --------------------------------------------------------------------------------------------
def _case(seed=6):
    gen = torch.Generator().manual_seed(seed)
    reso = [(6, 5, 7, 4), (12, 10, 14, 4)]
    ms = [_planes(gen, 8, r, 0.1, 0.5) for r in reso]
    pts = torch.rand(3000, 4, generator=gen) * 2.0 - 1.0
    return ms, fr.coords(_Pts(4, pts=pts)), torch.randn(3000, 16, generator=gen)


def _fp32_side(ms, pt, g, **kw):
    """The reference evaluated in fp32 stands in for a kernel."""
    out = fr.gather(pt, ms, 0x3F, True, dtype=torch.float32, **kw)
    grads, _, _ = fr.scatter(pt, ms, 0x3F, True, g, [True] * 12, dtype=torch.float32)
    return out, grads


def _ratios(ms, pt, g, out, grads):
    prior = [torch.zeros_like(x) for x in grads]
    return fr.gather_ratio(out, pt, ms, 0x3F, True), fr.scatter_ratio(grads, prior, pt, ms, 0x3F, True, g, [True] * 12)[0]


def test_unperturbed_fp32_evaluation_meets_the_bound():
    ms, pt, g = _case()
    rg, rs = _ratios(ms, pt, g, *_fp32_side(ms, pt, g))
    print(f"fp32 reference: gather err/bound {rg:.3g}, scatter err/bound {rs:.3g}")
    assert rg <= 1.0 and rs <= 1.0


def test_bound_rejects_one_corner_weight_off_by_2_pow_minus_16(monkeypatch):
    ms, pt, g = _case()
    real = fr.corners

    def skewed(pt_, planes, dtype=torch.float64):
        cs = real(pt_, planes, dtype)
        idx, w = cs[0]
        w = w.clone()
        w[:, 1] *= 1.0 + 2.0 ** -16
        return [(idx, w)] + cs[1:]

    monkeypatch.setattr(fr, "corners", skewed)
    out, grads = _fp32_side(ms, pt, g)
    monkeypatch.setattr(fr, "corners", real)
    rg, rs = _ratios(ms, pt, g, out, grads)
    print(f"corner weight * (1 + 2^-16): gather err/bound {rg:.3g}, scatter err/bound {rs:.3g}")
    assert rg > 1.0 and rs > 1.0


def test_bound_rejects_two_swapped_channels_in_one_plane():
    ms, pt, g = _case()
    bad = [list(s) for s in ms]
    bad[1][3] = bad[1][3][:, [0, 1, 2, 4, 3, 5, 6, 7]]
    out = fr.gather(pt, bad, 0x3F, True, dtype=torch.float32)
    grads, _, _ = fr.scatter(pt, bad, 0x3F, True, g, [True] * 12, dtype=torch.float32)
    rg, rs = _ratios(ms, pt, g, out, grads)
    print(f"channels 3/4 of one plane swapped: gather err/bound {rg:.3g}, scatter err/bound {rs:.3g}")
    assert rg > 1.0 and rs > 1.0
