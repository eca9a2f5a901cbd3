"""Parity of the CUDA path (through the C-ABI) against the reference-generated fixtures and the CPU oracle.

Bar (BASELINE.json north_star): integer outputs (searchsorted indices, median indices) bit-exact; sample bins
bit-exact; fp32 outputs within 1e-4 relative.  The norm for fp32 tensors is max|a-b| / max|b| (per tensor), which
for gradients means "relative to the largest gradient entry of that parameter" -- atomics reorder fp32 sums,
so entry-wise relative error on near-zero texels is not meaningful (SURVEY.md section 7, hard parts).
"""
import pytest
import torch

from oracle import kplanes_oracle as ko
from tests.conftest import load_golden, rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-4
DEV = "cuda"


def _nchw_to_param(p):
    from soccernerfs_b200 import ops

    return ops.as_channel_last(p.to(DEV)).requires_grad_(True)


def test_library_loaded_and_abi():
    from soccernerfs_b200 import _lib

    lib = _lib.load()
    assert lib.kp_abi_version() == 4


def test_hexplane_vs_reference_fixture():
    from soccernerfs_b200.fields.kplanes_field import interpolate_kplanes

    g = load_golden("interp")
    grids = [[_nchw_to_param(g[f"grid_{i}_{j}"]) for j in range(6)] for i in range(2)]
    pts = g["pts"].to(DEV)
    out = interpolate_kplanes(pts, grids, True)
    assert rel_err(out.cpu(), g["out_cat"]) < TOL
    (out * g["grad_out"].to(DEV)).sum().backward()
    for i in range(2):
        for j in range(6):
            assert rel_err(grids[i][j].grad.cpu(), g[f"ggrid_{i}_{j}"]) < TOL, (i, j)
    assert rel_err(interpolate_kplanes(pts, grids, False).cpu(), g["out_sum"]) < TOL
    g3 = [[_nchw_to_param(g[f"grid3_{j}"]) for j in range(3)]]
    assert rel_err(interpolate_kplanes(pts[:, :3].contiguous(), g3, True).cpu(), g["out_static"]) < TOL


def test_gather_ray_tile_only_changes_the_thread_mapping():
    """KpPoints.ray_tile (full-frame inference: a warp takes one sample index of neighbouring rays) writes every sample's
    features at its own row: bit-identical to the default mapping, also when the ray count is not a multiple of the tile and
    for both channel widths."""
    from soccernerfs_b200 import ops

    gen = torch.Generator().manual_seed(11)
    combos = [(0, 1), (0, 2), (0, 3), (1, 2), (1, 3), (2, 3)]
    for c, n_rays, s in ((32, 1027, 48), (8, 515, 7)):
        reso = [(8, 8, 8, 5), (16, 16, 16, 5)]
        planes = [[torch.rand(1, c, r[b], r[a], generator=gen).to(DEV).contiguous(memory_format=torch.channels_last)
                   for a, b in combos] for r in reso]
        o = (torch.rand(n_rays, 3, generator=gen) - 0.5).to(DEV)
        d = torch.nn.functional.normalize(torch.randn(n_rays, 3, generator=gen), dim=-1).to(DEV)
        edges = torch.sort(torch.rand(n_rays, s + 1, generator=gen) * 2.0, dim=-1).values.to(DEV)
        t = torch.rand(n_rays, generator=gen).to(DEV)
        aabb = (-1.0, -1.0, -1.0, 1.0, 1.0, 1.0)
        outs = []
        for tile in (-1, 0, 4, 16):  # -1: the float4-per-lane kernel; >= 0 with C = 32: the 8-channels-per-lane kernel
            pts = ops.points_from_rays(o, d, edges[:, :-1].contiguous(), edges[:, 1:].contiguous(), t, aabb, norm_mode=1,
                                       dynamic=True, ray_tile=tile)
            with torch.no_grad():
                outs.append(ops.hexplane_features(planes, pts, True))
        assert outs[0].abs().sum() > 0
        assert all(torch.equal(outs[0], o_) for o_ in outs[1:]), (c, n_rays, s)


def test_hexplane_freeze_flags():
    from soccernerfs_b200.fields.kplanes_field import interpolate_kplanes

    g = load_golden("interp")
    grids_cpu = [[g[f"grid_{i}_{j}"].clone().requires_grad_(True) for j in range(6)] for i in range(2)]
    ref = ko.interpolate_kplanes(g["pts"], grids_cpu, True, freeze_time_planes=True)
    grids = [[_nchw_to_param(g[f"grid_{i}_{j}"]) for j in range(6)] for i in range(2)]
    out = interpolate_kplanes(g["pts"].to(DEV), grids, True, freeze_time_planes=True, freeze_space_planes=True)
    assert rel_err(out.cpu(), ref) < TOL
    out.sum().backward()
    assert all(grids[i][j].grad is None for i in range(2) for j in range(6))  # time skipped, space frozen


def test_per_scale_scatter_equals_single_launch():
    """Scatter launched one scale at a time (finest first, hook after each) == the one-launch scatter."""
    from soccernerfs_b200 import ops

    gen = torch.Generator().manual_seed(5)
    reso = [(8, 8, 8, 5), (16, 16, 16, 5), (32, 32, 32, 5)]
    combos = [(0, 1), (0, 2), (0, 3), (1, 2), (1, 3), (2, 3)]
    pts = (torch.rand(3000, 4, generator=gen) * 2.2 - 1.1).to(DEV)
    gout = torch.randn(3000, 3 * 8, generator=gen).to(DEV)
    base = [[torch.rand(1, 8, r[b], r[a], generator=gen) for a, b in combos] for r in reso]
    grads, calls = {}, []
    for mode in ("single", "per_scale"):
        ms = [[ops.as_channel_last(p.to(DEV)).clone(memory_format=torch.preserve_format).requires_grad_(True) for p in g] for g in base]
        hook = None
        if mode == "per_scale":
            def hook(k=None):
                calls.append(k)
            hook.per_scale = True
        out = ops.hexplane_features(ms, ops.points_from_pts(pts), True, post_backward=hook)
        out.backward(gout)
        grads[mode] = [p.grad.clone() for g in ms for p in g]
    assert calls == [2, 1, 0]
    for a, b in zip(grads["single"], grads["per_scale"]):
        assert rel_err(b, a) < 1e-5 and float(a.abs().sum()) > 0


def test_empty_input():
    from soccernerfs_b200.fields.kplanes_field import interpolate_kplanes

    g = load_golden("interp")
    grids = [[_nchw_to_param(g[f"grid_{i}_{j}"]) for j in range(6)] for i in range(2)]
    out = interpolate_kplanes(torch.zeros(0, 4, device=DEV), grids, True)
    assert out.shape == (0, 16)


def test_samplers_bit_exact_vs_reference_fixture():
    from soccernerfs_b200 import ops

    g = load_golden("samplers")
    o, d, aabb = g["origins"].to(DEV), g["directions"].to(DEV), g["aabb"]
    for near_plane, key in ((0.05, "train"), (0.0, "eval")):
        n_, f_ = ops.aabb_intersect(o, d, aabb.flatten().tolist(), near_plane)
        assert torch.equal(n_.cpu()[:, None], g[f"nears_{key}"]) and torch.equal(f_.cpu()[:, None], g[f"fars_{key}"])
    nears, fars = g["nears_train"].to(DEV), g["fars_train"].to(DEV)
    for mode in ("train", "eval"):
        tr = g[f"{mode}_t_rand"].to(DEV) if mode == "train" else None
        ur = g[f"{mode}_u_rand"].to(DEV) if mode == "train" else None
        sb, eb = ops.uniform_bins(nears, fars, 40, tr)
        assert torch.equal(sb.cpu(), g[f"{mode}_bins0"])
        assert torch.equal(eb.cpu()[:, :-1], g[f"{mode}_starts0"]) and torch.equal(eb.cpu()[:, 1:], g[f"{mode}_ends0"])
        w = g[f"{mode}_weights"][..., 0].to(DEV)
        sb1, eb1, inds, cdf = ops.pdf_resample(w, sb, nears, fars, 24, ur, want_inds=True, want_cdf=True)
        ref_cdf = ko.pdf_cdf(g[f"{mode}_weights"][..., 0])
        # the stated bar: cdf, searchsorted indices, resampled bins and euclidean edges bit-identical on EVERY ray (the
        # kernel reproduces torch's CPU row-sum order and its double-accumulated cumsum)
        assert torch.equal(cdf.cpu(), ref_cdf)
        assert torch.equal(inds.cpu(), g[f"{mode}_inds1"])
        assert torch.equal(sb1.cpu(), g[f"{mode}_bins1"])
        assert torch.equal(eb1.cpu()[:, :-1], g[f"{mode}_starts1"]) and torch.equal(eb1.cpu()[:, 1:], g[f"{mode}_ends1"])


def test_pdf_search_bit_exact_given_cdf():
    """The inverse-CDF search itself: feed weights whose cdf is exactly representable -> indices must be identical."""
    from soccernerfs_b200 import ops

    gen = torch.Generator().manual_seed(7)
    n, s_in, s_out = 512, 64, 48
    w = torch.randint(0, 8, (n, s_in), generator=gen).float() / 4.0  # multiples of 0.25: sums exact in fp32
    w[:, 0] += 1.0
    bins = torch.sort(torch.rand(n, s_in + 1, generator=gen), -1).values
    rand = torch.rand(n, s_out + 1, generator=gen)
    nears, fars = torch.zeros(n, 1), torch.ones(n, 1) * 3
    prev = ko.Samples(torch.zeros(n, 3), torch.ones(n, 3), bins[:, :-1], bins[:, 1:], bins, nears, fars)
    # histogram_padding 0.25 keeps everything a multiple of 0.25
    cdf = ko.pdf_cdf(w, histogram_padding=0.25)
    u = ko.pdf_u(n, s_out, rand)
    ref_inds = torch.searchsorted(cdf, u, side="right")
    _, _, inds, kcdf = ops.pdf_resample(w.to(DEV), bins.to(DEV), nears.to(DEV), fars.to(DEV), s_out, rand.to(DEV),
                                        histogram_padding=0.25, want_inds=True, want_cdf=True)
    assert torch.equal(kcdf.cpu(), cdf)
    assert torch.equal(inds.cpu(), ref_inds)
    del prev


def test_sampler_frustum_outputs_and_in_kernel_anneal():
    """The extra kernel outputs are exactly the views the reference takes: starts = bins[:-1], ends = bins[1:],
    deltas = ends - starts; pow(weights, anneal) inside the PDF kernel == torch.pow before it."""
    from soccernerfs_b200 import ops

    gen = torch.Generator().manual_seed(11)
    n, s0, s1 = 300, 64, 48
    nears, fars = torch.rand(n, 1, generator=gen).to(DEV), (2 + torch.rand(n, 1, generator=gen)).to(DEV)
    for mode in (0, 1):
        t_rand = torch.rand(n, s0 + 1, generator=gen).to(DEV)
        sb, eb, st, en, de = ops.uniform_bins(nears, fars, s0, t_rand, mode, want_frustums=True)
        sb2, eb2 = ops.uniform_bins(nears, fars, s0, t_rand, mode)
        assert torch.equal(sb, sb2) and torch.equal(eb, eb2)
        assert torch.equal(st, eb[:, :-1]) and torch.equal(en, eb[:, 1:]) and torch.equal(de, eb[:, 1:] - eb[:, :-1])
        w = torch.rand(n, s0, generator=gen).to(DEV)
        rand = torch.rand(n, s1 + 1, generator=gen).to(DEV)
        for anneal in (0.37, torch.tensor(0.37, device=DEV)):
            a = ops.pdf_resample(w, sb, nears, fars, s1, rand, spacing=mode, anneal=anneal, want_frustums=True, want_inds=True)
            b = ops.pdf_resample(torch.pow(w, 0.37), sb, nears, fars, s1, rand, spacing=mode, want_inds=True)
            assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
            assert torch.equal(a[4], a[1][:, :-1]) and torch.equal(a[5], a[1][:, 1:])
            assert torch.equal(a[6], a[1][:, 1:] - a[1][:, :-1])


def test_compositing_vs_reference_fixture():
    from soccernerfs_b200 import ops

    g = load_golden("render")
    starts = g["starts"]
    deltas = (starts[:, 1:] - starts[:, :-1]).to(DEV)
    steps = ((starts[:, :-1] + starts[:, 1:]) / 2).to(DEV)
    density = g["density"][..., 0].to(DEV).requires_grad_(True)
    rgb = g["rgb"].to(DEV).requires_grad_(True)
    w = ops.get_weights(deltas, density)
    assert rel_err(w.cpu(), g["weights"][..., 0]) < TOL
    comp = ops.composite_rgb(w, rgb, g["bg"].to(DEV))
    acc = ops.accumulate(w)
    assert rel_err(comp.cpu(), g["comp"]) < TOL and rel_err(acc.cpu(), g["acc"][:, 0]) < TOL
    idx = ops.median_index(w)
    assert torch.equal(idx.cpu(), ko.median_index(g["weights"])[:, 0])  # int64, bit-exact
    assert torch.equal(torch.gather(steps, -1, idx[:, None]).cpu(), g["depth_median"])
    md = ops.median_depth(w, starts[:, :-1].to(DEV), starts[:, 1:].to(DEV))  # same thing, one kernel
    assert torch.equal(md.cpu(), g["depth_median"][:, 0])
    ed = ops.expected_depth(w, steps)
    assert rel_err(torch.clip(ed, steps.min(), steps.max()).cpu(), g["depth_expected"][:, 0]) < TOL
    ((comp * g["go_rgb"].to(DEV)).sum() + (acc * g["go_acc"][:, 0].to(DEV)).sum() + (w * g["go_w"][..., 0].to(DEV)).sum()).backward()
    assert rel_err(density.grad.cpu(), g["g_density"][..., 0]) < TOL
    assert rel_err(rgb.grad.cpu(), g["g_rgb"]) < TOL
    comp_eval = ops.composite_rgb(g["weights"][..., 0].to(DEV), g["rgb"].to(DEV), "last_sample", nan_to_num=True).clamp(0, 1)
    assert rel_err(comp_eval.cpu(), g["comp_eval"]) < TOL


def test_renderer_modules_vs_reference_fixture():
    from soccernerfs_b200.cameras.rays import Frustums, RaySamples
    from soccernerfs_b200.model_components import renderers as rr

    g = load_golden("render")
    n, s = g["density"].shape[:2]
    starts = g["starts"].to(DEV)
    fr = Frustums(origins=torch.zeros(n, s, 3, device=DEV), directions=torch.ones(n, s, 3, device=DEV),
                  starts=starts[:, :-1, None], ends=starts[:, 1:, None], pixel_area=torch.ones(n, s, 1, device=DEV))
    rs = RaySamples(frustums=fr, deltas=(starts[:, 1:] - starts[:, :-1])[..., None])
    w = rs.get_weights(g["density"].to(DEV))
    assert rel_err(w.cpu(), g["weights"]) < TOL
    r = rr.RGBRenderer(background_color=g["bg"].to(DEV))
    r.train()
    assert rel_err(r(g["rgb"].to(DEV), w).cpu(), g["comp"]) < TOL
    assert rel_err(rr.AccumulationRenderer()(w).cpu(), g["acc"]) < TOL
    assert torch.equal(rr.DepthRenderer("median")(w, rs).cpu(), g["depth_median"])
    assert rel_err(rr.DepthRenderer("expected")(w, rs).cpu(), g["depth_expected"]) < TOL
    m = rr.MedianRGBRenderer()
    m.train()
    assert torch.equal(m(g["rgb"].to(DEV), w).cpu(), g["median_rgb"])
    re = rr.RGBRenderer(background_color="last_sample")
    re.eval()
    assert rel_err(re(g["rgb"].to(DEV), w).cpu(), g["comp_eval"]) < TOL
    with rr.background_color_override_context(torch.tensor([0.25, 0.5, 0.75], device=DEV)):
        ov = r(g["rgb"].to(DEV), w)
    ref = ko.render_rgb(g["rgb"], g["weights"], torch.tensor([0.25, 0.5, 0.75]))
    assert rel_err(ov.cpu(), ref) < TOL


def test_losses_vs_reference_fixture():
    from soccernerfs_b200.model_components import losses as L

    g = load_golden("losses")

    class RS:
        def __init__(self, b):
            self.spacing_starts = b[:, :-1, None].to(DEV)
            self.spacing_ends = b[:, 1:, None].to(DEV)

    ws = [g[f"w{i}"].to(DEV).requires_grad_(True) for i in range(3)]
    rss = [RS(g[f"b{i}"]) for i in range(3)]
    il, dl = L.interlevel_loss(ws, rss), L.distortion_loss(ws, rss)
    assert rel_err(il.cpu(), g["interlevel"]) < TOL and rel_err(dl.cpu(), g["distortion"]) < TOL
    (il + dl).backward()
    for i in range(3):
        assert rel_err(ws[i].grad.cpu(), g[f"g_w{i}"]) < TOL, i
    grids = [[_nchw_to_param(g[f"grid_{i}_{j}"]) for j in range(6)] for i in range(2)]
    tv, ts, st = L.space_tv_loss(grids), L.time_smoothness_loss(grids), L.sparse_transients_loss(grids)
    assert rel_err(tv.cpu(), g["space_tv"]) < TOL and rel_err(ts.cpu(), g["time_smoothness"]) < TOL
    assert rel_err(st.cpu(), g["sparse_transients"]) < TOL
    (0.7 * tv + 1.3 * ts + 0.4 * st).backward()
    for i in range(2):
        for j in range(6):
            assert rel_err(grids[i][j].grad.cpu(), g[f"ggrid_{i}_{j}"]) < TOL, (i, j)
    g3 = [[_nchw_to_param(g[f"grid3_{j}"]) for j in range(3)]]
    assert rel_err(L.space_tv_loss(g3).cpu(), g["space_tv_static"]) < TOL
    assert float(L.time_smoothness_loss(g3)) == 0.0 and float(L.sparse_transients_loss(g3)) == 0.0
    p = grids[0][2].detach()
    assert rel_err(L.compute_plane_tv(p).cpu(), ko.compute_plane_tv(g["grid_0_2"])) < TOL
    assert rel_err(L.compute_plane_tv(p, only_w=True).cpu(), ko.compute_plane_tv(g["grid_0_2"], only_w=True)) < TOL
    assert rel_err(L.compute_plane_smoothness(p).cpu(), ko.compute_plane_smoothness(g["grid_0_2"])) < TOL


def test_loss_head_matches_torch_formulas():
    """ops.loss_head == coef * mse / mean / sum-of-means, total and PSNR as get_loss_dict / get_metrics_dict write
    them (kplanes.py:392-452), forward and backward, twice in a row (the kernel re-zeroes its workspace)."""
    from soccernerfs_b200 import ops

    gen = torch.Generator().manual_seed(3)
    n = 1000
    for rep in range(2):
        pred = torch.rand(n, 3, generator=gen).to(DEV).requires_grad_(True)
        image = torch.rand(n, 3, generator=gen).to(DEV)
        dist = torch.rand(n, generator=gen).to(DEV).requires_grad_(True)
        il = [torch.rand(n, s, generator=gen).to(DEV).requires_grad_(True) for s in (48, 37)]
        extra = torch.rand(6, generator=gen).to(DEV)
        c = (1.0, 0.001, 1.0)
        vals, total, psnr = ops.loss_head(pred, image, dist, il, *c, extra=extra)
        mse = torch.nn.functional.mse_loss(image, pred)
        ref_vals = torch.stack([c[0] * mse, c[1] * dist.mean(), c[2] * (il[0].mean() + il[1].mean())])
        ref_total = ref_vals.sum() + extra.sum()
        assert rel_err(vals.detach(), ref_vals.detach()) < 1e-6
        assert abs(float(total.detach() - ref_total.detach())) < 1e-6 * abs(float(ref_total.detach()))
        assert abs(float(psnr) - float(-10.0 * torch.log10(mse.detach()))) < 1e-4
        inputs = [pred, dist, *il]
        g = torch.autograd.grad(total + 0.5 * vals[1], inputs)
        g_ref = torch.autograd.grad(ref_total + 0.5 * ref_vals[1], inputs)
        for a, b in zip(g, g_ref):
            assert rel_err(a, b) < 1e-6
    # without distortion / interlevel terms
    vals, total, _ = ops.loss_head(pred.detach(), image, None, [], 2.0, 0.0, 0.0)
    assert abs(float(total) - 2.0 * float(torch.nn.functional.mse_loss(image, pred.detach()))) < 1e-6


def test_decoders_and_density_field_vs_oracle():
    from soccernerfs_b200.fields.kplanes_field import KPlanesDensityField, KPlanesField

    gen = torch.Generator().manual_seed(11)
    n, s = 37, 9
    origins, directions, times, aabb = ko.synthetic_rays(n, gen)
    for view_dep, hid in ((True, 64), (False, 128), (False, 64)):
        fp = ko.make_field_params(aabb, (12, 10, 14, 5), 32, (1, 2, 4), gen, sigma_hidden=hid, view_dependent=view_dep)
        nears, fars = ko.aabb_collider(origins, directions, aabb)
        smp = ko.uniform_sampler(origins, directions, nears, fars, times, s, torch.rand(n, s + 1, generator=gen))
        for t in fp.tensors():
            t.requires_grad_(True)
        density, rgb, _ = ko.field_forward(fp, smp)
        gd, gr = torch.randn(density.shape, generator=gen), torch.randn(rgb.shape, generator=gen)
        ((density * gd).sum() + (rgb * gr).sum()).backward()

        field = KPlanesField(aabb, spacetime_resolution=(12, 10, 14, 5), feat_dim=32, multiscale_res=(1, 2, 4),
                             concat_features_across_scales=True, linear_decoder=False, disable_viewing_dependent=not view_dep,
                             sigma_net_hidden_dim=hid).to(DEV)
        mine = [q for gs in field.grids for q in gs] + list(field.sigma_net.weights) + list(field.color_net.weights)
        with torch.no_grad():
            for dst, src in zip(mine, fp.tensors()):
                dst.copy_(src.detach().to(DEV))
        from tests.helpers import ray_bundle

        rb = ray_bundle(origins, directions, times, DEV)
        rs = rb.get_ray_samples(bin_starts=smp.starts[..., None].to(DEV), bin_ends=smp.ends[..., None].to(DEV))
        out = field(rs)
        from soccernerfs_b200.fields.base_field import FieldHeadNames as FH

        assert rel_err(out[FH.DENSITY].cpu(), density) < TOL and rel_err(out[FH.RGB].cpu(), rgb) < TOL
        ((out[FH.DENSITY] * gd.to(DEV)).sum() + (out[FH.RGB] * gr.to(DEV)).sum()).backward()
        for i, (a, b) in enumerate(zip(mine, fp.tensors())):
            assert rel_err(a.grad.cpu(), b.grad) < TOL, (view_dep, i)

    # proposal density field: ray form (fused path) and density_fn(positions) (point form) agree with the oracle
    dp = ko.make_density_params(aabb, [20, 18, 22, 7], 8, gen)
    for t in dp.tensors():
        t.requires_grad_(True)
    ref = ko.density_field(dp, smp.positions(), times)
    gd = torch.randn(ref.shape, generator=gen)
    (ref * gd).sum().backward()
    dfield = KPlanesDensityField(aabb, resolution=[20, 18, 22, 7], feature_dim=8, linear_decoder=False).to(DEV)
    mine = list(dfield.grids) + list(dfield.sigma_net.weights)
    with torch.no_grad():
        for dst, src in zip(mine, dp.tensors()):
            dst.copy_(src.detach().to(DEV))
    d1, _ = dfield.get_density(rs)
    assert rel_err(d1.cpu(), ref) < TOL
    (d1 * gd.to(DEV)).sum().backward()
    for i, (a, b) in enumerate(zip(mine, dp.tensors())):
        assert rel_err(a.grad.cpu(), b.grad) < TOL, i
    d2 = dfield.density_fn(rs.frustums.get_positions(), times=rb.times)
    assert rel_err(d2.cpu(), ref) < TOL
    assert rel_err(d2, d1) < 1e-6


def test_model_step_vs_reference_fixture():
    """Whole training step (collider, proposal sampling, field, compositing, losses, backward) vs the fixture the
    REAL reference produced (oracle/make_golden.py: gen_model)."""
    from tests.helpers import build_model, train_step_cuda
    from tests.test_oracle_golden import load_tiny_model

    g = load_golden("model_tiny")
    mp = load_tiny_model(g)
    model = build_model("tiny", mp, g["aabb"], DEV)
    rand = {k[5:]: v for k, v in g.items() if k.startswith("rand_")}
    out, ld, grads = train_step_cuda(model, g["origins"], g["directions"], g["times"], g["image"], rand, float(g["anneal"]), DEV)
    # sampling: bins / indices
    # sampling: level 0 is bit-exact; levels 1-2 resample UPSTREAM densities that differ from the CPU's in the last bit
    # (expf, fused multiply-adds), so an index may differ where u is within an ulp of a cdf edge -- the resampled bin is a
    # continuous function across that edge and must still agree to fp32 rounding
    assert torch.equal(out["ray_samples_list"][0].spacing_starts[..., 0].cpu(), g["bins_0"][:, :-1])
    for lvl, key in ((0, "inds1"), (1, "inds2")):
        mism = (out["inds_list"][lvl].cpu() != g[key]).float().mean()
        assert mism < 2e-3, (lvl, float(mism))
    for i in range(3):
        rs = out["ray_samples_list"][i]
        bins = torch.cat([rs.spacing_starts[..., 0], rs.spacing_ends[..., -1:, 0]], -1).cpu()
        assert (bins - g[f"bins_{i}"]).abs().max() < 5e-6, i
        assert rel_err(out["weights_list"][i].cpu(), g[f"weights_{i}"]) < 1e-4, i
    # the stated fp32 bar, 1e-4, on outputs, every loss term and every gradient tensor
    for k in ("rgb", "accumulation", "depth", "prop_depth_0", "prop_depth_1"):
        assert rel_err(out[k].cpu(), g[k]) < 1e-4, k
    for k, v in ld.items():
        assert rel_err(v.detach().cpu(), g["loss_" + k]) < 1e-4, k
    for i, gr in enumerate(grads):
        assert rel_err(gr.cpu(), g[f"grad_{i}"]) < 1e-4, i


def test_fused_adam_matches_torch_adam():
    from soccernerfs_b200 import ops
    from soccernerfs_b200.engine.optimizers import FusedAdam

    gen = torch.Generator().manual_seed(3)
    shapes = [(1, 8, 13, 9), (64, 31), (3,), (1, 32, 16, 16)]
    ps = [torch.randn(s, generator=gen) for s in shapes]
    mine = [torch.nn.Parameter(ops.as_channel_last(p.to(DEV)) if p.dim() == 4 else p.to(DEV)) for p in ps]
    ref = [torch.nn.Parameter(p.clone()) for p in ps]
    a, b = FusedAdam(mine, lr=1e-2, eps=1e-12), torch.optim.Adam(ref, lr=1e-2, eps=1e-12)
    for _ in range(5):
        for m, r in zip(mine, ref):
            gr = torch.randn(r.shape, generator=gen)
            r.grad = gr.clone()
            m.grad = torch.empty_like(m).copy_(gr.to(DEV))
        a.step()
        b.step()
    for m, r in zip(mine, ref):
        assert rel_err(m.detach().cpu(), r.detach()) < 1e-5


def test_fused_adam_mixed_step_counts_matches_torch_adam():
    """A parameter without a gradient for the first two steps lags two steps behind the others: FusedAdam then launches
    kp_adam_multi once per step count.  Its size is not a multiple of 4, so the kernel's scalar tail runs too."""
    from soccernerfs_b200 import ops
    from soccernerfs_b200.engine.optimizers import FusedAdam

    gen = torch.Generator().manual_seed(4)
    shapes = [(1, 8, 13, 9), (64, 31), (37,), (1, 32, 16, 16)]
    late = 2
    ps = [torch.randn(s, generator=gen) for s in shapes]
    mine = [torch.nn.Parameter(ops.as_channel_last(p.to(DEV)) if p.dim() == 4 else p.to(DEV)) for p in ps]
    ref = [torch.nn.Parameter(p.clone()) for p in ps]
    a, b = FusedAdam(mine, lr=1e-2, eps=1e-12), torch.optim.Adam(ref, lr=1e-2, eps=1e-12)
    for it in range(5):
        for i, (m, r) in enumerate(zip(mine, ref)):
            if i == late and it < 2:
                continue
            gr = torch.randn(r.shape, generator=gen)
            r.grad = gr.clone()
            m.grad = torch.empty_like(m).copy_(gr.to(DEV))
        a.step()
        b.step()
    assert [a.state[p]["step"] for p in mine] == [5, 5, 3, 5]
    for m, r in zip(mine, ref):
        assert rel_err(m.detach().cpu(), r.detach()) < 1e-5


def test_adam_kernels_share_one_update_rule():
    """kp_adam_multi, kp_plane_reg_adam with no regulariser term and both sharded kernels at world 1 (kp_peer_sharded_adam,
    and kp_peer_sharded_adam_sparse with every line marked) give the same bits for the same p, g, m, v and grad_scale
    (weight_decay 0, as in the presets)."""
    from ctypes import byref, c_void_p, create_string_buffer

    from soccernerfs_b200 import _lib, ops
    from soccernerfs_b200.distributed import PeerArena, _RawCudaMemory

    C, H, W = 32, 37, 29
    n = C * H * W  # a multiple of 32 floats: the sparse kernel exchanges whole 128-byte lines
    gen = torch.Generator().manual_seed(9)
    p0, g0 = torch.randn(n, generator=gen).to(DEV), torch.randn(n, generator=gen).to(DEV)
    m0, v0 = (0.1 * torch.randn(n, generator=gen)).to(DEV), (0.01 * torch.rand(n, generator=gen)).to(DEV)
    lr, b1, b2, eps, wd, step, gs = 1e-2, 0.9, 0.999, 1e-12, 0.0, 7, 0.5

    p, m, v = p0.clone(), m0.clone(), v0.clone()
    ops.adam_multi_([p], [g0.clone()], [m], [v], lr, b1, b2, eps, wd, step, gs)
    ref = (p, m, v)
    assert not torch.equal(p, p0)
    got = {}

    def plane(t):  # channel-last [1,C,H,W] view of a flat buffer
        return t.view(1, H, W, C).permute(0, 3, 1, 2)

    p, m, v = p0.clone(), m0.clone(), v0.clone()
    scratch = torch.empty(ops.plane_reg_adam_scratch_bytes([plane(p)]), dtype=torch.uint8, device=DEV)
    coef = torch.rand(1, 4, generator=gen).to(DEV)  # unused: terms = 0 selects no regulariser
    ops.plane_reg_adam_([plane(p)], [plane(g0.clone())], [plane(m)], [plane(v)], [0], coef, lr, b1, b2, eps, wd, step, gs,
                        scratch, zero_grads=False)
    got["plane_reg_adam"] = (p, m, v)

    # one arena, data region = [gradients | parameters | touched marks]; at world 1 the barriers wait on the own flags only
    own, handle = c_void_p(), create_string_buffer(64)
    _lib.call("kp_peer_alloc", 3 * n * 4, byref(own), handle)
    try:
        data = torch.as_tensor(_RawCudaMemory(own.value + PeerArena.SIGNAL_BYTES, 3 * n), device=DEV)
        arenas = (c_void_p * 1)(own.value)
        for sparse in (False, True):
            data[:n].copy_(g0)
            data[n:2 * n].copy_(p0)
            data[2 * n:].view(torch.uint8)[: n // 32].fill_(1)
            m, v = m0.clone(), v0.clone()
            name = "kp_peer_sharded_adam_sparse" if sparse else "kp_peer_sharded_adam"
            offsets = (0, n, 2 * n) if sparse else (0, n)
            _lib.call(name, arenas, 0, 1, *offsets, n, c_void_p(m.data_ptr()), c_void_p(v.data_ptr()), lr, b1, b2, eps, wd, step,
                      gs, c_void_p(0), 0, _lib.stream_ptr())
            got[name] = (data[n:2 * n].clone(), m, v)
        torch.cuda.synchronize()
    finally:
        _lib.call("kp_peer_free", own)
    for name, (p, m, v) in got.items():
        assert torch.equal(p, ref[0]) and torch.equal(m, ref[1]) and torch.equal(v, ref[2]), name


def test_eval_mode_and_chunked_full_frame():
    """Eval path: deterministic samplers, last_sample background, chunked get_outputs_for_camera_ray_bundle."""
    from soccernerfs_b200.cameras.rays import RayBundle
    from tests.helpers import build_model
    from tests.test_oracle_golden import load_tiny_model

    g = load_golden("model_tiny")
    mp = load_tiny_model(g)
    model = build_model("tiny", mp, g["aabb"], DEV)
    model.eval()
    model.config.eval_num_rays_per_chunk = 40
    n = g["origins"].shape[0]
    h, w = 8, n // 8
    rb = RayBundle(origins=g["origins"].view(h, w, 3).to(DEV), directions=g["directions"].view(h, w, 3).to(DEV),
                   pixel_area=torch.ones(h, w, 1, device=DEV), times=g["times"].view(h, w, 1).to(DEV))
    out = model.get_outputs_for_camera_ray_bundle(rb)
    nears, fars = ko.aabb_collider(g["origins"], g["directions"], g["aabb"], 0.0)
    ref = ko.model_forward(mp, g["origins"], g["directions"], g["times"], nears, fars, None, training=False)
    assert out["rgb"].shape == (h, w, 3)
    assert rel_err(out["rgb"].view(-1, 3).cpu(), ref["rgb"].detach()) < 2e-4
    assert rel_err(out["accumulation"].view(-1, 1).cpu(), ref["accumulation"].detach()) < 2e-4
    assert rel_err(out["depth"].view(-1, 1).cpu(), ref["depth"].detach()) < 2e-4


def test_cuda_graph_train_step_matches_eager():
    """The CUDA-graph replay of the whole iteration (device-side LR / bias-correction / anneal tables) must follow
    the eager loop: same model, RNG-free samplers (train_stratified off, black background), 8 steps."""
    import copy

    from soccernerfs_b200.engine.trainer import TrainStep
    from tests.helpers import build_model, ray_bundle
    from tests.test_oracle_golden import load_tiny_model

    g = load_golden("model_tiny")
    mp = load_tiny_model(g)
    runs = {}
    for mode in ("eager", "graph"):
        model = build_model("tiny", mp, g["aabb"], DEV)
        model.config.background_color_train = "black"
        model.proposal_sampler.initial_sampler.train_stratified = False
        model.proposal_sampler.pdf_sampler.train_stratified = False
        step = TrainStep(model, max_steps=100, warm_up_end=4, use_cuda_graph=(mode == "graph"))
        losses = []
        for i in range(8):
            rb = ray_bundle(g["origins"], g["directions"], g["times"], DEV)
            out = step(rb, {"image": g["image"].to(DEV)})
            losses.append(float(out["loss"]))
        runs[mode] = (losses, [p.detach().clone() for p in model.parameters()])
        if mode == "graph":
            assert len(step._graphs) >= 1  # a graph was captured and replayed
    le, lg = runs["eager"][0], runs["graph"][0]
    assert le[-1] < le[1]  # it trains (step 0 has lr = 0 under the warm-up schedule)
    for a, b in zip(le, lg):
        assert abs(a - b) <= 2e-4 * abs(a), (le, lg)
    for a, b in zip(runs["eager"][1], runs["graph"][1]):
        if a.numel():
            assert rel_err(b, a) < 1e-2  # Adam normalises gradients: atomics-order noise on tiny gradients is amplified
    del copy


def test_branch_overlap_streams_do_not_change_the_step():
    """Regularisers and proposal-network backward on side streams (TrainStep(overlap_branches=True)) vs everything
    on one stream: same losses and parameters, eagerly and from the captured graph."""
    from soccernerfs_b200.engine.trainer import TrainStep
    from tests.helpers import build_model, ray_bundle
    from tests.test_oracle_golden import load_tiny_model

    g = load_golden("model_tiny")
    mp = load_tiny_model(g)
    runs = {}
    for mode in ("serial", "overlap", "overlap-graph"):
        model = build_model("tiny", mp, g["aabb"], DEV)
        model.config.background_color_train = "black"
        model.proposal_sampler.initial_sampler.train_stratified = False
        model.proposal_sampler.pdf_sampler.train_stratified = False
        step = TrainStep(model, max_steps=100, warm_up_end=4, use_cuda_graph=mode.endswith("graph"),
                         overlap_branches=mode != "serial")
        assert step.overlap == (mode != "serial")
        losses, regs = [], []
        for i in range(6):
            rb = ray_bundle(g["origins"], g["directions"], g["times"], DEV)
            out = step(rb, {"image": g["image"].to(DEV)})
            losses.append(float(out["loss"]))
            regs.append(float(out["space_tv_loss"]))
        torch.cuda.synchronize()
        runs[mode] = (losses, regs, [p.detach().clone() for p in model.parameters()])
    for mode in ("overlap", "overlap-graph"):
        for a, b in zip(runs["serial"][0], runs[mode][0]):
            assert abs(a - b) <= 2e-4 * abs(a), (mode, runs["serial"][0], runs[mode][0])
        for a, b in zip(runs["serial"][1], runs[mode][1]):
            assert abs(a - b) <= 2e-4 * abs(a) and a > 0
        for a, b in zip(runs["serial"][2], runs[mode][2]):
            if a.numel():
                assert rel_err(b, a) < 1e-2


def test_grad_sinks_match_autograd_accumulation():
    """Gradient-accumulation fusion (kernels accumulate straight into the flat bucket, autograd gets None) must give
    the same gradients as the plain autograd path, and must actually be active."""
    from soccernerfs_b200.distributed import GradBucket
    from tests.helpers import build_model, model_params_in_oracle_order, ray_bundle
    from tests.test_oracle_golden import load_tiny_model

    g = load_golden("model_tiny")
    mp = load_tiny_model(g)
    grads = {}
    for mode in ("autograd", "sink"):
        model = build_model("tiny", mp, g["aabb"], DEV)
        model.config.background_color_train = "black"
        model.proposal_sampler.initial_sampler.train_stratified = False
        model.proposal_sampler.pdf_sampler.train_stratified = False
        model.train()
        params = [p for ps in model.get_param_groups().values() for p in ps]
        if mode == "sink":
            bucket = GradBucket(params)
            bucket.attach_zeroed(sink=True)
        out = model(ray_bundle(g["origins"], g["directions"], g["times"], DEV))
        ld = model.get_loss_dict(out, {"image": g["image"].to(DEV)}, {})
        sum(ld.values()).backward()
        if mode == "sink":
            # autograd never replaced the bucket views: the kernels wrote into them directly
            assert all(p.grad.data_ptr() == v.data_ptr() for p, v in zip(bucket.params, bucket.views))
            assert float(bucket.flat.abs().sum()) > 0
        grads[mode] = [p.grad.detach().clone() for p in model_params_in_oracle_order(model)]
    for a, b in zip(grads["autograd"], grads["sink"]):
        assert rel_err(b, a) < 1e-5


def test_tile_sharded_eval_equals_unsharded():
    """config 5: a frame rendered as round-robin ray chunks by 3 'ranks' equals the single-process chunked render."""
    from soccernerfs_b200.cameras.rays import RayBundle
    from soccernerfs_b200.distributed import assemble_frame, render_frame_sharded
    from tests.helpers import build_model
    from tests.test_oracle_golden import load_tiny_model

    g = load_golden("model_tiny")
    model = build_model("tiny", load_tiny_model(g), g["aabb"], DEV)
    model.eval()
    model.config.eval_num_rays_per_chunk = 17
    n = g["origins"].shape[0]
    h, w = 8, n // 8
    rb = RayBundle(origins=g["origins"].view(h, w, 3).to(DEV), directions=g["directions"].view(h, w, 3).to(DEV),
                   pixel_area=torch.ones(h, w, 1, device=DEV), times=g["times"].view(h, w, 1).to(DEV))
    full = model.get_outputs_for_camera_ray_bundle(rb)
    pieces = [render_frame_sharded(model, rb, r, 3) for r in range(3)]
    assert sum(len(p) for p in pieces) == -(-n // 17) and all(len(p) > 0 for p in pieces)
    frame = assemble_frame(pieces, h, w)
    for k in ("rgb", "depth", "accumulation", "median_rgb"):
        assert torch.equal(frame[k], full[k]), k


def test_ray_generation_vs_reference_fixture():
    """(f2) kp_generate_rays vs rays produced by the reference's own Cameras: explicit (camera,row,col) triplets through
    the RayGenerator mirror, the generate_rays(camera_indices, coords) form, and one whole frame."""
    from soccernerfs_b200.cameras.cameras import Cameras
    from soccernerfs_b200.model_components.ray_generators import RayGenerator

    g = load_golden("raygen")
    h, w = (int(v) for v in g["hw"])
    cams = Cameras(g["c2w"].to(DEV), g["fx"].to(DEV), g["fy"].to(DEV), g["cx"].to(DEV), g["cy"].to(DEV), w, h,
                   times=g["times"].to(DEV))
    ri = g["ray_indices"].to(DEV)
    gen = RayGenerator(cams)
    coords = gen.image_coords.to(DEV)[ri[:, 1], ri[:, 2]]
    for rb in (gen(ri), cams.generate_rays(camera_indices=ri[:, 0:1], coords=coords)):
        assert torch.equal(rb.origins.cpu(), g["origins"]) and torch.equal(rb.times.cpu(), g["ray_times"])
        assert rel_err(rb.directions.cpu(), g["directions"]) < 1e-6
        assert rel_err(rb.pixel_area.cpu(), g["pixel_area"]) < 1e-5
        assert rel_err(rb.metadata["directions_norm"].cpu(), g["directions_norm"]) < 1e-6
        assert torch.equal(rb.camera_indices.cpu(), g["ray_indices"][:, 0:1])
    frame = cams.generate_rays(camera_indices=int(g["frame_cam"]), keep_shape=True)
    assert frame.origins.shape == (h, w, 3)
    assert torch.equal(frame.origins.cpu(), g["frame_origins"]) and torch.equal(frame.times.cpu(), g["frame_times"])
    assert rel_err(frame.directions.cpu(), g["frame_directions"]) < 1e-6
    assert rel_err(frame.pixel_area.cpu(), g["frame_pixel_area"]) < 1e-5
    # fraction of bit-identical direction components (the arithmetic follows the reference's order)
    same = (frame.directions.cpu() == g["frame_directions"]).float().mean()
    assert same > 0.9, float(same)


def test_lens_ray_generation_vs_reference_fixture():
    """(f2) kp_generate_rays' lens kernel vs rays of the reference's own Cameras (fixture raygen_lens): OpenCV distortion
    undone by 10 Newton iterations, fisheye and equirectangular direction models, the three camera types mixed in one
    batch; explicit triplets, whole frames through the tile form, disable_distortion, and the dataparsers' perspective
    batch with one shared distortion row.  The undistortion is rounded operation by operation in the reference's order,
    so perspective rays differ from the reference only where the plain kernel's do (rotation sum / norm); sin / cos of
    the fisheye and equirectangular models are CUDA's instead of the host libm's."""
    from soccernerfs_b200.cameras.cameras import Cameras, CameraType

    g = load_golden("raygen_lens")
    h, w = (int(v) for v in g["hw"])
    args = [g[k].to(DEV) for k in ("c2w", "fx", "fy", "cx", "cy")]
    cams = Cameras(*args, w, h, times=g["times"].to(DEV), distortion_params=g["dist"], camera_type=g["types"])
    ri = g["ray_indices"].to(DEV)
    coords = cams.get_image_coords().to(DEV)[ri[:, 1], ri[:, 2]]
    for rb in (cams.generate_rays_from_indices(ri), cams.generate_rays(camera_indices=ri[:, 0:1], coords=coords)):
        assert torch.equal(rb.origins.cpu(), g["origins"]) and torch.equal(rb.times.cpu(), g["ray_times"])
        assert rel_err(rb.directions.cpu(), g["directions"]) < 1e-6
        assert rel_err(rb.pixel_area.cpu(), g["pixel_area"]) < 1e-5
        assert rel_err(rb.metadata["directions_norm"].cpu(), g["directions_norm"]) < 1e-6
    rb = cams.generate_rays(camera_indices=ri[:, 0:1], coords=coords, disable_distortion=True)
    assert rel_err(rb.directions.cpu(), g["nodist_directions"]) < 1e-6 and rel_err(rb.pixel_area.cpu(), g["nodist_pixel_area"]) < 1e-5
    for c in (0, 3, 4, 5):
        frame = cams.generate_rays(camera_indices=c, keep_shape=True)
        assert frame.directions.shape == (h, w, 3)
        assert rel_err(frame.directions.cpu(), g[f"frame{c}_directions"]) < 1e-6, c
        assert rel_err(frame.metadata["directions_norm"].cpu(), g[f"frame{c}_directions_norm"]) < 1e-6, c
        ref = g[f"frame{c}_pixel_area"]
        assert rel_err(frame.pixel_area.cpu(), ref) < 1e-5, c  # the bar's norm (max error / max value)
        # stricter than the bar, per element: a product of two differences of unit vectors, 1e-2 each, so a 1-ulp
        # direction difference is 1e-5 of it (measured 1.5e-5 with the kernel body compiled for the host)
        assert ((frame.pixel_area.cpu() - ref).abs() / ref.abs().clamp_min(1e-12)).max() < 2e-4, c
    persp = Cameras(*args, w, h, times=g["times"].to(DEV), distortion_params=g["dist"][0], camera_type=CameraType.PERSPECTIVE)
    assert persp._cam_types is None and persp._distortion is not None
    rb = persp.generate_rays_from_indices(ri)
    assert rel_err(rb.directions.cpu(), g["persp_directions"]) < 1e-6 and rel_err(rb.pixel_area.cpu(), g["persp_pixel_area"]) < 1e-5
    same = (rb.directions.cpu() == g["persp_directions"]).float().mean()
    assert same > 0.85, float(same)
    # an all-zero distortion table and all-perspective types are the plain kernel: bit-identical rays
    g0 = load_golden("raygen")
    a0 = [g0[k].to(DEV) for k in ("c2w", "fx", "fy", "cx", "cy")]
    h0, w0 = (int(v) for v in g0["hw"])
    plain = Cameras(*a0, w0, h0, times=g0["times"].to(DEV))
    tiny = Cameras(*a0, w0, h0, times=g0["times"].to(DEV), distortion_params=torch.full((6,), 1e-30),
                   camera_type=torch.ones(5, 1, dtype=torch.int64))
    assert tiny._distortion is not None
    ra, rb = plain.generate_rays_from_indices(g0["ray_indices"].to(DEV)), tiny.generate_rays_from_indices(g0["ray_indices"].to(DEV))
    assert torch.equal(ra.directions, rb.directions) and torch.equal(ra.pixel_area, rb.pixel_area)


def test_depth_supervision_goes_through_every_sampling_level():
    """kplanes.py:395-410 / :447-449: with a depth image in the batch the depth loss is the mean over ALL levels (proposal
    levels included) of losses.depth_loss, scaled by its coefficient; the step with such a batch is not graph-capturable
    (only origins / directions / times / image have static buffers) and must take the eager iteration, not drop the key."""
    from soccernerfs_b200.engine.trainer import TrainStep
    from soccernerfs_b200.model_components.losses import depth_loss
    from tests.helpers import build_model, ray_bundle
    from tests.test_oracle_golden import load_tiny_model

    g = load_golden("model_tiny")
    model = build_model("tiny", load_tiny_model(g), g["aabb"], DEV)
    model.train()
    n = g["origins"].shape[0]
    rb = ray_bundle(g["origins"], g["directions"], g["times"], DEV)
    rb.metadata = {"directions_norm": torch.ones(n, 1, device=DEV)}
    batch = {"image": g["image"].to(DEV), "depth_image": (1.0 + torch.rand(n, 1, generator=torch.Generator().manual_seed(1))).to(DEV)}
    torch.manual_seed(0)
    outputs = model(rb)
    metrics = model.get_metrics_dict(outputs, batch)
    sigma = model._get_sigma().to(DEV)
    ref = sum(depth_loss(weights=w, ray_samples=rs, termination_depth=batch["depth_image"], predicted_depth=outputs["depth"],
                         sigma=sigma, directions_norm=outputs["directions_norm"], is_euclidean=model.config.is_euclidean_depth,
                         depth_loss_type=model.config.depth_loss_type)
              for w, rs in zip(outputs["weights_list"], outputs["ray_samples_list"])) / len(outputs["weights_list"])
    assert len(outputs["weights_list"]) == model.config.num_proposal_iterations + 1
    assert rel_err(metrics["depth_loss"].detach(), ref.detach()) < 1e-6 and float(ref.detach()) > 0
    losses = model.get_loss_dict(outputs, batch, metrics)
    assert rel_err(losses["depth_loss"], model.config.loss_coefficients["depth_loss"] * ref) < 1e-6
    step = TrainStep(model, max_steps=100, warm_up_end=4, use_cuda_graph=True)
    try:
        assert not step._graphable(rb, batch)
        out = step(rb, batch)
        assert "depth_loss" in out and bool(torch.isfinite(out["loss"]))
    finally:
        step.close()


def test_frame_renderer_equals_chunked_camera_bundle():
    """config 5: the tile queue (device ray generation + chunked forward + async copies to pinned frames) gives the
    same image as generate_rays(keep_shape=True) -> get_outputs_for_camera_ray_bundle, also when 3 ranks share it."""
    from soccernerfs_b200.cameras.cameras import Cameras
    from soccernerfs_b200.engine.frame_renderer import FrameRenderer
    from tests.helpers import build_model
    from tests.test_oracle_golden import load_tiny_model

    gm = load_golden("model_tiny")
    model = build_model("tiny", load_tiny_model(gm), gm["aabb"], DEV)
    model.eval()
    h, w = 24, 40
    c2w = torch.tensor([[[1.0, 0, 0, 0.1], [0, 1.0, 0, -0.2], [0, 0, 1.0, 2.5]]])
    cams = Cameras(c2w.to(DEV), 40.0, 40.0, w / 2, h / 2, w, h, times=torch.tensor([0.4]).to(DEV))
    full = cams.generate_rays(camera_indices=0, keep_shape=True)
    model.config.eval_num_rays_per_chunk = 200
    with torch.no_grad():
        ref = model.get_outputs_for_camera_ray_bundle(full)
    one = FrameRenderer(model, cams, chunk=200).render(0)  # one CUDA-graph replay per tile (two tile sizes: 200 and 160)
    eager = FrameRenderer(model, cams, chunk=200, use_cuda_graph=False, ray_tile=0).render(0)
    for k in ("rgb", "depth", "accumulation"):
        assert one[k].shape[:2] == (h, w) and one[k].is_pinned()
        assert torch.equal(one[k], ref[k].cpu()), k
        assert torch.equal(eager[k], ref[k].cpu()), k
    again = FrameRenderer(model, cams, chunk=200)
    again.render(0)
    second = again.render(0)  # replays of the captured tiles (static index buffer refilled per tile)
    for k in ("rgb", "depth", "accumulation"):
        assert torch.equal(second[k], ref[k].cpu()), k
    total = {k: torch.zeros_like(v) for k, v in one.items()}
    for r in range(3):
        part = FrameRenderer(model, cams, chunk=200, rank=r, world=3).render(0)
        for k in total:
            total[k] += part[k]
    for k in total:
        assert torch.equal(total[k], one[k]), k


def test_crop_box_render_vs_reference_fixture():
    """(f2) crop-box rendering, scripts/render.py:101-106: kp_intersect_aabb bit-identical to the reference's slab test
    (NaN / 1e10 / infinite-slab rays included), Cameras.generate_rays(aabb_box=...) stores the same nears / fars as the
    reference's Cameras for a whole frame, the model keeps them (the collider only fills missing bounds,
    scene_colliders.py:41-45), and the tile queue with ``aabb_box`` renders the same image as the bundle form."""
    from soccernerfs_b200 import ops
    from soccernerfs_b200.cameras.cameras import Cameras
    from soccernerfs_b200.data.scene_box import SceneBox
    from soccernerfs_b200.engine.frame_renderer import FrameRenderer
    from tests.helpers import build_model
    from tests.test_oracle_golden import _same_with_nans, load_tiny_model

    g = load_golden("raygen_crop")
    t_min, t_max = ops.intersect_aabb(g["origins"].to(DEV), g["directions"].to(DEV), g["aabb"].tolist())
    assert _same_with_nans(t_min.cpu(), g["t_min"]) and _same_with_nans(t_max.cpu(), g["t_max"])
    e0, e1 = ops.intersect_aabb(torch.zeros(0, 3, device=DEV), torch.zeros(0, 3, device=DEV), g["aabb"].tolist())
    assert e0.shape == (0,) and e1.shape == (0,)
    # the reference's own property test (tests/utils/test_aabb_intersection.py:120-147): entry and exit points of the
    # rays that hit lie on the box's boundary
    hit = (g["t_min"] < 1e10) & ~torch.isnan(g["t_min"])
    o, d, a = g["origins"][hit], g["directions"][hit], g["aabb"]
    assert int(hit.sum()) > 10 and bool((t_max.cpu()[hit] >= t_min.cpu()[hit]).all())
    for t in (t_max.cpu()[hit],):  # exits are always on a face (entries are 0 for origins inside the box)
        p = o + d * t[:, None]
        inside = ((p >= a[:3] - 1e-4) & (p <= a[3:] + 1e-4)).all(dim=-1)
        on_face = (torch.minimum((p - a[:3]).abs(), (p - a[3:]).abs()).min(dim=-1).values < 1e-4)
        assert bool((inside & on_face).all())

    r = load_golden("raygen")
    h, w = (int(v) for v in r["hw"])
    cams = Cameras(*[r[k].to(DEV) for k in ("c2w", "fx", "fy", "cx", "cy")], w, h, times=r["times"].to(DEV))
    cam = int(g["frame_cam"])
    box = SceneBox(aabb=g["box"].to(DEV))
    frame = cams.generate_rays(camera_indices=cam, aabb_box=box)
    assert frame.nears.shape == (h, w, 1) and frame.fars.shape == (h, w, 1)
    # our directions differ from the reference's in the last bit on ~10 % of the rays, so do the bounds: 1e-5 relative
    # where both hit, and the same hit / miss decision except on rays within rounding of grazing the box
    ours_hit, ref_hit = frame.nears.cpu() < 1e10, g["frame_nears"] < 1e10
    both = ours_hit & ref_hit
    assert float((ours_hit != ref_hit).float().mean()) < 2e-3
    assert rel_err(frame.nears.cpu()[both], g["frame_nears"][both]) < 1e-5 and rel_err(frame.fars.cpu()[both], g["frame_fars"][both]) < 1e-5
    # given the reference's rays the bounds are bit-identical
    t0, t1 = ops.intersect_aabb(r["frame_origins"].reshape(-1, 3).to(DEV), r["frame_directions"].reshape(-1, 3).to(DEV), Cameras.box6(box))
    assert torch.equal(t0.cpu().view(h, w, 1), g["frame_nears"]) and torch.equal(t1.cpu().view(h, w, 1), g["frame_fars"])

    gm = load_golden("model_tiny")
    model = build_model("tiny", load_tiny_model(gm), gm["aabb"], DEV)
    model.eval()
    hh, ww = 24, 40
    c2w = torch.tensor([[[1.0, 0, 0, 0.1], [0, 1.0, 0, -0.2], [0, 0, 1.0, 2.5]]])
    cams = Cameras(c2w.to(DEV), 40.0, 40.0, ww / 2, hh / 2, ww, hh, times=torch.tensor([0.4]).to(DEV))
    crop = SceneBox(aabb=torch.tensor([[-0.4, -0.5, -0.3], [0.5, 0.2, 0.6]]))
    full = cams.generate_rays(camera_indices=0, aabb_box=crop)
    frac = float((full.nears < 1e10).float().mean())
    assert 0.02 < frac < 0.9, frac
    model.config.eval_num_rays_per_chunk = 200
    with torch.no_grad():
        ref = model.get_outputs_for_camera_ray_bundle(full)
        uncropped = model.get_outputs_for_camera_ray_bundle(cams.generate_rays(camera_indices=0))
    kept = model.collider(full)  # bounds already set: the collider returns the bundle as it is
    assert kept.nears is full.nears and kept.fars is full.fars
    assert not torch.equal(ref["rgb"], uncropped["rgb"])
    for graph in (True, False):
        out = FrameRenderer(model, cams, chunk=200, use_cuda_graph=graph, aabb_box=crop).render(0)
        for k in ("rgb", "depth", "accumulation"):
            assert torch.equal(out[k], ref[k].cpu()), (k, graph)


def test_compositing_edge_shapes_and_non_finite_densities():
    """Ragged / degenerate inputs the reference code accepts: one ray, one sample; S not a multiple of the warp; an
    infinite density (alpha = 1, everything behind it gets weight 0) and a NaN (nan_to_num -> 0), rays.py:137-149."""
    from soccernerfs_b200 import ops

    gen = torch.Generator().manual_seed(21)
    for n, s in ((1, 1), (3, 33), (5, 7)):
        deltas = torch.rand(n, s, generator=gen) + 0.01
        dens = torch.rand(n, s, generator=gen) * 5
        if s > 3:
            dens[0, 2] = float("inf")
            dens[-1, 1] = float("nan")
        ref = ko.get_weights(deltas[..., None], dens[..., None])[..., 0]
        w = ops.get_weights(deltas.to(DEV), dens.to(DEV))
        assert w.shape == (n, s) and bool(torch.isfinite(w).all())
        finite_rows = torch.isfinite(dens).all(-1)
        assert rel_err(w.cpu()[finite_rows], ref[finite_rows]) < TOL if bool(finite_rows.any()) else True
        if s > 3:
            assert float(w[0, 2]) == pytest.approx(float(ref[0, 2]), rel=1e-5) and bool((w[0, 3:] == 0).all())
            assert float(w[-1, 1]) == 0.0  # the NaN sample itself
        rgb = torch.rand(n, s, 3, generator=gen)
        comp = ops.composite_rgb(w, rgb.to(DEV), torch.zeros(n, 3, device=DEV))
        assert rel_err(comp.cpu(), (w.cpu()[..., None] * rgb).sum(-2)) < TOL
        assert rel_err(ops.accumulate(w).cpu(), w.cpu().sum(-1)) < TOL
        idx = ops.median_index(w)
        assert torch.equal(idx.cpu(), ko.median_index(w.cpu()[..., None])[:, 0])


def test_trainer_checkpoint_resume():
    """TrainStep.state_dict / load_state_dict (the reference's checkpoint layout, trainer.py:352-380): 3 steps, save,
    3 more steps == load into a fresh trainer and run the same 3 steps -- eagerly and with the CUDA graph."""
    import copy

    from soccernerfs_b200.engine.trainer import TrainStep
    from tests.helpers import build_model, ray_bundle
    from tests.test_oracle_golden import load_tiny_model

    g = load_golden("model_tiny")
    mp = load_tiny_model(g)

    def make(graph):
        model = build_model("tiny", mp, g["aabb"], DEV)
        model.config.background_color_train = "black"
        model.proposal_sampler.initial_sampler.train_stratified = False
        model.proposal_sampler.pdf_sampler.train_stratified = False
        return model, TrainStep(model, max_steps=100, warm_up_end=4, use_cuda_graph=graph)

    def run(step, n):
        out = None
        for _ in range(n):
            out = step(ray_bundle(g["origins"], g["directions"], g["times"], DEV), {"image": g["image"].to(DEV)})
        return float(out["loss"])

    for graph in (False, True):
        model_a, step_a = make(graph)
        run(step_a, 3 if not graph else 5)  # graph mode: past the two eager visits, so a graph exists when saving
        saved = copy.deepcopy(step_a.state_dict())
        assert saved["step"] == step_a.step and "_model.field.grids.0.0" in saved["pipeline"]
        assert set(saved["optimizers"]) == {"proposal_networks", "fields"}
        loss_a = run(step_a, 3)
        model_b, step_b = make(graph)
        step_b.load_state_dict(saved)
        assert step_b.step == saved["step"]
        loss_b = run(step_b, 3)
        assert abs(loss_a - loss_b) <= 2e-4 * abs(loss_a), (graph, loss_a, loss_b)
        for pa, pb in zip(model_a.parameters(), model_b.parameters()):
            if pa.numel():
                assert rel_err(pb, pa) < 1e-2


def test_cfg4_piecewise_single_jitter_samplers_vs_reference_fixture():
    """BASELINE config 4 (nerfplayer-nerfacto shares only the samplers + compositing): piecewise initial sampler and
    PDF resampling with one jitter per ray, through the sampler modules, vs the reference's own classes; expected depth."""
    from soccernerfs_b200.cameras.rays import RayBundle
    from soccernerfs_b200.model_components.ray_samplers import PDFSampler, UniformLinDispPiecewiseSampler
    from soccernerfs_b200.model_components.renderers import DepthRenderer
    from tests.helpers import rand_queue

    g = load_golden("samplers_cfg4")
    n = g["origins"].shape[0]
    for mode in ("train", "eval"):
        ini = UniformLinDispPiecewiseSampler(single_jitter=True)
        pdf = PDFSampler(include_original=False, single_jitter=True)
        ini.train(mode == "train")
        pdf.train(mode == "train")
        pdf.record_inds = True
        rb = RayBundle(origins=g["origins"].to(DEV), directions=g["directions"].to(DEV), pixel_area=torch.ones(n, 1, device=DEV),
                       times=g["times"].to(DEV), nears=g["nears"].to(DEV), fars=g["fars"].to(DEV))
        queue = [g[f"{mode}_t_rand"], g[f"{mode}_u_rand"]] if mode == "train" else []
        with rand_queue(queue, DEV):
            rs0 = ini(rb, num_samples=64)
            rs1 = pdf(rb, rs0, g[f"{mode}_weights"].to(DEV), num_samples=24)
        bins0 = torch.cat([rs0.spacing_starts[..., 0], rs0.spacing_ends[..., -1:, 0]], -1).cpu()
        assert torch.equal(bins0, g[f"{mode}_bins0"])
        # euclidean edges: 1 / (2 - 2x) etc. with IEEE division, like torch's CPU ops
        assert (rs0.frustums.starts[..., 0].cpu() - g[f"{mode}_starts0"]).abs().max() < 1e-6
        assert (rs0.frustums.starts[..., 0].cpu() == g[f"{mode}_starts0"]).float().mean() > 0.99
        assert (rs0.frustums.ends[..., 0].cpu() - g[f"{mode}_ends0"]).abs().max() < 1e-6
        bins1 = torch.cat([rs1.spacing_starts[..., 0], rs1.spacing_ends[..., -1:, 0]], -1).cpu()
        assert torch.equal(pdf.last_inds.cpu(), g[f"{mode}_inds1"])  # bit-exact indices and spacing bins on every ray
        assert torch.equal(bins1, g[f"{mode}_bins1"])
        rel = (rs1.frustums.starts[..., 0].cpu() - g[f"{mode}_starts1"]).abs() / g[f"{mode}_starts1"].abs().clamp_min(1e-3)
        assert rel.max() < 2e-5  # the disparity branch amplifies a 1-ulp spacing difference near the far plane
        depth = DepthRenderer(method="expected")(weights=g[f"{mode}_w1"].to(DEV), ray_samples=rs1)
        assert rel_err(depth.cpu(), g[f"{mode}_depth_expected"]) < 1e-4


def test_fused_regularizer_sweep_matches_autograd_path():
    """kp_plane_reg_fused in the training step's form (one sweep: values + gradient written into the sinks) vs the
    autograd path (ops.plane_reg_sums: a sums-only sweep forward, gradient-only sweeps backward): same six scaled loss
    values, same plane gradients; accumulate mode adds on top."""
    from soccernerfs_b200.distributed import GradBucket
    from soccernerfs_b200.models.kplanes import scale_dict
    from tests.helpers import build_model
    from tests.test_oracle_golden import load_tiny_model

    g = load_golden("model_tiny")
    model = build_model("tiny", load_tiny_model(g), g["aabb"], DEV)
    planes = model.regularized_planes()
    ref = scale_dict(model.regularizer_losses(), model.config.loss_coefficients)
    sum(ref.values()).backward()
    ref_grads = [p.grad.detach().clone() for p in planes]
    for p in model.parameters():
        p.grad = None
    bucket = GradBucket([p for ps in model.get_param_groups().values() for p in ps])
    bucket.attach_zeroed(sink=True, skip=frozenset(id(p) for p in planes))
    bucket.flat.fill_(123.0)  # the sweep must overwrite every plane element (it replaces the memset)
    vals = model.regularizers_into_grads(accumulate=False)
    for k, v in ref.items():
        assert rel_err(vals[k], v.detach()) < 1e-6, k
    for p, r in zip(planes, ref_grads):
        assert rel_err(p.grad, r) < 1e-6
    model.regularizers_into_grads(accumulate=True)
    for p, r in zip(planes, ref_grads):
        assert rel_err(p.grad, 2 * r) < 1e-6


def test_plane_reg_sums_and_gradients_vs_oracle_across_tiles():
    """ops.plane_reg_sums and its autograd gradients against the torch formulas of the oracle (compute_plane_tv,
    compute_plane_smoothness, |1 - t|) in float64, for every term combination the model uses.  The planes cross the
    sweep's 32-row and 256-float4 tile edges (C = 8, 16 and 32); half of them carry a gradient sink, so the accumulating
    and the writing backward sweeps both run in one backward."""
    from soccernerfs_b200 import ops

    torch.manual_seed(11)
    T_H, T_W, T_SMOOTH, T_L1 = 1, 2, 4, 8
    shapes = [(1, 32, 150, 70), (1, 32, 100, 64), (1, 8, 130, 200), (1, 8, 67, 128), (1, 32, 5, 3), (1, 16, 64, 64)]
    base = [0.3 + 0.4 * torch.rand(sh) for sh in shapes]  # 1 - t keeps its sign: |1 - t| is differentiable everywhere

    def oracle_sums(t):  # [4] float64: the four sums whose means the reference's losses take
        _, c, h, w = t.shape
        w_tv = ko.compute_plane_tv(t, only_w=True)
        return torch.stack([(ko.compute_plane_tv(t) - w_tv) * (c * (h - 1) * w), w_tv * (c * h * (w - 1)),
                            ko.compute_plane_smoothness(t) * (c * (h - 2) * w), torch.abs(1 - t).sum()])

    for combo in (T_H | T_W, T_W, T_SMOOTH, T_L1, T_W | T_SMOOTH | T_L1):
        mask = torch.tensor([(combo >> i) & 1 for i in range(4)], dtype=torch.float64)
        weights = torch.rand(len(shapes), 4, dtype=torch.float64) * mask
        planes = [ops.as_channel_last(b.to(DEV)).requires_grad_(True) for b in base]
        for p in planes[::2]:
            p._kp_grad_sink = torch.full_like(p, 0.25, memory_format=torch.preserve_format)
            p.grad = p._kp_grad_sink
        sums = ops.plane_reg_sums(planes, [combo] * len(planes))
        (sums * weights.float().to(DEV)).sum().backward()
        ref_planes = [b.double().requires_grad_(True) for b in base]
        ref = torch.stack([oracle_sums(t) for t in ref_planes]) * mask
        (ref * weights).sum().backward()
        got = sums.detach().cpu().double()
        for i in range(len(planes)):
            for k in range(4):
                assert rel_err(got[i, k], ref[i, k].detach()) < TOL, (combo, i, k)
            grad = planes[i].grad - 0.25 if i % 2 == 0 else planes[i].grad
            assert rel_err(grad.cpu(), ref_planes[i].grad) < TOL, (combo, i)
        for p in planes[::2]:
            del p._kp_grad_sink


def test_plane_reg_adam_matches_regulariser_sweep_plus_adam():
    """(f1) kp_plane_reg_adam -- regulariser stencil + Adam in one in-place streaming pass with a halo snapshot -- against
    the two-pass path (kp_plane_reg_fused adds the regulariser gradient, kp_adam_multi steps): same sums, same planes and
    moments after two steps, gradient buffers left zeroed.  Shapes cross tile boundaries in both directions (rows not a
    multiple of 64, rows of 256+ float4, C = 8 and 32) so every halo path is exercised."""
    from soccernerfs_b200 import ops

    torch.manual_seed(3)
    T_H, T_W, T_SMOOTH, T_L1 = 1, 2, 4, 8
    specs = [((1, 32, 150, 70), T_H | T_W), ((1, 32, 100, 64), T_W | T_SMOOTH | T_L1), ((1, 8, 130, 200), T_H | T_W),
             ((1, 8, 67, 128), T_W | T_SMOOTH | T_L1), ((1, 32, 5, 3), T_H | T_W), ((1, 16, 64, 64), T_W | T_SMOOTH | T_L1)]
    planes = [(0.3 + 0.2 * torch.rand(sh, device=DEV)).contiguous(memory_format=torch.channels_last) for sh, _ in specs]
    terms = [t for _, t in specs]
    coef = (torch.rand(len(planes), 4, device=DEV) * 1e-2).contiguous()
    lr, b1, b2, eps = 1e-2, 0.9, 0.999, 1e-12

    def fresh():
        return ([p.clone(memory_format=torch.preserve_format) for p in planes],
                [torch.zeros_like(p, memory_format=torch.preserve_format) for p in planes],
                [torch.zeros_like(p, memory_format=torch.preserve_format) for p in planes])

    pa, ma, va = fresh()
    pb, mb, vb = fresh()
    scratch = torch.empty(ops.plane_reg_adam_scratch_bytes(planes), dtype=torch.uint8, device=DEV)
    gb = [torch.zeros_like(p, memory_format=torch.preserve_format) for p in planes]
    for step in (1, 2):
        data = [1e-3 * torch.randn_like(p, memory_format=torch.preserve_format) for p in planes]
        # two passes: the regulariser sweep adds onto the data gradient, then Adam
        ga = [d.clone(memory_format=torch.preserve_format) * 0.5 for d in data]
        sums_a = ops.plane_reg_fused(pa, terms, coef, ga, accumulate=True)
        ops.adam_multi_(pa, ga, ma, va, lr, b1, b2, eps, 0.0, step, 1.0)
        # one pass: data gradient scaled by grad_scale inside, regulariser gradient from the pre-update planes
        for g_, d in zip(gb, data):
            assert float(g_.abs().max()) == 0.0  # zeroed by the previous pass
            g_.copy_(d)
        sums_b = torch.zeros(len(planes), 4, dtype=torch.float64, device=DEV)
        ops.plane_reg_adam_(pb, gb, mb, vb, terms, coef, lr, b1, b2, eps, 0.0, step, 0.5, scratch, sums=sums_b, zero_grads=True)
        assert rel_err(sums_b.float(), sums_a.float()) < 1e-6
        for i in range(len(planes)):
            assert rel_err(mb[i], ma[i]) < 1e-5, (step, i)
            assert rel_err(vb[i], va[i]) < 1e-5, (step, i)
            assert float((pb[i] - pa[i]).abs().max()) < 1e-5 * lr * 100, (step, i)


def test_fused_regularizer_sweep_write_range_and_touched_marks():
    """The two pieces the sparse gradient exchange adds to single-GPU kernels: (1) kp_plane_reg_fused_range writes the
    gradient only inside a per-plane float4 range (sums unchanged); (2) kp_hexplane_bwd_flags marks exactly the texels that
    received a reduction and produces the same gradients as the unmarked scatter."""
    from soccernerfs_b200 import ops

    torch.manual_seed(5)
    specs = [((1, 32, 70, 40), 3), ((1, 32, 30, 64), 14), ((1, 8, 50, 128), 3)]
    planes = [(0.3 + 0.2 * torch.rand(sh, device=DEV)).contiguous(memory_format=torch.channels_last) for sh, _ in specs]
    terms = [t for _, t in specs]
    coef = (torch.rand(len(planes), 4, device=DEV) * 1e-2).contiguous()
    full = [torch.zeros_like(p, memory_format=torch.preserve_format) for p in planes]
    sums_full = ops.plane_reg_fused(planes, terms, coef, full, accumulate=False)
    rng = torch.tensor([[100, 5000], [0, 0], [37, 12000]], dtype=torch.int64, device=DEV)
    part = [torch.full_like(p, 7.0, memory_format=torch.preserve_format) for p in planes]
    sums_part = ops.plane_reg_fused(planes, terms, coef, part, accumulate=False, write_range=rng)
    assert torch.equal(sums_full, sums_part)
    for f, q, (a, b) in zip(full, part, rng.tolist()):
        fl = f.permute(0, 2, 3, 1).reshape(-1, 4)  # physical order, float4 rows
        ql = q.permute(0, 2, 3, 1).reshape(-1, 4)
        assert torch.equal(ql[a:b], fl[a:b])
        assert bool((ql[:a] == 7.0).all()) and bool((ql[b:] == 7.0).all())

    # (1b) shard form: the SUMS are restricted to the range as well, so the shares of a partition add up to the full sums
    # (every term counted exactly once), and the gradient inside each range equals the full sweep's
    sizes4 = [p.numel() // 4 for p in planes]
    cuts = [[0, n4 // 3 + 5, 2 * n4 // 3 - 7, n4] for n4 in sizes4]
    total = torch.zeros_like(sums_full)
    for r in range(3):
        rng_r = torch.tensor([[c_[r], c_[r + 1]] for c_ in cuts], dtype=torch.int64, device=DEV)
        part_r = [torch.full_like(p, 7.0, memory_format=torch.preserve_format) for p in planes]
        total += ops.plane_reg_fused(planes, terms, coef, part_r, accumulate=False, write_range=rng_r, sums_in_range=True)
        for f, q, (a, b) in zip(full, part_r, rng_r.tolist()):
            fl, ql = f.permute(0, 2, 3, 1).reshape(-1, 4), q.permute(0, 2, 3, 1).reshape(-1, 4)
            assert torch.equal(ql[a:b], fl[a:b])
            assert bool((ql[:a] == 7.0).all()) and bool((ql[b:] == 7.0).all())
    assert torch.allclose(total, sums_full, rtol=1e-6, atol=0.0), (total, sums_full)

    # (2) marks
    n, c = 3000, 32
    ms = [[(torch.rand(1, c, h, w, device=DEV)).contiguous(memory_format=torch.channels_last).requires_grad_(True)
           for (w, h) in ((24, 20), (24, 16), (24, 9), (20, 16), (20, 9), (16, 9))]]
    pts = torch.rand(n, 4, device=DEV) * 2 - 1
    gout = torch.randn(n, c, device=DEV)
    feats = ops.hexplane_features(ms, ops.points_from_pts(pts), concat=True)
    ref = torch.autograd.grad(feats, ms[0], gout)
    sinks, marks = [], []
    for p in ms[0]:
        p._kp_grad_sink = torch.zeros_like(p, memory_format=torch.preserve_format)
        p.grad = p._kp_grad_sink  # a sink is honoured only while it is the parameter's .grad
        p._kp_touched = torch.zeros(p.shape[2] * p.shape[3], dtype=torch.uint8, device=DEV)
        sinks.append(p._kp_grad_sink)
        marks.append(p._kp_touched)
    feats = ops.hexplane_features(ms, ops.points_from_pts(pts), concat=True)
    feats.backward(gout)
    for r, s_, m_ in zip(ref, sinks, marks):
        assert rel_err(s_, r) < 1e-5
        touched = (s_.permute(0, 2, 3, 1).reshape(-1, c) != 0).any(dim=1)
        assert bool((m_.bool() | ~touched).all())  # every texel that holds a gradient is marked
        assert int(m_.max()) == 1 and int(m_.bool().sum()) <= 4 * n
    for p in ms[0]:
        del p._kp_grad_sink, p._kp_touched


def test_train_step_with_and_without_fused_regularizers():
    """TrainStep(fuse_regularizers=True) (no memset of the planes' gradients, one regulariser sweep) follows the
    two-sweep step: same losses over 6 steps, eagerly and from the graph."""
    from soccernerfs_b200.engine.trainer import TrainStep
    from tests.helpers import build_model, ray_bundle
    from tests.test_oracle_golden import load_tiny_model

    g = load_golden("model_tiny")
    mp = load_tiny_model(g)
    runs = {}
    for mode in ("two-sweep", "fused", "fused-serial", "fused-graph", "reg-adam", "reg-adam-graph"):
        model = build_model("tiny", mp, g["aabb"], DEV)
        model.config.background_color_train = "black"
        model.proposal_sampler.initial_sampler.train_stratified = False
        model.proposal_sampler.pdf_sampler.train_stratified = False
        step = TrainStep(model, max_steps=100, warm_up_end=4, use_cuda_graph=mode.endswith("graph"),
                         overlap_branches=mode != "fused-serial", fuse_regularizers=mode != "two-sweep",
                         fuse_reg_adam=mode.startswith("reg-adam"))
        assert (step._reg_written is not None) == (mode != "two-sweep")
        assert (step._reg_adam is not None) == mode.startswith("reg-adam")
        losses = []
        for i in range(6):
            out = step(ray_bundle(g["origins"], g["directions"], g["times"], DEV), {"image": g["image"].to(DEV)})
            losses.append((float(out["loss"]), float(out["space_tv_loss"]), float(out["time_smoothness_proposal_loss"])))
        torch.cuda.synchronize()
        runs[mode] = (losses, [p.detach().clone() for p in model.parameters()])
        step.close()
    for mode in ("fused", "fused-serial", "fused-graph", "reg-adam", "reg-adam-graph"):
        for a, b in zip(runs["two-sweep"][0], runs[mode][0]):
            for x, y in zip(a, b):
                assert abs(x - y) <= 2e-4 * abs(x) and x > 0, (mode, a, b)
        for a, b in zip(runs["two-sweep"][1], runs[mode][1]):
            if a.numel():
                assert rel_err(b, a) < 1e-2


def test_reference_checkpoint_loads_on_device():
    """f3 on the GPU: a reference-layout pipeline state (planes NCHW-contiguous, flat tcnn params) is repacked into the
    channel-last CUDA model through kp_repack_nchw_to_hwc, exported back through kp_repack_hwc_to_nchw, and the loaded
    model renders exactly like the one that produced the checkpoint."""
    from soccernerfs_b200.utils.checkpoint import load_reference_state_dict, to_reference_state_dict
    from tests.helpers import build_model, ray_bundle
    from tests.test_oracle_golden import load_tiny_model

    g = load_golden("model_tiny")
    mp = load_tiny_model(g)
    a = build_model("tiny", mp, g["aabb"], DEV)
    torch.manual_seed(5)
    b = build_model("tiny", mp, g["aabb"], DEV)
    with torch.no_grad():
        for p in b.parameters():
            if p.requires_grad:
                p.add_(torch.randn_like(p))
    sd = to_reference_state_dict(a)  # CUDA tensors, reference layouts
    plane = sd["_model.field.grids.1.2"]
    assert plane.is_cuda and plane.is_contiguous() and torch.equal(plane, a.field.grids[1][2].detach().contiguous())
    unused = load_reference_state_dict(b, {"step": 3, "pipeline": sd})
    assert unused == ["_model.field.direction_encoder.params"]
    for (na, pa), (nb, pb) in zip(a.named_parameters(), b.named_parameters()):
        assert torch.equal(pa, pb), na
    a.eval(), b.eval()
    with torch.no_grad():
        oa = a(ray_bundle(g["origins"], g["directions"], g["times"], DEV))
        ob = b(ray_bundle(g["origins"], g["directions"], g["times"], DEV))
    assert torch.equal(oa["rgb"], ob["rgb"]) and torch.equal(oa["depth"], ob["depth"])


def _variant_samples(g):
    from soccernerfs_b200.cameras.rays import RayBundle

    n = g["origins"].shape[0]
    rb = RayBundle(origins=g["origins"].to(DEV), directions=g["directions"].to(DEV), pixel_area=torch.ones(n, 1, device=DEV),
                   times=g["times"].to(DEV), nears=torch.zeros(n, 1, device=DEV), fars=torch.full((n, 1), 5.0, device=DEV))
    bins = g["bins"].to(DEV)
    return rb.get_ray_samples(bin_starts=bins[:, :-1, None], bin_ends=bins[:, 1:, None])


def _load_planes(grids, g, prefix, multi=True):
    with torch.no_grad():
        for i, gs in enumerate(grids if multi else [grids]):
            for j, p in enumerate(gs):
                p.copy_(g[f"{prefix}_{i}_{j}" if multi else f"{prefix}_{j}"].to(DEV))


def test_scene_contraction_fields_vs_reference_fixture():
    """bounded=False: SceneContraction(order=inf) evaluated inside the gather / scatter / proposal kernels (norm_mode 2)
    vs the reference's KPlanesField / KPlanesDensityField with its own SceneContraction (tests/golden/field_variants.npz)."""
    from soccernerfs_b200.field_components.spatial_distortions import SceneContraction
    from soccernerfs_b200.fields.base_field import FieldHeadNames
    from soccernerfs_b200.fields.kplanes_field import KPlanesDensityField, KPlanesField

    g = load_golden("field_variants")
    rs = _variant_samples(g)
    f = KPlanesField(g["aabb"], spacetime_resolution=(12, 10, 14, 5), feat_dim=8, multiscale_res=(1, 2), concat_features_across_scales=True,
                     linear_decoder=False, spatial_distortion=SceneContraction(order=float("inf"))).to(DEV)
    _load_planes(f.grids, g, "con_grid")
    with torch.no_grad():
        for name, net in (("sigma", f.sigma_net), ("color", f.color_net)):
            for i, w in enumerate(net.weights):
                w.copy_(g[f"con_{name}_w{i}"].to(DEV))
    out = f(rs)
    dens, rgb = out[FieldHeadNames.DENSITY], out[FieldHeadNames.RGB]
    assert rel_err(dens.cpu(), g["con_density"]) < TOL and rel_err(rgb.cpu(), g["con_rgb"]) < TOL
    ((dens * g["con_gd"].to(DEV)).sum() + (rgb * g["con_gr"].to(DEV)).sum()).backward()
    for i, gs in enumerate(f.grids):
        for j, p in enumerate(gs):
            assert rel_err(p.grad.cpu(), g[f"con_ggrid_{i}_{j}"]) < TOL, (i, j)
    for name, net in (("sigma", f.sigma_net), ("color", f.color_net)):
        for i, w in enumerate(net.weights):
            assert rel_err(w.grad.cpu(), g[f"con_{name}_gw{i}"]) < TOL, (name, i)
    # the same field through explicit positions (non-ray-form samples) takes the tensor form of the contraction
    df = KPlanesDensityField(g["aabb"], resolution=[16, 14, 18, 5], feature_dim=8, linear_decoder=False,
                             spatial_distortion=SceneContraction(order=float("inf"))).to(DEV)
    _load_planes(df.grids, g, "pcon_grid", multi=False)
    with torch.no_grad():
        for i, w in enumerate(df.sigma_net.weights):
            w.copy_(g[f"pcon_w{i}"].to(DEV))
    dd, _ = df.get_density(rs)
    assert rel_err(dd.cpu(), g["pcon_density"]) < TOL
    (dd * g["pcon_gd"].to(DEV)).sum().backward()
    for j, p in enumerate(df.grids):
        assert rel_err(p.grad.cpu(), g[f"pcon_ggrid_{j}"]) < TOL, j
    for i, w in enumerate(df.sigma_net.weights):
        assert rel_err(w.grad.cpu(), g[f"pcon_gw{i}"]) < TOL, i
    positions = rs.frustums.get_positions()
    dfn = df.density_fn(positions, times=rs.times[:, 0])
    assert rel_err(dfn.cpu(), g["pcon_density"]) < TOL


def test_decoder_depths_vs_reference_fixture():
    """sigma_net_layers / rgb_net_layers / hidden widths other than the presets' (KPlanesModelConfig, kplanes.py:96-103):
    the same networks layer by layer on the tensor-core dense layer vs the reference's own KPlanesField (fixture
    field_depths: 2 hidden sigma layers of 32 + 1 hidden colour layer of 48 with view dependence; no hidden sigma layer
    + 3 hidden colour layers without it): outputs and all gradients; the model config reaches the field."""
    from soccernerfs_b200.data.scene_box import SceneBox
    from soccernerfs_b200.fields.base_field import FieldHeadNames
    from soccernerfs_b200.fields.kplanes_field import KPlanesField
    from soccernerfs_b200.models.kplanes import KPlanesModelConfig

    g = load_golden("field_depths")
    n = g["origins"].shape[0]
    from soccernerfs_b200.cameras.rays import RayBundle

    rb = RayBundle(origins=g["origins"].to(DEV), directions=g["directions"].to(DEV), pixel_area=torch.ones(n, 1, device=DEV),
                   times=g["times"].to(DEV), nears=torch.zeros(n, 1, device=DEV), fars=torch.full((n, 1), 1.5, device=DEV))
    bins = g["bins"].to(DEV)
    rs = rb.get_ray_samples(bin_starts=bins[:, :-1, None], bin_ends=bins[:, 1:, None])
    variants = {"a": dict(sigma_net_layers=2, sigma_net_hidden_dim=32, rgb_net_layers=1, rgb_net_hidden_dim=48),
                "b": dict(sigma_net_layers=0, rgb_net_layers=3, rgb_net_hidden_dim=64, disable_viewing_dependent=True)}
    for tag, kw in variants.items():
        f = KPlanesField(g["aabb"], spacetime_resolution=(12, 10, 14, 5), feat_dim=8, multiscale_res=(1, 2),
                         concat_features_across_scales=True, linear_decoder=False, **kw).to(DEV)
        assert len(f.sigma_net.weights) == kw["sigma_net_layers"] + 1 and len(f.color_net.weights) == kw["rgb_net_layers"] + 1
        _load_planes(f.grids, g, f"{tag}_grid")
        with torch.no_grad():
            for name, net in (("sigma", f.sigma_net), ("color", f.color_net)):
                for i, w in enumerate(net.weights):
                    w.copy_(g[f"{tag}_{name}_w{i}"].to(DEV))
        out = f(rs)
        dens, rgb = out[FieldHeadNames.DENSITY], out[FieldHeadNames.RGB]
        assert rel_err(dens.cpu(), g[f"{tag}_density"]) < TOL and rel_err(rgb.cpu(), g[f"{tag}_rgb"]) < TOL, tag
        ((dens * g[f"{tag}_gd"].to(DEV)).sum() + (rgb * g[f"{tag}_gr"].to(DEV)).sum()).backward()
        for i, gs in enumerate(f.grids):
            for j, p in enumerate(gs):
                assert rel_err(p.grad.cpu(), g[f"{tag}_ggrid_{i}_{j}"]) < TOL, (tag, i, j)
        for name, net in (("sigma", f.sigma_net), ("color", f.color_net)):
            for i, w in enumerate(net.weights):
                assert rel_err(w.grad.cpu(), g[f"{tag}_{name}_gw{i}"]) < TOL, (tag, name, i)
    cfg = KPlanesModelConfig(spacetime_resolution=(8, 8, 8, 4), multiscale_res=(1, 2), sigma_net_layers=2, rgb_net_layers=3,
                             sigma_net_hidden_dim=32, proposal_net_args_list=[{"feature_dim": 8, "resolution": [8, 8, 8, 4]}] * 2)
    model = cfg.setup(scene_box=SceneBox(aabb=g["aabb"]), num_train_data=1).to(DEV)
    assert [tuple(w.shape) for w in model.field.sigma_net.weights] == [(32, 64), (32, 32), (16, 32)]
    assert len(model.field.color_net.weights) == 4
    from soccernerfs_b200.engine.trainer import TrainStep
    from tests.helpers import ray_bundle

    gold = load_golden("model_tiny")
    step = TrainStep(model, max_steps=50, warm_up_end=2)
    try:
        losses = [float(step(ray_bundle(gold["origins"], gold["directions"], gold["times"], DEV), {"image": gold["image"].to(DEV)})["loss"])
                  for _ in range(4)]
    finally:
        step.close()
    assert all(l == l and l < 1e3 for l in losses) and losses[-1] < losses[1], losses


def test_linear_decoder_field_vs_reference_fixture():
    """linear_decoder=True (learned colour basis, linear density) composed from the tensor-core dense layer vs the
    reference's KPlanesField(linear_decoder=True) (tests/golden/field_variants.npz): outputs and all gradients."""
    from soccernerfs_b200.fields.base_field import FieldHeadNames
    from soccernerfs_b200.fields.kplanes_field import KPlanesField

    g = load_golden("field_variants")
    rs = _variant_samples(g)
    f = KPlanesField(g["lin_aabb"], spacetime_resolution=(12, 10, 14, 5), feat_dim=8, multiscale_res=(1, 2),
                     concat_features_across_scales=True, linear_decoder=True, linear_decoder_layers=2).to(DEV)
    _load_planes(f.grids, g, "lin_grid")
    with torch.no_grad():
        for name, net in (("sigma", f.sigma_net), ("basis", f.color_basis)):
            for i, w in enumerate(net.weights):
                w.copy_(g[f"lin_{name}_w{i}"].to(DEV))
    out = f(rs)
    dens, rgb = out[FieldHeadNames.DENSITY], out[FieldHeadNames.RGB]
    assert rel_err(dens.cpu(), g["lin_density"]) < TOL and rel_err(rgb.cpu(), g["lin_rgb"]) < TOL
    ((dens * g["lin_gd"].to(DEV)).sum() + (rgb * g["lin_gr"].to(DEV)).sum()).backward()
    for i, gs in enumerate(f.grids):
        for j, p in enumerate(gs):
            assert rel_err(p.grad.cpu(), g[f"lin_ggrid_{i}_{j}"]) < TOL, (i, j)
    for name, net in (("sigma", f.sigma_net), ("basis", f.color_basis)):
        for i, w in enumerate(net.weights):
            assert rel_err(w.grad.cpu(), g[f"lin_{name}_gw{i}"]) < TOL, (name, i)


def test_appearance_embedding_and_unbounded_model_run():
    """use_appearance_embedding (unpinnable: the reference's own branch raises for S > 1, see KPlanesField._appearance):
    the composed colour net equals the fused default net when the codes' weights are zero, trains the codes, and uses the
    mean code in eval; KPlanesModel(bounded=False) runs a training step end to end (NearFarCollider + piecewise sampler +
    contraction)."""
    from soccernerfs_b200.data.scene_box import SceneBox
    from soccernerfs_b200.fields.base_field import FieldHeadNames
    from soccernerfs_b200.fields.kplanes_field import KPlanesField
    from soccernerfs_b200.models.kplanes import KPlanesModelConfig

    g = load_golden("field_variants")
    rs = _variant_samples(g)
    rs.camera_indices = torch.randint(0, 7, (rs.frustums.shape[0], 1, 1), device=DEV).expand(-1, rs.frustums.shape[1], 1)
    kw = dict(spacetime_resolution=(12, 10, 14, 5), feat_dim=8, multiscale_res=(1, 2), concat_features_across_scales=True,
              linear_decoder=False)
    torch.manual_seed(3)
    base = KPlanesField(g["lin_aabb"], **kw).to(DEV)
    app = KPlanesField(g["lin_aabb"], use_appearance_embedding=True, appearance_dim=5, num_images=7, **kw).to(DEV)
    with torch.no_grad():
        for a, b in zip(app.grids.parameters(), base.grids.parameters()):
            a.copy_(b)
        for a, b in zip(app.sigma_net.weights, base.sigma_net.weights):
            a.copy_(b)
        app.color_net.weights[0].zero_()
        app.color_net.weights[0][:, :31].copy_(base.color_net.weights[0])  # the 5 code columns stay zero
        for a, b in zip(list(app.color_net.weights)[1:], list(base.color_net.weights)[1:]):
            a.copy_(b)
    o_app, o_base = app(rs), base(rs)
    assert rel_err(o_app[FieldHeadNames.RGB], o_base[FieldHeadNames.RGB]) < 1e-5
    o_app[FieldHeadNames.RGB].sum().backward()
    assert app.appearance_embedding.embedding.weight.grad is not None  # zero first-layer columns: zero, but connected
    assert float(app.color_net.weights[0].grad[:, 31:].abs().sum()) > 0
    app.eval()
    with torch.no_grad():
        assert rel_err(app(rs)[FieldHeadNames.RGB], o_base[FieldHeadNames.RGB]) < 1e-5
    # unbounded model, one training step
    from soccernerfs_b200.engine.trainer import TrainStep
    from tests.helpers import ray_bundle

    cfg = KPlanesModelConfig(bounded=False, near_plane=0.05, far_plane=20.0, spacetime_resolution=(16, 16, 16, 6), multiscale_res=(1, 2),
                             num_nerf_samples_per_ray=16, num_proposal_samples_per_ray=(32, 24),
                             proposal_net_args_list=[{"feature_dim": 8, "resolution": [24, 24, 24, 6]},
                                                     {"feature_dim": 8, "resolution": [32, 32, 32, 6]}])
    model = cfg.setup(scene_box=SceneBox(aabb=g["aabb"]), num_train_data=3).to(DEV)
    step = TrainStep(model, max_steps=50, warm_up_end=2)
    gold = load_golden("model_tiny")
    losses = []
    for _ in range(4):
        out = step(ray_bundle(gold["origins"], gold["directions"], gold["times"], DEV), {"image": gold["image"].to(DEV)})
        losses.append(float(out["loss"]))
    assert all(l == l and l < 1e3 for l in losses) and losses[-1] < losses[1]
    step.close()
