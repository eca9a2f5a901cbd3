"""The hexplane gather / scatter and the fused proposal density field against the float64 reference, element by element, on
every dispatch path of soccernerfs_b200/csrc/hexplane.cu.

Each output element is compared with tests/field_reference.py against gamma * u * A (A: the same function of |inputs|;
gamma: the rounding count derived there).  Every kernel launch runs under torch.profiler, and the last test checks that
the launches of this module covered each template instantiation the dispatchers can choose (wide and float4 gathers give
identical bits, so only the kernel names can show which one ran).
"""
import itertools
import re

import pytest
import torch

from tests import field_reference as fr

pytestmark = pytest.mark.gpu
DEV = "cuda"
SEEN = set()  # kernel instantiations launched by this module's tests


def _run(fn):
    """Run ``fn`` under torch.profiler (CUDA activity only, nothing written) and record the field kernels that ran."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = set()
    for e in prof.key_averages():
        m = re.search(r"((?:hexplane|density_field)_\w+)<([^>]*)>", e.key)
        if m:
            names.add(f"{m.group(1)}<{', '.join(x.strip() for x in m.group(2).split(','))}>")
    SEEN.update(names)
    return out, names


def _lib_ops():
    from soccernerfs_b200 import _lib, ops

    return _lib, ops


def _plane(gen, c, h, w, lo=-1.5, hi=1.5, offset=0):
    """[1,C,H,W] channel-last plane; ``offset`` floats into a fresh flat buffer (4: 16- but not 32-byte aligned)."""
    flat = torch.empty(offset + h * w * c, device=DEV).uniform_(lo, hi, generator=gen)
    return flat[offset:].view(1, h, w, c).permute(0, 3, 1, 2)


def _field(gen, c, d, scales=(1, 2), t_res=4, base=(7, 5, 9), offset=0):
    """Non-square planes: coordinates x, y, z have different resolutions; the time axis has ``t_res`` (1 allowed)."""
    combos = list(itertools.combinations(range(d), 2))
    ms = []
    for s in scales:
        reso = [r * s for r in base] + [t_res]
        ms.append([_plane(gen, c, reso[b], reso[a], offset=offset) for a, b in combos])
    return ms


def _points(gen, form, d, n, s=1, ray_tile=0, reso0=(7, 5, 9)):
    """``pts``: random in [-1.1, 1.1] with a share of texel centres of the first scale and of exact +-1; ``ray<mode>``: n rays
    of s samples, normalised with norm_mode 0, 1 or 2 (the contraction sees points inside and outside the unit cube)."""
    _, ops = _lib_ops()
    if form == "pts":
        pts = torch.rand(n, d, device=DEV, generator=gen) * 2.2 - 1.1
        for j in range(min(d, 3)):
            r = reso0[j]
            centre = torch.randint(0, r, (n,), device=DEV, generator=gen).float() / (r - 1) * 2.0 - 1.0
            edge = torch.randint(0, 2, (n,), device=DEV, generator=gen).float() * 2.0 - 1.0
            pick = torch.randint(0, 4, (n,), device=DEV, generator=gen)
            pts[:, j] = torch.where(pick == 0, centre, torch.where(pick == 1, edge, pts[:, j]))
        return ops.points_from_pts(pts)
    mode = int(form[3:])
    spread = 2.0 if mode == 2 else 0.8
    o = (torch.rand(n, 3, device=DEV, generator=gen) - 0.5) * spread
    dr = torch.nn.functional.normalize(torch.randn(n, 3, device=DEV, generator=gen), dim=-1)
    edges = torch.sort(torch.rand(n, s + 1, device=DEV, generator=gen) * 1.5, dim=-1).values
    t = torch.rand(n, device=DEV, generator=gen)
    aabb = (-1.0, -1.2, -0.9, 1.1, 1.0, 1.3)
    return ops.points_from_rays(o, dr, edges[:, :-1].contiguous(), edges[:, 1:].contiguous(), t, aabb, norm_mode=mode,
                                dynamic=d == 4, ray_tile=ray_tile)


def _gather(ms, P, concat, mask):
    _, ops = _lib_ops()
    with torch.no_grad():
        return _run(lambda: ops.hexplane_features(ms, P, concat, mask))


def _scatter_check(gen, ms, P, concat, mask, need):
    """Scatter a random upstream gradient into pre-filled targets (planes with need False get none) with touched bytes on
    every plane; -> worst err / bound, kernel names.  Asserts the touched bytes equal the reference's touched set exactly
    and that every texel outside it keeps its exact prior value."""
    _lib, ops = _lib_ops()
    flat = [p for s in ms for p in s]
    n_planes, c = len(ms[0]), flat[0].shape[1]
    g = torch.randn(P.M, len(ms) * c if concat else c, device=DEV, generator=gen)
    prior = [torch.empty_like(p).uniform_(-1, 1, generator=gen) if n else None for p, n in zip(flat, need)]
    targets = [None if p is None else p.clone() for p in prior]
    touched = [torch.zeros(p.shape[2] * p.shape[3], dtype=torch.uint8, device=DEV) for p in flat]
    _, names = _run(lambda: _lib.call("kp_hexplane_bwd_flags", ops._plane_ptrs(flat), ops._plane_ptrs(targets),
                                      ops._plane_ptrs(touched), ops._plane_hw(flat), len(ms), n_planes, c, P.struct(), P.M,
                                      int(concat), mask, _lib.ptr(g), _lib.stream_ptr()))
    pt = fr.coords(P)
    got = [None if t is None else fr.texels(t, torch.float32) for t in targets]
    p0 = [None if p is None else fr.texels(p, torch.float32) for p in prior]
    worst, want = fr.scatter_ratio(got, p0, pt, ms, mask, concat, g, need)
    for i, t in enumerate(touched):
        expect = want[i] if want[i] is not None else torch.zeros_like(t, dtype=torch.bool)
        assert torch.equal(t, expect.to(torch.uint8)), f"touched bytes of plane {i}"
        if got[i] is not None:
            assert torch.equal(got[i][~expect], p0[i][~expect]), f"untouched texels of plane {i} changed"
    return worst, names


# (C, D, concat, point form, ray_tile, use_mask, rays, samples per ray, scales, time resolution, targets)
# M = rays * samples: 1, 31, 33, 32/LPS*k + 1 (97 for LPS 1, 65 for LPS 16, ...) and ~200 000.
# targets: "all", "some" (every third plane none), "scale" (the first scale has none: its whole scatter is skipped).
CASES = [
    (4, 4, True, "pts", 0, 0x3F, 97, 1, (1, 2), 4, "all"),
    (4, 3, False, "ray1", 4, 0x7, 11, 3, (1, 2, 4), 1, "some"),
    (4, 4, False, "ray2", 0, 0x1B, 1, 1, (1,), 1, "all"),
    (8, 4, False, "ray0", 0, 0x0B, 4000, 50, (1, 2), 4, "scale"),
    (8, 3, True, "pts", 0, 0x7, 31, 1, (1, 2), 1, "all"),
    (8, 4, True, "ray1", 16, 0x3F, 37, 7, (1, 2), 1, "some"),
    (16, 4, True, "ray2", 16, 0x1B, 1, 1, (1, 2), 4, "all"),
    (16, 3, False, "ray1", -1, 0x7, 11, 3, (1, 2), 1, "scale"),
    (16, 4, False, "pts", 0, 0x3F, 200001, 1, (1, 2, 4), 4, "some"),
    (32, 4, True, "ray1", 0, 0x3F, 4000, 50, (1, 2), 4, "all"),
    (32, 3, True, "pts", 0, 0x7, 33, 1, (1, 2), 1, "some"),
    (32, 4, False, "ray2", -1, 0x3F, 200, 9, (1, 2), 4, "scale"),
    (32, 3, False, "ray0", -1, 0x7, 31, 1, (1,), 1, "all"),
    (32, 4, True, "ray1", 16, 0x0B, 37, 7, (1, 2), 1, "all"),
    (32, 4, False, "ray0", 4, 0x1B, 1, 31, (1, 2), 4, "some"),
    (64, 4, True, "pts", 0, 0x3F, 65, 1, (1, 2), 4, "all"),
    (64, 3, False, "ray2", 4, 0x7, 13, 5, (1, 2), 1, "scale"),
    (64, 4, True, "ray1", 0, 0x1B, 31, 1, (1,), 1, "some"),
    (64, 3, True, "ray0", 0, 0x7, 2000, 33, (1, 2), 1, "all"),
]


def _need(kind, n_scales, n_planes):
    if kind == "some":
        return [i % 3 != 1 for i in range(n_scales * n_planes)]
    if kind == "scale":
        return [i >= n_planes for i in range(n_scales * n_planes)]
    return [True] * (n_scales * n_planes)


@pytest.mark.parametrize("case", CASES, ids=lambda c: "C{}-D{}-{}-{}-tile{}-m{:x}-M{}-{}".format(
    c[0], c[1], "cat" if c[2] else "sum", c[3], c[4], c[5], c[6] * c[7], c[10]))
def test_gather_and_scatter_vs_float64(case):
    c, d, concat, form, tile, mask, n, s, scales, t_res, kind = case
    gen = torch.Generator(device=DEV).manual_seed(CASES.index(case))
    ms = _field(gen, c, d, scales, t_res)
    P = _points(gen, form, d, n, s, tile)
    out, fwd = _gather(ms, P, concat, mask)
    rg = fr.gather_ratio(out, fr.coords(P), ms, mask, concat)
    rs, bwd = _scatter_check(gen, ms, P, concat, mask, _need(kind, len(scales), len(ms[0])))
    print(f"\n{case}: gather err/bound {rg:.3g} {sorted(fwd)}, scatter err/bound {rs:.3g} {sorted(bwd)}")
    assert rg <= 1.0 and rs <= 1.0


@pytest.mark.parametrize("what", ["planes", "output"])
def test_16_byte_aligned_views_take_the_float4_gather(what):
    """Planes (or the output) carved 4 floats into a flat buffer are 16- but not 32-byte aligned: the C = 32 gather must
    fall back from the 256-bit wide kernel to the float4 kernel and still meet the bound."""
    _lib, ops = _lib_ops()
    gen = torch.Generator(device=DEV).manual_seed(7)
    ms = _field(gen, 32, 4, (1, 2), 4, offset=4 if what == "planes" else 0)
    P = _points(gen, "ray1", 4, 97, 5)
    flat = [p for s in ms for p in s]
    buf = torch.zeros(4 + P.M * 64, device=DEV)
    out = buf[4:].view(P.M, 64) if what == "output" else buf[:P.M * 64].view(P.M, 64)
    _, names = _run(lambda: _lib.call("kp_hexplane_fwd", ops._plane_ptrs(flat), ops._plane_hw(flat), 2, 6, 32, P.struct(), P.M,
                                      1, 0x3F, _lib.ptr(out), _lib.stream_ptr()))
    r = fr.gather_ratio(out, fr.coords(P), ms, 0x3F, True)
    print(f"\n{what} at +16 bytes: gather err/bound {r:.3g} {sorted(names)}")
    assert names == {"hexplane_fwd_kernel<32, 6, false>"} and r <= 1.0


def test_streaming_field_gather_and_scatter():
    """A 512 MiB field (C = 32, reso 1024 x 1024 x 1536 x 8) streams its planes of at least 16 MiB with the evict_first
    policy: XY (128 MiB), XZ and YZ (192 MiB) stream and the time planes (1 - 1.5 MiB) do not, in the same launch."""
    _lib, ops = _lib_ops()
    gen = torch.Generator(device=DEV).manual_seed(8)
    ms = _field(gen, 32, 4, (1,), 8, base=(1024, 1024, 1536))
    assert sum(p.numel() for p in ms[0]) * 4 >= 512 << 20
    try:
        P = _points(gen, "pts", 4, 100000)
        out, names = _gather(ms, P, True, 0x3F)
        r1 = fr.gather_ratio(out, fr.coords(P), ms, 0x3F, True)
        assert names == {"hexplane_fwd_kernel<32, 6, true>"}
        Pr = _points(gen, "ray1", 4, 2003, 50, ray_tile=16)
        out, names = _gather(ms, Pr, True, 0x3F)
        r2 = fr.gather_ratio(out, fr.coords(Pr), ms, 0x3F, True)
        assert names == {"hexplane_fwd_wide_kernel<6, true>"}
        r3, names = _scatter_check(gen, ms, P, True, 0x3F, [True] * 6)
        assert names == {"hexplane_bwd_kernel<32, 6, true>"}
        print(f"\nstreaming field: gather float4 {r1:.3g}, wide {r2:.3g}; scatter {r3:.3g}")
        assert max(r1, r2, r3) <= 1.0
    finally:
        del ms
        torch.cuda.empty_cache()


# ---- fused proposal density field ----------------------------------------------------------------------------------------
def _density_inputs(gen, c, n_planes, hidden, offset=0, form="ray0", m=333):
    d = 3 if n_planes == 3 else 4
    planes = _field(gen, c, d, (1,), 5, base=(11, 9, 13), offset=offset)[0]
    for p in planes:  # proposal-field-like magnitudes: the product of six planes stays O(0.1..1)
        p.copy_(p.abs() * 0.4 + 0.6)
    bound = (6.0 / (c + hidden)) ** 0.5
    w1 = torch.empty(hidden, c, device=DEV).uniform_(-bound, bound, generator=gen)
    w2 = torch.empty(1, hidden, device=DEV).uniform_(-1.0, 1.0, generator=gen) * (6.0 / (hidden + 1)) ** 0.5
    if form == "pts":
        P = _points(gen, "pts", d, m, reso0=(11, 9, 13))
    else:
        s = 7 if m % 7 == 0 else 1
        P = _points(gen, form, d, m // s, s)
    return planes, w1, w2, P


DENSITY = [(c, n_planes, relu) for c in (4, 8, 16) for n_planes in (3, 6) for relu in (True, False)]


@pytest.mark.parametrize("c,n_planes,relu", DENSITY)
def test_density_forward_and_backward_vs_float64(c, n_planes, relu):
    _lib, ops = _lib_ops()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    big = 4 * sms * 128 + 1000  # more than one grid-stride pass of the backward's 4-blocks-per-SM grid
    gen = torch.Generator(device=DEV).manual_seed(200 + 10 * c + n_planes + int(relu))
    mask = (1 << n_planes) - 1
    for m, offset, form in ((1, 0, "pts"), (31, 4, "ray0"), (33, 0, "ray1"), (big + 7 * 3, 0, "ray0"), (big, 4, "pts")):
        if offset and c != 8:
            continue  # the 16-byte-aligned variant only exists for C = 8
        planes, w1, w2, P = _density_inputs(gen, c, n_planes, 64, offset, form, m)
        pt = fr.coords(P)
        with torch.no_grad():
            dens, fwd = _run(lambda: ops.density_field(planes, w1, w2, P, relu, mask))
        rf = fr.density_ratio(dens, pt, planes, w1, w2, relu, mask)
        # upstream gradient: at the large sizes a whole warp of zeros, a warp with every other lane zero and zero lanes before
        # the ragged tail (whose padding lanes the kernel zeroes itself); ReLU ties dropped everywhere
        g = torch.randn(P.M, device=DEV, generator=gen)
        if P.M > 64:
            g[:32] = 0
            g[32:64:2] = 0
            g[-5:] = 0
        ties = fr.relu_ties(pt, planes, w1, w2, mask) if relu else torch.zeros_like(g, dtype=torch.bool)
        g[ties] = 0
        prior = ([torch.empty_like(p).uniform_(-1, 1, generator=gen) for p in planes], torch.randn(64, c, device=DEV, generator=gen),
                 torch.randn(64, device=DEV, generator=gen))
        got = ([p.clone() for p in prior[0]], prior[1].clone(), prior[2].clone())
        _, bwd = _run(lambda: _lib.call("kp_density_field_bwd", ops._plane_ptrs(planes), ops._plane_ptrs(got[0]), ops._plane_hw(planes),
                                        n_planes, c, _lib.ptr(w1), _lib.ptr(w2), 64, int(relu), P.struct(), P.M, mask, _lib.ptr(g),
                                        _lib.ptr(got[1]), _lib.ptr(got[2]), _lib.stream_ptr()))
        tex = lambda ts: [fr.texels(t, torch.float32) for t in ts]  # noqa: E731
        rb = fr.density_backward_ratios((tex(got[0]), got[1], got[2]), (tex(prior[0]), prior[1], prior[2]), pt, planes, w1, w2,
                                        relu, mask, g, [True] * n_planes, sms)
        print(f"\nC={c} planes={n_planes} relu={relu} M={P.M} offset={offset}: forward err/bound {rf:.3g}, backward "
              f"{ {k: round(v, 3) for k, v in rb.items()} }, ReLU ties dropped {float(ties.float().mean()):.2%} "
              f"{sorted(fwd | bwd)}")
        assert float(ties.float().mean()) < 0.01
        assert rf <= 1.0 and max(rb.values()) <= 1.0


@pytest.mark.parametrize("hidden", [1, 17, 64, 256])
def test_density_forward_hidden_widths(hidden):
    """The forward pairs hidden units (an odd last unit with a zero partner); the backward supports hidden = 64 only."""
    _lib, ops = _lib_ops()
    gen = torch.Generator(device=DEV).manual_seed(300 + hidden)
    for c, relu in ((8, True), (16, False)):
        planes, w1, w2, P = _density_inputs(gen, c, 6, hidden, m=1001)
        with torch.no_grad():
            dens, _ = _run(lambda: ops.density_field(planes, w1, w2, P, relu))
        r = fr.density_ratio(dens, fr.coords(P), planes, w1, w2, relu, 0x3F)
        print(f"\nhidden={hidden} C={c} relu={relu}: forward err/bound {r:.3g}")
        assert r <= 1.0
        if hidden != 64:
            g = torch.ones(P.M, device=DEV)
            gw1, gw2 = torch.zeros_like(w1), torch.zeros(hidden, device=DEV)
            with pytest.raises(RuntimeError, match=f"hidden={hidden} unsupported"):
                _lib.call("kp_density_field_bwd", ops._plane_ptrs(planes), ops._plane_ptrs(planes), ops._plane_hw(planes), 6, c,
                          _lib.ptr(w1), _lib.ptr(w2), hidden, int(relu), P.struct(), P.M, 0x3F, _lib.ptr(g), _lib.ptr(gw1),
                          _lib.ptr(gw2), _lib.stream_ptr())


# ---- every dispatch path ran -----------------------------------------------------------------------------------------------
EXPECTED = (
    {f"hexplane_fwd_kernel<{c}, {n}, false>" for c in (4, 8, 16, 32, 64) for n in (3, 6)}
    | {f"hexplane_bwd_kernel<{c}, {n}, false>" for c in (4, 8, 16, 32, 64) for n in (3, 6)}
    | {"hexplane_fwd_wide_kernel<3, false>", "hexplane_fwd_wide_kernel<6, false>", "hexplane_fwd_wide_kernel<6, true>",
       "hexplane_fwd_kernel<32, 6, true>", "hexplane_bwd_kernel<32, 6, true>"}
    | {f"density_field_fwd_kernel<{c}, {n}, {w}>" for c in (4, 8, 16) for n in (3, 6) for w in (("false", "true") if c == 8 else ("false",))}
    | {f"density_field_bwd_kernel<{c}, {n}, 64, {w}>" for c in (4, 8, 16) for n in (3, 6)
       for w in (("false", "true") if c == 8 else ("false",))}
)


def test_every_dispatch_path_ran():
    """Checks the launches of the tests above (run the whole module): each instantiation listed in EXPECTED ran."""
    if not SEEN:
        pytest.skip("no field kernel launched in this session: run the whole module")
    missing = sorted(EXPECTED - SEEN)
    print(f"\n{len(SEEN)} field kernel instantiations ran")
    assert not missing, missing
