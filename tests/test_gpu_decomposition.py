"""The space-time decomposition of a dynamic scene on the device: kp_hexplane_fwd_dyn (the features of kp_hexplane_fwd bit
for bit and the dynamics score against a float64 restatement over the oracle's grid_sample), the static render
(models.base_model.static_scene) against a copy of the model whose time planes are 1, the ``dynamic`` output leaving every
other output's bits alone, the composition of the new panels, and camera-path files with them."""
import copy
import io
import itertools
import re
import types

import numpy as np
import pytest
import torch

from tests import field_reference as fr
from tests.test_gpu_field_kernels import _field, _points

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TIME = (2, 4, 5)  # XT, YT, ZT


def _dyn_run(ms, P, concat, mask):
    """(features of kp_hexplane_fwd, (features, delta) of kp_hexplane_fwd_dyn, kernel names of the dyn launch)."""
    from torch.profiler import ProfilerActivity, profile

    from soccernerfs_b200 import ops

    with torch.no_grad():
        plain = ops.hexplane_features(ms, P, concat, mask)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            feats, delta = ops.hexplane_features_dyn(ms, P, concat, mask)
            torch.cuda.synchronize()
    names = set()
    for e in prof.key_averages():
        m = re.search(r"(hexplane_\w+)<([^>]*)>", e.key)
        if m:
            names.add(f"{m.group(1)}<{', '.join(x.strip() for x in m.group(2).split(','))}>")
    return plain, feats, delta, names


def _delta64(P, ms, mask):
    """delta restated in float64: per scale the product of the kept time planes' grid_sample interpolants (oracle), then
    the mean over scales and channels of |1 - T|."""
    from oracle.kplanes_oracle import grid_sample_plane

    pt = fr.coords(P).double()
    combos = list(itertools.combinations(range(4), 2))
    total = 0.0
    for planes in ms:
        t = torch.ones(pt.shape[0], planes[0].shape[1], dtype=torch.float64, device=pt.device)
        for p in TIME:
            if (mask >> p) & 1:
                a, b = combos[p]
                t = t * grid_sample_plane(planes[p].double().contiguous(), pt[:, [a, b]])
        total = total + (1.0 - t).abs().sum(dim=1)
    return total / (len(ms) * ms[0][0].shape[1])


def _time_planes(ms, kind, gen):
    """``random``: the planes as drawn; ``ones``: time planes exactly 1; ``perturbed``: ones + perturb_time_planes' noise."""
    from soccernerfs_b200.data.synthetic import perturb_time_planes

    if kind == "random":
        return
    with torch.no_grad():
        for planes in ms:
            for p in TIME:
                planes[p].fill_(1.0)
    if kind == "perturbed":
        perturb_time_planes(types.SimpleNamespace(field=types.SimpleNamespace(grids=ms), proposal_networks=[]),
                            seed=int(torch.randint(0, 1 << 30, (1,), generator=gen, device=DEV)))


# (C, concat, point form, ray_tile, use_mask, rays, samples per ray, scales): every C, concat and summed scales, the float4
# and the wide gathers (ray_tile -1 forces float4), coherent rays, a time plane masked out, and M = 1, 31, 65, 97, 200 000.
CASES = [
    (4, True, "pts", 0, 0x3F, 97, 1, (1, 2)),
    (4, False, "ray1", 4, 0x1B, 11, 3, (1, 2, 4)),
    (8, False, "ray0", 0, 0x3F, 4000, 50, (1, 2)),
    (8, True, "ray1", 16, 0x3F, 37, 7, (1, 2)),
    (16, True, "ray2", 16, 0x3F, 1, 1, (1, 2)),
    (16, False, "pts", 0, 0x2F, 200001, 1, (1, 2, 4)),
    (32, True, "ray1", 0, 0x3F, 4000, 50, (1, 2)),
    (32, False, "ray2", -1, 0x3F, 200, 9, (1, 2)),
    (32, True, "ray1", 16, 0x1B, 37, 7, (1, 2)),
    (32, False, "ray0", 4, 0x3F, 1, 31, (1, 2)),
    (32, True, "pts", -1, 0x3F, 33, 1, (1,)),
    (64, True, "pts", 0, 0x3F, 65, 1, (1, 2)),
    (64, False, "ray1", 4, 0x3F, 13, 5, (1,)),
]
SEEN = set()


@pytest.mark.parametrize("planes", ["random", "ones", "perturbed"])
@pytest.mark.parametrize("case", CASES, ids=lambda c: "C{}-{}-{}-tile{}-m{:x}-M{}".format(
    c[0], "cat" if c[1] else "sum", c[2], c[3], c[4], c[5] * c[6]))
def test_dyn_gather_vs_plain_gather_and_float64(case, planes):
    c, concat, form, tile, mask, n, s, scales = case
    gen = torch.Generator(device=DEV).manual_seed(CASES.index(case))
    ms = _field(gen, c, 4, scales, 4)
    _time_planes(ms, planes, gen)
    P = _points(gen, form, 4, n, s, tile)
    plain, feats, delta, names = _dyn_run(ms, P, concat, mask)
    SEEN.update(names)
    assert torch.equal(feats.view(torch.int32), plain.view(torch.int32)), "features differ from kp_hexplane_fwd's bits"
    assert delta.shape == (P.M,) and delta.dtype == torch.float32
    want = _delta64(P, ms, mask)
    if planes == "ones":
        # T is the bilinear interpolant of a constant 1: 1 up to the rounding of the four corner weights' products
        assert float(want.max()) < 1e-12 and float(delta.max()) < 1e-6, float(delta.max())
        return
    err = (delta.double() - want).abs()
    print(f"\n{case} {planes}: max |delta - fp64| {float(err.max()):.3g}, delta in [{float(want.min()):.3g}, "
          f"{float(want.max()):.3g}] {sorted(names)}")
    assert bool((err <= 1e-5 + 1e-5 * want.abs()).all())
    assert float(want.max()) > 0


def test_dyn_streaming_field():
    """A field of at least 512 MiB streams its large planes (evict_first): the streaming float4 and wide dyn kernels."""
    gen = torch.Generator(device=DEV).manual_seed(99)
    ms = _field(gen, 32, 4, (1,), 8, base=(1024, 1024, 1536))
    try:
        _time_planes(ms, "perturbed", gen)
        for form, tile, n, s in (("pts", 0, 100000, 1), ("ray1", 16, 2003, 50)):
            P = _points(gen, form, 4, n, s, tile)
            plain, feats, delta, names = _dyn_run(ms, P, True, 0x3F)
            SEEN.update(names)
            assert torch.equal(feats.view(torch.int32), plain.view(torch.int32))
            want = _delta64(P, ms, 0x3F)
            assert bool(((delta.double() - want).abs() <= 1e-5 + 1e-5 * want.abs()).all()), form
    finally:
        del ms
        torch.cuda.empty_cache()


def test_dyn_every_dispatch_path_ran():
    """Checks the launches of the tests above (run the whole module): every dyn instantiation the dispatcher can pick."""
    if not SEEN:
        pytest.skip("no dyn gather launched in this session: run the whole module")
    expected = ({f"hexplane_fwd_dyn_kernel<{c}, false>" for c in (4, 8, 16, 32, 64)}
                | {"hexplane_fwd_dyn_kernel<32, true>", "hexplane_fwd_wide_dyn_kernel<false>", "hexplane_fwd_wide_dyn_kernel<true>"})
    assert not (expected - SEEN), sorted(expected - SEEN)


def test_dyn_rejects_a_static_field():
    from soccernerfs_b200 import _lib, ops

    gen = torch.Generator(device=DEV).manual_seed(5)
    ms = _field(gen, 8, 3, (1,), 1)
    P = _points(gen, "pts", 3, 10)
    with torch.no_grad(), pytest.raises(RuntimeError, match="static field"):
        ops.hexplane_features_dyn(ms, P, True, 0x7)
    assert b"static field" in _lib.load().kp_last_error()


# ---- the model ------------------------------------------------------------------------------------------------------------
def _tiny_model():
    from tests.test_gpu_render_path import _tiny_model as tiny

    return tiny()


def _cameras(times=(0.3,), untimed=False):
    """Cameras of one pose with the given render times; ``untimed``: the same cameras without times."""
    from soccernerfs_b200.cameras.camera_paths import get_path_from_json
    from tests.test_gpu_render_path import _camera_path

    path = _camera_path(n=len(times), times=list(times), same_pose=True)
    if untimed:
        for cam in path["camera_path"]:
            del cam["render_time"]
    return get_path_from_json(path).to(DEV)


def _render(model, cams, outputs, i=0, **kw):
    from soccernerfs_b200.engine.frame_renderer import FrameRenderer

    return FrameRenderer(model, cams, outputs=outputs, **kw).render(i, device_frames=True)


def _time_planes_to_one(model):
    twin = copy.deepcopy(model)
    with torch.no_grad():
        for grids in list(twin.field.grids) + [p.grids for p in twin.proposal_networks]:
            for p in TIME:
                grids[p].fill_(1.0)
    return twin


def test_static_render_matches_time_planes_of_one():
    model = _tiny_model()
    cams = _cameras((0.3,))
    got = _render(model, cams, ("rgb_static", "depth_static", "accumulation_static"))
    want = _render(_time_planes_to_one(model), cams, ("rgb", "depth", "accumulation"))
    for name in ("rgb", "depth", "accumulation"):
        a, b = got[f"{name}_static"], want[name]
        err = float((a - b).abs().max())
        print(f"\n{name}_static vs time planes of 1: max abs diff {err:.3g}")
        assert torch.allclose(a, b, rtol=1e-5, atol=1e-5), (name, err)
    # the model's own time planes are not 1: its ordinary render differs from the static one
    assert not torch.allclose(_render(model, cams, ("rgb",))["rgb"], got["rgb_static"], rtol=1e-5, atol=1e-5)
    for m in [model.field] + list(model.proposal_networks):  # the mode ends with the context
        assert m.static_scene is False


def test_static_render_needs_no_times_and_ignores_them():
    model = _tiny_model()
    names = ("rgb_static", "depth_static", "accumulation_static")
    two = _cameras((0.0, 1.0))
    t0, t1 = _render(model, two, names, 0), _render(model, two, names, 1)
    untimed = _cameras((0.0, 1.0), untimed=True)
    assert untimed.times is None
    none = _render(model, untimed, names, 0)
    for name in names:
        assert torch.equal(t0[name], t1[name]), name
        assert torch.equal(t0[name], none[name]), name
    with torch.no_grad(), pytest.raises(RuntimeError, match="times"):  # an ordinary render still needs them
        _render(model, untimed, ("rgb",), 0)


@pytest.mark.parametrize("graph", [True, False])
@pytest.mark.parametrize("world", [1, 2])
def test_dynamic_output_leaves_the_other_outputs_bit_identical(graph, world):
    model = _tiny_model()
    cams = _cameras((0.7,))
    base = ("rgb", "depth", "accumulation")
    for rank in range(world):
        kw = dict(use_cuda_graph=graph, rank=rank, world=world)
        plain = _render(model, cams, base, **kw)
        more = _render(model, cams, base + ("dynamic", "rgb_static"), **kw)
        for name in base:
            assert torch.equal(plain[name].view(torch.int32), more[name].view(torch.int32)), (name, rank)
        dyn = more["dynamic"]
        assert dyn.shape == (37, 53, 1) and bool((dyn >= 0).all()) and float(dyn.max()) > 0
    # graphed and eager renders agree on the new outputs, and time planes of 1 move nothing
    a = _render(model, cams, ("dynamic", "rgb_static"), use_cuda_graph=True)
    b = _render(model, cams, ("dynamic", "rgb_static"), use_cuda_graph=False)
    assert torch.equal(a["dynamic"], b["dynamic"]) and torch.equal(a["rgb_static"], b["rgb_static"])
    still = _render(_time_planes_to_one(model), cams, ("dynamic",), use_cuda_graph=graph)["dynamic"]
    assert float(still.max()) < 1e-6  # the rounding of bilinear weights only


def test_dynamic_is_the_weighted_sum_of_the_sample_scores():
    """model.get_outputs' ``dynamic`` is sum_i w_i delta_i with the final level's weights and the field's own scores."""
    from soccernerfs_b200.fields.base_field import FieldHeadNames
    from soccernerfs_b200.models.base_model import dynamics_output

    model = _tiny_model()
    bundle = _cameras((0.4,)).generate_tile(0, 0, 256)
    seen = {}
    orig = model.field.forward

    def spy(ray_samples, *a, **k):
        out = orig(ray_samples, *a, **k)
        seen["delta"], seen["density"], seen["samples"] = out.get("dynamic"), out[FieldHeadNames.DENSITY], ray_samples
        return out

    model.field.forward = spy
    with torch.no_grad(), dynamics_output(model):
        out = model.forward(ray_bundle=bundle)
    weights = seen["samples"].get_weights(seen["density"])
    want = (weights.double() * seen["delta"].double()).sum(dim=-2)
    assert out["dynamic"].shape == (256, 1)
    assert torch.allclose(out["dynamic"].double(), want, rtol=1e-6, atol=1e-7)


# ---- composition ----------------------------------------------------------------------------------------------------------
def test_compose_static_depth_with_its_own_accumulation():
    from soccernerfs_b200 import ops
    from soccernerfs_b200.utils import colormaps
    from tests.test_gpu_render_path import _cmap_clamped, _quantise, _random_frames

    frames = _random_frames(135, 240, 11)
    g = torch.Generator(device=DEV).manual_seed(12)
    frames["depth_static"] = 1.0 + 9.0 * torch.rand((135, 240, 1), generator=g, device=DEV)
    frames["accumulation_static"] = torch.rand((135, 240, 1), generator=g, device=DEV)
    frames["dynamic"] = 1.3 * torch.rand((135, 240, 1), generator=g, device=DEV)  # above 1 in places: clamped
    depth = colormaps.apply_depth_colormap(frames["depth"], accumulation=frames["accumulation"])
    depth_static = colormaps.apply_depth_colormap(frames["depth_static"], accumulation=frames["accumulation_static"])
    got = ops.compose_frame(frames, ["depth_static", "accumulation_static"])
    want = _quantise(torch.cat([depth_static, colormaps.apply_colormap(frames["accumulation_static"])], dim=1))
    assert torch.equal(got, want)
    assert torch.equal(ops.compose_frame(frames, ["dynamic"]), _quantise(_cmap_clamped(frames["dynamic"], "viridis")))
    # side by side, every panel is composed as it is alone: each depth panel with its own accumulation
    names = ["depth", "depth_static", "dynamic", "rgb"]
    got = ops.compose_frame(frames, names)
    for k, name in enumerate(names):
        assert torch.equal(got[:, 240 * k:240 * (k + 1)], ops.compose_frame(frames, [name])), name
    assert torch.equal(got[:, 240:480], want[:, :240])
    wrong = colormaps.apply_depth_colormap(frames["depth_static"], accumulation=frames["accumulation"])
    assert not torch.equal(got[:, 240:480], _quantise(wrong))
    with pytest.raises(ValueError, match="accumulation_static"):
        ops.compose_frame({k: v for k, v in frames.items() if k != "accumulation_static"}, ["depth_static"])


# ---- camera-path files ----------------------------------------------------------------------------------------------------
def test_camera_path_jpeg_and_video_with_the_decomposition(tmp_path):
    from PIL import Image

    from soccernerfs_b200.engine.path_renderer import load_camera_path, render_camera_path, render_camera_path_video
    from tests.test_gpu_render_path import _camera_path
    from tests.test_video_host import _parse_avi

    model = _tiny_model()
    cams, _ = load_camera_path(_camera_path(n=3))
    names = ("rgb", "rgb_static", "dynamic")
    assert render_camera_path(model, cams, tmp_path / "jpg", rendered_output_names=names, image_format="jpeg") == [0, 1, 2]
    for i in range(3):
        with Image.open(tmp_path / "jpg" / f"{i:05d}.jpg") as im:
            im.load()
            assert im.size == (53 * 3, 37) and im.mode == "RGB"
    render_camera_path_video(model, cams, tmp_path / "path.avi", 1.5, rendered_output_names=names)
    avi = _parse_avi(tmp_path / "path.avi")
    assert (avi["width"], avi["height"]) == (53 * 3, 37) and len(avi["frames"]) == 3
    for data in avi["frames"]:
        with Image.open(io.BytesIO(data)) as im:
            im.load()
            assert im.size == (53 * 3, 37)
    # a static-only path needs no render times; the depth panel is blended with the static accumulation
    untimed = _camera_path(n=2)
    for cam in untimed["camera_path"]:
        del cam["render_time"]
    cams_nt, _ = load_camera_path(untimed)
    assert cams_nt.times is None
    render_camera_path(model, cams_nt, tmp_path / "static", rendered_output_names=("rgb_static", "depth_static"))
    with Image.open(tmp_path / "static" / "00001.png") as im:
        assert np.asarray(im).shape == (37, 53 * 2, 3)
