"""CPU-side checks of the space-time decomposition outputs: the names the renderers offer, the input errors, the static
mode's guard and state, and the new C-ABI entry points (declared, exported, arguments validated before any device work)."""
import types
from ctypes import c_void_p

import pytest
import torch

from soccernerfs_b200.cameras.camera_paths import get_path_from_json
from soccernerfs_b200.engine import path_renderer as pr
from tests.test_abi import _declared_symbols
from tests.test_render_path_host import _path, _stub_model

NEW = ["rgb_static", "depth_static", "accumulation_static", "dynamic"]


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge

    ge.build()
    from soccernerfs_b200 import _lib

    return _lib.load()


def test_available_outputs_of_dynamic_models_only():
    assert pr.available_outputs(_stub_model(dynamic=True))[-4:] == NEW
    static = pr.available_outputs(_stub_model(dynamic=False))
    assert not set(NEW) & set(static)


def test_render_input_errors(tmp_path):
    timed = get_path_from_json(_path(n=2, h=24, w=40))
    no_times = get_path_from_json(_path(n=2, h=24, w=40, times="some"))
    assert timed.times is not None and no_times.times is None
    for name in NEW:  # a static model has no decomposition
        with pytest.raises(ValueError, match="unknown rendered output"):
            pr.check_render_inputs(_stub_model(dynamic=False), timed, ["rgb", name])
    # outputs that depend on time need the cameras' times; the static render does not
    for names in (["dynamic"], ["rgb_static", "dynamic"], ["depth_static", "rgb"]):
        with pytest.raises(ValueError, match="render_time"):
            pr.check_render_inputs(_stub_model(dynamic=True), no_times, names)
    pr.check_render_inputs(_stub_model(dynamic=True), no_times, ["rgb_static", "depth_static", "accumulation_static"])
    pr.check_render_inputs(_stub_model(dynamic=True), timed, ["rgb", "rgb_static", "dynamic", "depth_static"])
    assert list(tmp_path.iterdir()) == []


def test_panel_kinds_and_accumulations():
    from soccernerfs_b200 import ops

    assert [ops.panel_kind(n) for n in NEW] == [0, 2, 1, 1]
    assert ops.accumulation_of("depth_static") == "accumulation_static"
    assert [ops.accumulation_of(n) for n in ("depth", "prop_depth_0")] == ["accumulation", "accumulation"]


def test_static_scene_is_inference_only_and_restores_the_model():
    from soccernerfs_b200.models.base_model import static_scene

    model = types.SimpleNamespace(field=types.SimpleNamespace(static_scene=False),
                                  proposal_networks=[types.SimpleNamespace(static_scene=False) for _ in range(2)])
    parts = [model.field] + model.proposal_networks
    with pytest.raises(RuntimeError, match="no_grad"):
        with static_scene(model):
            pass
    assert not any(m.static_scene for m in parts)
    with torch.no_grad():
        with static_scene(model):
            assert all(m.static_scene for m in parts)  # the field and both proposal networks
        assert not any(m.static_scene for m in parts)
        with pytest.raises(KeyError), static_scene(model):
            raise KeyError("restored on errors too")
        assert not any(m.static_scene for m in parts)


def test_new_symbols_are_declared_and_exported(lib):
    from soccernerfs_b200 import _lib

    for name in ("kp_hexplane_fwd_dyn", "kp_compose_frame_accs"):
        assert name in _declared_symbols() and name in _lib.SIGNATURES and hasattr(lib, name)


def test_dyn_gather_rejects_static_fields_without_gpu(lib):
    from soccernerfs_b200 import _lib

    pts = _lib.make_points(D=3)
    rc = lib.kp_hexplane_fwd_dyn(c_void_p(0), c_void_p(0), 1, 3, 32, pts, 0, 1, 0x7, c_void_p(0), c_void_p(0), c_void_p(0))
    assert rc != 0 and b"static field" in lib.kp_last_error()
    pts = _lib.make_points(D=5)
    rc = lib.kp_hexplane_fwd_dyn(c_void_p(0), c_void_p(0), 1, 6, 32, pts, 0, 1, 0x3F, c_void_p(0), c_void_p(0), c_void_p(0))
    assert rc != 0 and b"points.D" in lib.kp_last_error()
