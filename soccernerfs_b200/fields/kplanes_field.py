"""K-Planes field and proposal density field on the B200 kernels.

Same constructor arguments, parameter names/shapes and method surface as NS/fields/kplanes_field.py:129-463
(``KPlanesField.get_density/get_outputs/forward``, ``KPlanesDensityField.density_fn/get_density``,
``interpolate_kplanes``, ``init_kplanes_field``), so the reference's ``KPlanesModel`` can use them unchanged.
Differences, all internal:
  * plane parameters keep the logical shape [1,C,H,W] but are stored channel-last ([H][W][C] in memory);
  * the 6*K ``F.grid_sample`` calls + Hadamard + cat run as one gather kernel (one scatter kernel backward);
  * the tiny-cuda-nn decoders are bias-free fp32 MLPs (``FusedMLP``) executed by the decoder kernels.
There is no CPU path: calling these modules with CPU tensors raises.
"""
from __future__ import annotations

import itertools
from typing import Collection, Iterable, List, Optional, Sequence

import torch
from torch import nn
from torch.nn.parameter import Parameter

from .. import ops
from ..cameras.rays import Frustums, RaySamples
from ..data.scene_box import SceneBox
from ..field_components.embedding import Embedding
from .base_field import Field, FieldHeadNames

TIME_PLANES = (2, 4, 5)  # XT, YT, ZT in combinations(range(4), 2) order (kplanes_field.py:62-64)


def get_normalized_directions(directions: torch.Tensor) -> torch.Tensor:
    """SH encoding input range [0,1] (kplanes_field.py:39-44)."""
    return (directions + 1.0) / 2.0


def init_kplanes_field(out_dim: int, reso: Sequence[int], a: float = 0.1, b: float = 0.5) -> nn.ParameterList:
    """k-choose-2 planes of one scale: plane (i,j) has shape [1, out_dim, reso[j], reso[i]]; time planes = 1,
    space planes ~ U(a,b) (kplanes_field.py:47-74).  Memory is channel-last."""
    has_time = len(reso) == 4
    grids = nn.ParameterList()
    for comb in itertools.combinations(range(len(reso)), 2):
        plane = ops.new_plane(out_dim, reso[comb[1]], reso[comb[0]])
        if has_time and 3 in comb:
            nn.init.ones_(plane)
        else:
            nn.init.uniform_(plane, a=a, b=b)
        grids.append(nn.Parameter(plane))
    return grids


def _use_mask(n_planes: int, freeze_time_planes: bool) -> int:
    mask = (1 << n_planes) - 1
    if freeze_time_planes and n_planes == 6:
        for p in TIME_PLANES:  # frozen time planes are skipped entirely (kplanes_field.py:97-100)
            mask &= ~(1 << p)
    return mask


def _maybe_frozen(grids: Iterable[torch.Tensor], freeze_space_planes: bool) -> List[torch.Tensor]:
    grids = list(grids)
    if not freeze_space_planes:
        return grids
    n = len(grids)  # space planes get no gradient (kplanes_field.py:102-105)
    return [g.detach() if (n == 3 or i not in TIME_PLANES) else g for i, g in enumerate(grids)]


def interpolate_kplanes(pts: torch.Tensor, ms_grids: Collection[Iterable[nn.Module]], concat_features: bool,
                        freeze_time_planes: bool = False, freeze_space_planes: bool = False) -> torch.Tensor:
    """Query multi-scale planes at ``pts`` [M, 3|4] in [-1,1] -> [M, K*C] / [M, C] (kplanes_field.py:77-126)."""
    ms = [_maybe_frozen(g, freeze_space_planes) for g in ms_grids]
    if not torch.is_grad_enabled():
        ms = [[p.detach() for p in g] for g in ms]
    return ops.hexplane_features(ms, ops.points_from_pts(pts), concat_features, _use_mask(len(ms[0]), freeze_time_planes))


class FusedMLP(nn.Module):
    """Bias-free dense stack (tcnn ``FullyFusedMLP`` semantics, fp32): ``weights[i]`` is [out_i, in_i]."""

    def __init__(self, n_input_dims: int, n_output_dims: int, n_neurons: int, n_hidden_layers: int,
                 activation: str = "ReLU", output_activation: str = "None") -> None:
        super().__init__()
        dims = [n_input_dims] + [n_neurons] * n_hidden_layers + [n_output_dims]
        self.weights = nn.ParameterList()
        for i, o in zip(dims[:-1], dims[1:]):
            w = torch.empty(o, i)
            nn.init.xavier_uniform_(w)
            self.weights.append(nn.Parameter(w))
        self.n_input_dims, self.n_output_dims = n_input_dims, n_output_dims
        self.activation, self.output_activation = activation, output_activation


def _static_time(like: torch.Tensor) -> torch.Tensor:
    """The time coordinate of every point of a static render (models.base_model.static_scene): a constant, 0, that the
    masked-out time planes never read -- it only lets a dynamic field's points keep their four coordinates, with or
    without the cameras' times."""
    return torch.zeros(like.shape[:-1] + (1,), dtype=torch.float32, device=like.device)


def _ray_form(ray_samples: RaySamples):
    """(origins [N,3], directions [N,3], starts [N,S], ends [N,S], times [N]|None) if the samples are the usual
    per-ray broadcast of a RayBundle (RayBundle.get_ray_samples), else None."""
    fr = ray_samples.frustums
    if fr.offsets is not None or fr.origins.dim() < 2 or len(fr.shape) < 2:
        return None
    s = fr.shape[-1]
    if s > 1 and (fr.origins.stride(-2) != 0 or fr.directions.stride(-2) != 0):
        return None
    times = ray_samples.times
    if times is not None:
        if s > 1 and times.stride(-2) != 0:
            return None
        times = times[..., 0, 0].reshape(-1)
    return (fr.origins[..., 0, :].reshape(-1, 3), fr.directions[..., 0, :].reshape(-1, 3),
            fr.starts[..., 0].reshape(-1, s), fr.ends[..., 0].reshape(-1, s), times)


def _contraction_mode(spatial_distortion) -> bool:
    """True if ``spatial_distortion`` is the L-infinity SceneContraction the kernels evaluate in place (norm_mode 2)."""
    if spatial_distortion is None:
        return False
    order = getattr(spatial_distortion, "order", "missing")
    if type(spatial_distortion).__name__ != "SceneContraction" or order != float("inf"):
        raise NotImplementedError("only SceneContraction(order=float('inf')) -- what KPlanesModel(bounded=False) uses, "
                                  "NS/models/kplanes.py:203-206 -- is evaluated by the kernels")
    return True


class _AabbHostMixin:
    """Keeps a host copy of the aabb so kernel launches never sync on a device->host read."""

    def _aabb6(self):
        key = (self.aabb.data_ptr(), self.aabb._version)
        if getattr(self, "_aabb_key", None) != key:
            self._aabb_host = tuple(float(v) for v in self.aabb.detach().flatten().tolist())
            self._aabb_key = key
        return self._aabb_host


class KPlanesField(Field, _AabbHostMixin):
    """Multiscale hexplane radiance field (kplanes_field.py:129-370).

    Inference modes, set by context managers of models.base_model: ``static_scene`` (the time planes are left out of
    every feature product, as ``freeze_time_planes`` leaves them out, and the points carry a constant time) and
    ``dynamics_output`` (``forward`` also returns "dynamic" [..., 1]: per sample the dynamics score of
    ops.hexplane_features_dyn)."""

    static_scene = False
    dynamic_output = False

    def __init__(
        self,
        aabb,
        spacetime_resolution: Sequence[int] = (256, 256, 256, 150),
        feat_dim: int = 16,
        appearance_dim: int = 27,
        spatial_distortion=None,
        num_images: int = 0,
        multiscale_res: Optional[Sequence[int]] = None,
        concat_features_across_scales: bool = False,
        linear_decoder: bool = True,
        linear_decoder_layers: Optional[int] = None,
        use_appearance_embedding: bool = False,
        disable_viewing_dependent: bool = False,
        sigma_net_layers: int = 1,
        sigma_net_hidden_dim: int = 64,
        rgb_net_layers: int = 2,
        rgb_net_hidden_dim: int = 64,
        freeze_time_planes: bool = False,
        freeze_space_planes: bool = False,
    ) -> None:
        super().__init__()
        if sigma_net_layers < 0 or rgb_net_layers < 0:
            raise ValueError("sigma_net_layers / rgb_net_layers count hidden layers and cannot be negative")
        # the fused decoder kernels cover the depths every preset uses (kplanes.py:96-103: one hidden sigma layer, two
        # hidden colour layers); other depths run the same networks layer by layer on the tensor-core dense layer
        self._preset_depth = sigma_net_layers == 1 and rgb_net_layers == 2
        self.aabb = Parameter(aabb, requires_grad=False)
        self.spatial_distortion = spatial_distortion
        self._contract = _contraction_mode(spatial_distortion)
        self.multiscale_res_multipliers: Sequence[int] = multiscale_res or [1]
        self.concat_features_across_scales = concat_features_across_scales
        self.linear_decoder = linear_decoder
        self.has_time_planes = len(spacetime_resolution) == 4
        self.feature_dim = feat_dim * len(self.multiscale_res_multipliers) if concat_features_across_scales else feat_dim
        self.freeze_time_planes = freeze_time_planes
        self.freeze_space_planes = freeze_space_planes
        self.use_appearance_embedding = use_appearance_embedding
        self.appearance_embedding = None
        self.appearance_embedding_dim = 0
        if use_appearance_embedding:  # normal_(0, 1) initialised per-image codes (kplanes_field.py:196-203)
            assert num_images is not None
            self.appearance_embedding_dim = appearance_dim
            self.appearance_embedding = Embedding(num_images, self.appearance_embedding_dim)
        self.disable_viewing_dependent = disable_viewing_dependent

        self.grids = nn.ModuleList()
        for res in self.multiscale_res_multipliers:
            resolution = [r * res for r in spacetime_resolution[:3]]
            if len(spacetime_resolution) > 3:  # time does not get the multi-scale treatment (:181-182)
                resolution.append(spacetime_resolution[3])
            self.grids.append(init_kplanes_field(out_dim=feat_dim, reso=resolution))

        if self.linear_decoder:
            # learned colour basis instead of SH + MLP (kplanes_field.py:219-246): directions (+ appearance code) ->
            # 3 * feature_dim weights that combine the plane features into rgb; density is a linear map of the features
            assert linear_decoder_layers is not None
            self.color_basis = FusedMLP(3 + self.appearance_embedding_dim, 3 * self.feature_dim, 128, linear_decoder_layers)
            self.sigma_net = FusedMLP(self.feature_dim, 1, 128, 0, activation="None")
        else:
            self.geo_feat_dim = 15
            self.sigma_net = FusedMLP(self.feature_dim, self.geo_feat_dim + 1, sigma_net_hidden_dim, sigma_net_layers)
            self.in_dim_color = self.geo_feat_dim + self.appearance_embedding_dim + (0 if disable_viewing_dependent else 16)
            self.color_net = FusedMLP(self.in_dim_color, 3, rgb_net_hidden_dim, rgb_net_layers, output_activation="Sigmoid")

    # -- helpers ---------------------------------------------------------------------------------------
    def _points(self, ray_samples: RaySamples) -> ops.Points:
        static = self.static_scene and self.has_time_planes
        rf = _ray_form(ray_samples)
        if rf is not None:
            o, d, st, en, t = rf
            if static:
                t = _static_time(o)[:, 0]
            return ops.points_from_rays(o, d, st, en, t, self._aabb6(), norm_mode=2 if self._contract else 1,
                                        dynamic=self.has_time_planes and t is not None,
                                        ray_tile=0 if torch.is_grad_enabled() else int(getattr(self, "coherent_ray_tile", 0)))
        positions = ray_samples.frustums.get_positions()
        if self._contract:
            positions = self.spatial_distortion(positions) / 2.0  # from [-2, 2] to [-1, 1]
        else:
            positions = SceneBox.get_normalized_positions(positions, self.aabb) * 2.0 - 1.0
        if static:
            positions = torch.cat((positions, _static_time(positions)), dim=-1)
        elif self.has_time_planes and ray_samples.times is not None:
            positions = torch.cat((positions, ray_samples.times * 2 - 1), dim=-1)
        return ops.points_from_pts(positions.reshape(-1, positions.shape[-1]))

    def _planes(self):
        ms = [_maybe_frozen(g, self.freeze_space_planes) for g in self.grids]
        if not torch.is_grad_enabled():
            ms = [[p.detach() for p in g] for g in ms]
        return ms

    def _features(self, points: ops.Points) -> torch.Tensor:
        """The gather of get_density / _forward_fused; in dynamics_output mode also keeps the samples' dynamics scores
        for ``forward`` (``_last_dynamic``)."""
        ms = self._planes()
        if points.D != (4 if len(ms[0]) == 6 else 3):
            raise RuntimeError("dynamic K-Planes field needs ray_samples.times")
        self._last_points = points  # (bench.py's per-scale probe re-runs the gather / scatter on the step's own samples)
        mask = _use_mask(len(ms[0]), self.freeze_time_planes or self.static_scene)
        if self.dynamic_output and len(ms[0]) == 6 and not torch.is_grad_enabled():
            feats, self._last_dynamic = ops.hexplane_features_dyn(ms, points, self.concat_features_across_scales, mask)
            return feats
        return ops.hexplane_features(ms, points, self.concat_features_across_scales, mask,
                                     post_backward=getattr(self, "_kp_post_backward", None))

    # -- Field surface ---------------------------------------------------------------------------------
    def get_density(self, ray_samples: RaySamples):
        """-> (density [N,S,1], geometry features [M,15]).  kplanes_field.py:275-312."""
        batch = ray_samples.frustums.shape
        feats = self._features(self._points(ray_samples))
        if self.linear_decoder:  # density = trunc_exp(linear(features)); the features themselves feed the colour basis
            density = ops.trunc_exp(ops.linear(feats, self.sigma_net.weights[0]))
            return density.view(*batch, 1), feats
        if len(self.sigma_net.weights) != 2:  # any other depth (kplanes_field.py:249-273 with n_hidden_layers != 1)
            o = feats
            ws = self.sigma_net.weights
            for i, w in enumerate(ws):
                o = ops.linear(o, w, "relu" if i + 1 < len(ws) else "none")
            density = ops.trunc_exp(o[:, self.geo_feat_dim:self.geo_feat_dim + 1])  # kplanes_field.py:308-311
            return density.reshape(*batch, 1), o[:, : self.geo_feat_dim]
        o, density = ops.sigma_net(feats, self.sigma_net.weights[0], self.sigma_net.weights[1])
        return density.view(*batch, 1), o[:, : self.geo_feat_dim]

    def _appearance(self, ray_samples: RaySamples, n_rays: int, n_samples: int) -> torch.Tensor:
        """[M, dim]: every ray's per-image code repeated over its samples in training, the mean code in evaluation
        (kplanes_field.py:326-345).  NOTE: the reference's own expansion (``view(-1, 1, dim).expand(n_rays, n_samples, -1)``
        of an already per-sample lookup) raises for more than one sample per ray, so this branch -- off in every preset --
        cannot be pinned against it; it is implemented per its evident intent (one code per ray = per training image)."""
        dim = self.appearance_embedding_dim
        if self.training:
            assert ray_samples.camera_indices is not None
            ci = ray_samples.camera_indices[..., 0]
            if ci.dim() > 1:  # [N, S] broadcast of the bundle's per-ray indices
                ci = ci.reshape(n_rays, -1)[:, 0]
            emb = self.appearance_embedding(ci.reshape(n_rays))
        else:
            emb = self.appearance_embedding.mean(dim=0)[None, :].expand(n_rays, dim)
        return emb[:, None, :].expand(n_rays, n_samples, dim).reshape(-1, dim)

    def _get_outputs_composed(self, ray_samples: RaySamples, density_embedding: torch.Tensor) -> torch.Tensor:
        """The non-default colour branches (linear decoder / appearance embedding / a colour net of another depth than the
        presets'), composed from the tensor-core dense layer (ops.linear) exactly as kplanes_field.py:314-358 composes
        them from tcnn networks."""
        batch = ray_samples.frustums.shape
        n_samples = batch[-1]
        n_rays = 1
        for b in batch[:-1]:
            n_rays *= int(b)
        directions = ray_samples.frustums.directions.reshape(-1, 3)
        if self.linear_decoder or self.disable_viewing_dependent:
            color_features = [density_embedding]
        else:
            color_features = [ops.sh4(get_normalized_directions(directions)), density_embedding]
        if self.use_appearance_embedding:
            emb = self._appearance(ray_samples, n_rays, n_samples)
            if self.linear_decoder:
                directions = torch.cat((directions, emb), dim=-1)
            else:
                color_features.append(emb)
        color_features = torch.cat(color_features, dim=-1)
        if self.linear_decoder:
            x = directions
            ws = self.color_basis.weights
            for i, w in enumerate(ws):
                x = ops.linear(x, w, "relu" if i + 1 < len(ws) else "none")
            basis_values = x.view(color_features.shape[0], 3, -1)  # [M, 3, feature_dim]
            rgb = torch.sigmoid(torch.sum(color_features[:, None, :] * basis_values, dim=-1))
        else:
            x = color_features
            ws = self.color_net.weights
            for i, w in enumerate(ws):
                x = ops.linear(x, w, "relu" if i + 1 < len(ws) else "sigmoid")
            rgb = x
        return rgb.view(*batch, 3)

    def get_outputs(self, ray_samples: RaySamples, density_embedding: Optional[torch.Tensor] = None) -> torch.Tensor:
        """-> rgb [N,S,3] (bare tensor, like kplanes_field.py:314-358)."""
        assert density_embedding is not None
        if self.linear_decoder or self.use_appearance_embedding or len(self.color_net.weights) != 3:
            return self._get_outputs_composed(ray_samples, density_embedding)
        batch = ray_samples.frustums.shape
        n_samples = batch[-1]
        w3, w4, w5 = self.color_net.weights
        if self.disable_viewing_dependent:
            rgb = ops.color_net(None, n_samples, density_embedding, w3, w4, w5)
        else:
            dirs = ray_samples.frustums.directions
            if n_samples > 1 and dirs.stride(-2) == 0:
                rgb = ops.color_net(dirs[..., 0, :].reshape(-1, 3), n_samples, density_embedding, w3, w4, w5)
            else:
                rgb = ops.color_net(dirs.reshape(-1, 3), 1, density_embedding, w3, w4, w5)
        return rgb.view(*batch, 3)

    def forward(self, ray_samples: RaySamples, compute_normals: bool = False, mask=None, bg_color=None):
        self._last_dynamic = None
        out = self._forward_fused(ray_samples)
        if out is None:
            density, density_features = self.get_density(ray_samples)
            out = {FieldHeadNames.DENSITY: density, FieldHeadNames.RGB: self.get_outputs(ray_samples, density_features)}
        if self._last_dynamic is not None:
            out["dynamic"] = self._last_dynamic.view(*ray_samples.frustums.shape, 1)
            self._last_dynamic = None
        return out

    def _forward_fused(self, ray_samples: RaySamples):
        """get_density + get_outputs with both decoders in ONE tensor-core kernel (same numbers as the two-call path);
        None when the decoder shape is not covered (e.g. the 192 -> 128 sigma net of the 32x config)."""
        if self.linear_decoder or self.use_appearance_embedding or not self._preset_depth:
            return None
        w1, w2 = self.sigma_net.weights
        w3, w4, w5 = self.color_net.weights
        if not ops.decoder_fused_supported(self.feature_dim, w1.shape[0], w3.shape[0]):
            return None
        batch = ray_samples.frustums.shape
        n_samples = batch[-1]
        dirs = None
        if not self.disable_viewing_dependent:
            d = ray_samples.frustums.directions
            if not (n_samples > 1 and d.stride(-2) == 0):
                return None
            dirs = d[..., 0, :].reshape(-1, 3)
        feats = self._features(self._points(ray_samples))
        _, density, rgb = ops.decoder_fused(feats, dirs, n_samples, w1, w2, w3, w4, w5)
        return {FieldHeadNames.DENSITY: density.view(*batch, 1), FieldHeadNames.RGB: rgb.view(*batch, 3)}


class KPlanesDensityField(Field, _AabbHostMixin):
    """Proposal density field (kplanes_field.py:373-463): one fused gather + 8->64->1 MLP + trunc_exp kernel.
    ``static_scene``: as KPlanesField's (models.base_model.static_scene sets it on every proposal network too)."""

    static_scene = False

    def __init__(self, aabb, resolution, feature_dim, spatial_distortion=None, linear_decoder: bool = True,
                 freeze_time_planes: bool = False, freeze_space_planes: bool = False) -> None:
        super().__init__()
        self.aabb = Parameter(aabb, requires_grad=False)
        self.spatial_distortion = spatial_distortion
        self._contract = _contraction_mode(spatial_distortion)
        self.has_time_planes = len(resolution) == 4
        self.freeze_time_planes = freeze_time_planes
        self.freeze_space_planes = freeze_space_planes
        self.relu = not linear_decoder  # activation "None" when linear_decoder (:391-393)
        self.grids = init_kplanes_field(out_dim=feature_dim, reso=resolution, a=0.1, b=0.15)
        self.sigma_net = FusedMLP(feature_dim, 1, 64, 1, activation="ReLU" if self.relu else "None")

    def density_fn(self, positions: torch.Tensor, times: Optional[torch.Tensor] = None) -> torch.Tensor:
        """positions [..., 3] (world), times [N,1] -> density [..., 1].  kplanes_field.py:410-432."""
        if times is not None and len(positions.shape) == 3 and len(times.shape) == 2:
            times = times[:, None]
        ray_samples = RaySamples(
            frustums=Frustums(
                origins=positions,
                directions=torch.ones_like(positions),
                starts=torch.zeros_like(positions[..., :1]),
                ends=torch.zeros_like(positions[..., :1]),
                pixel_area=torch.ones_like(positions[..., :1]),
            ),
            times=times,
        )
        density, _ = self.get_density(ray_samples)
        return density

    def get_density(self, ray_samples: RaySamples):
        """-> (density [N,S,1], None).  NOTE: positions are normalised to [0,1] only, not [-1,1], exactly like
        the reference (kplanes_field.py:439-440; SURVEY.md finding 3)."""
        batch = ray_samples.frustums.shape
        static = self.static_scene and self.has_time_planes
        rf = _ray_form(ray_samples)
        if rf is not None:
            o, d, st, en, t = rf
            if static:
                t = _static_time(o)[:, 0]
            points = ops.points_from_rays(o, d, st, en, t, self._aabb6(), norm_mode=2 if self._contract else 0,
                                          dynamic=self.has_time_planes and t is not None)
        else:
            positions = ray_samples.frustums.get_positions()
            if self._contract:
                positions = self.spatial_distortion(positions) / 2.0  # from [-2, 2] to [-1, 1] (kplanes_field.py:436-438)
            else:
                positions = SceneBox.get_normalized_positions(positions, self.aabb)
            if static:
                positions = torch.cat((positions, _static_time(positions)), dim=-1)
            elif self.has_time_planes and ray_samples.times is not None:
                positions = torch.cat((positions, ray_samples.times * 2 - 1), dim=-1)
            points = ops.points_from_pts(positions.reshape(-1, positions.shape[-1]))
        grids = _maybe_frozen(self.grids, self.freeze_space_planes)
        if not torch.is_grad_enabled():
            grids = [p.detach() for p in grids]
        if points.D != (4 if len(grids) == 6 else 3):
            raise RuntimeError("dynamic K-Planes density field needs times")
        density = ops.density_field(grids, self.sigma_net.weights[0], self.sigma_net.weights[1], points, relu=self.relu,
                                    use_mask=_use_mask(len(grids), self.freeze_time_planes or self.static_scene))
        return density.view(*batch, 1), None

    def get_outputs(self, ray_samples: RaySamples, density_embedding: Optional[torch.Tensor] = None):
        return {}
