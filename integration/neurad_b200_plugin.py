"""Reference-side plugin: NeuRAD with the B200-native NFF backend, registered through nerfstudio's own plugin mechanism.

This file is imported INSIDE an installation of the reference (georghess/neurad-studio): it subclasses the reference's
`NeuRADModel` / `NeuRADModelConfig` (nerfstudio/models/neurad.py:97-165) and exports a `MethodSpecification`
(nerfstudio/plugins/types.py:23-33) that `discover_methods()` (nerfstudio/plugins/registry.py:34-79) picks up from

    export NERFSTUDIO_METHOD_CONFIGS="neurad-b200=integration.neurad_b200_plugin:spec"

(with this repository's root on PYTHONPATH), after which `ns-train neurad-b200 ...`, `ns-render`, `ns-eval` and
`eval_setup` use it like any other method.  What changes for the reference: `get_nff_outputs` -- the whole of
`neurad.py:368-421` in eval mode -- becomes one call into libb200nerf.so (ray sampling, both proposal rounds, main field,
compositing, appearance), `get_outputs_for_camera_ray_bundle` renders an image in ONE call instead of the 32 768-ray chunk
loop (`neurad.py:650-659`), and in eval mode the rgb / lidar decoders run on the library's tcgen05 kernels.  Parameters stay
the reference's own `nn.Parameter`s in the `implementation="torch"` layout (bound zero-copy by pointer), so checkpoints,
optimizers and `state_dict()` are untouched.  Training (grad mode) falls through to the reference's own module walk.

Nothing in `neurad-studio_b200/` imports this file; `oracle/make_golden_reference_recipe.py` builds its model through the
reference's own config system and `discover_methods()` and checks it against the reference's torch path before writing
the golden data of `tests/test_reference_recipe.py`.
"""
from __future__ import annotations

from copy import deepcopy
from dataclasses import dataclass, field
from typing import Dict, Optional, Tuple, Type

import torch
from torch import Tensor

from nerfstudio.cameras.rays import RayBundle
from nerfstudio.configs.method_configs import method_configs
from nerfstudio.models.neurad import NeuRADModel, NeuRADModelConfig
from nerfstudio.plugins.types import MethodSpecification

import neurad_studio_b200 as nsb
from neurad_studio_b200 import nerfstudio_api as _api


def config_from_reference(model: NeuRADModel) -> nsb.NeuRADConfig:
    """The numbers of the reference model's config tree that shape the path (neurad.py:97-162, neurad_field.py:44-75,
    155-182, neurad_encoding.py:34-82) as the backend's flat config."""
    mc = model.config

    def grid(src) -> nsb.NeuRADHashEncodingConfig:
        def settings(s):
            return nsb.HashGridSettings(s.hashgrid_dim, s.num_levels, s.base_res, s.max_res, s.log2_hashmap_size)

        return nsb.NeuRADHashEncodingConfig(static=settings(src.static), actor=settings(src.actor),
                                            actor_scale=float(src.actor.actor_scale), flip_prob=float(src.actor.flip_prob))

    sp = mc.sampling
    if mc.num_proposal_rounds != 2 or not mc.field.use_sdf or not mc.use_temporal_appearance:
        raise NotImplementedError("the b200 backend implements NeuRAD's default structure: 2 proposal rounds, SDF field, "
                                  "temporal appearance embedding")
    return nsb.NeuRADConfig(
        grid=grid(mc.field.grid), proposal_grid_1=grid(sp.proposal_field_1.grid), proposal_grid_2=grid(sp.proposal_field_2.grid),
        sampling=nsb.SamplingSettings(num_proposal_samples=tuple(sp.num_proposal_samples), num_nerf_samples=sp.num_nerf_samples,
                                      power_lambda=sp.power_lambda, power_scaling=sp.power_scaling, sky_distance=sp.sky_distance,
                                      single_jitter=sp.single_jitter),
        geo_hidden_dim=mc.field.geo_hidden_dim, nff_hidden_dim=mc.field.nff_hidden_dim, nff_out_dim=mc.field.nff_out_dim,
        num_multisamples=mc.field.num_multisamples, appearance_dim=mc.appearance_dim,
        temporal_appearance_freq=mc.temporal_appearance_freq, rgb_upsample_factor=mc.rgb_upsample_factor,
        rgb_hidden_dim=mc.rgb_hidden_dim, actor_bbox_padding=tuple(mc.dynamic_actors.actor_bbox_padding),
        static_scale=float(model.scene_box.aabb.max()), duration=float(model._duration),
        num_sensors=model.appearance_embedding.num_embeddings // model._num_embeds_per_sensor,
        n_actors=int(model.dynamic_actors.n_actors),
    )


@dataclass
class B200NeuRADModelConfig(NeuRADModelConfig):
    """NeuRADModelConfig with the B200 backend.  `implementation` stays "torch": the parameters then have the layout the
    library binds by pointer (fp32 `[L*T, F]` tables, nn.Linear MLPs), and checkpoints interchange with the reference's
    torch mode."""

    _target: Type = field(default_factory=lambda: B200NeuRADModel)
    implementation: str = "torch"
    eval_num_rays_per_chunk: int = 1 << 22  # one launch per image: the chunk loop exists for the torch path's memory
    b200_decoders: bool = True
    """Run rgb_decoder / lidar_decoder on the library's kernels in eval mode (False: the reference's own modules)."""


class B200NeuRADModel(NeuRADModel):
    """`NeuRADModel` whose eval-mode NFF path is the sm_100a library."""

    config: B200NeuRADModelConfig

    def populate_modules(self):
        if self.config.implementation != "torch":
            raise ValueError("B200NeuRADModel binds the torch-layout parameters: implementation must be 'torch'")
        super().populate_modules()
        self._b200_uid = next(_api._UIDS)
        self._b200_cfg: Optional[nsb.NeuRADConfig] = None

    # ---------------------------------------------------------------------------------------------- binding
    _B200_PREFIXES = ("field.", "proposal_fields.", "lidar_decoder.", "appearance_embedding.", "dynamic_actors.")

    def _b200_tensors(self) -> Dict[str, Tensor]:
        """The reference's own parameters / buffers of this path under their state_dict names (no copies)."""
        out: Dict[str, Tensor] = {}
        for k, v in list(self.named_parameters()) + list(self.named_buffers()):
            if k.startswith(self._B200_PREFIXES) and ".hashgrid.actors." not in k:  # aliases of `dynamic_actors`
                out[k] = v
        return out

    def _b200_bind(self):
        be = _api.get_backend(self.appearance_embedding.weight.device)
        tensors = self._b200_tensors()
        token = (self._b200_uid, tuple(t._version for t in tensors.values()), tuple(t.data_ptr() for t in tensors.values()))
        if getattr(be, "_owner", None) != token:  # another model (or an optimizer step / checkpoint load) came in between
            if self._b200_cfg is None:
                self._b200_cfg = config_from_reference(self)
            params = dict(tensors)
            params["static_scale"] = self.scene_box.aabb.max()
            be.load_params(self._b200_cfg, params)  # both rounds -> proposal_fields[1], the reference's effective behaviour
            be._owner = token
        return be

    # ---------------------------------------------------------------------------------------------- hot path
    def get_nff_outputs(self, ray_bundle: RayBundle, calc_lidar_losses: bool = False) -> Dict[str, Tensor]:
        """neurad.py:368-421.  Inference: one fused launch pair.  Training / grad mode: the reference's own walk."""
        if self.training or (torch.is_grad_enabled() and any(p.requires_grad for p in self.field.parameters())):
            return super().get_nff_outputs(ray_bundle, calc_lidar_losses)
        be = self._b200_bind()
        md = ray_bundle.metadata
        rays = {"origins": ray_bundle.origins, "directions": ray_bundle.directions, "pixel_area": ray_bundle.pixel_area,
                "times": ray_bundle.times}
        for key, val in (("nears", ray_bundle.nears), ("fars", ray_bundle.fars), ("sensor_idx", md.get("sensor_idxs")),
                         ("is_lidar", md.get("is_lidar"))):
            if val is not None:
                rays[key] = val
        if "sensor_idx" not in rays:  # neurad.py:425-428: the viewer's fallback sensor
            rays["sensor_idx"] = torch.full_like(ray_bundle.pixel_area, self.fallback_sensor_idx.value, dtype=torch.long)
        with torch.no_grad():
            out = be.render(rays)
        # the reference's function also edits the bundle in place (pixel areas scaled, far clamp, nears filled in:
        # neurad.py:370, 445-449); callers downstream see the same bundle they would have seen
        self._scale_pixel_area(ray_bundle)
        sky = self.config.sampling.sky_distance
        if ray_bundle.fars is not None:
            ray_bundle.fars.clamp_max_(sky)
        else:
            ray_bundle.fars = torch.full_like(ray_bundle.pixel_area, sky)
        if ray_bundle.nears is None:
            ray_bundle.nears = torch.zeros_like(ray_bundle.fars)
        return {k: out[k] for k in ("features", "depth", "accumulation", "prop_depth_0", "prop_depth_1")}

    def decode_features(self, features: Tensor, patch_size: Tuple[int, int], is_lidar: Optional[Tensor] = None,
                        intensity_for_cam: bool = False):
        """neurad.py:337-366.  Eval mode: lidar MLP and camera CNN on the library's tcgen05 kernels (channels-last in and
        out, so the reference's two permutes disappear); training: the reference's modules (BatchNorm statistics, autograd)."""
        if self.training or torch.is_grad_enabled() or not self.config.b200_decoders:
            return super().decode_features(features, patch_size, is_lidar, intensity_for_cam)
        be = self._b200_bind()
        if is_lidar is None:
            lidar_features, cam_features = features[:0], features
        else:
            lidar_features, cam_features = features[is_lidar[..., 0]], features[~is_lidar[..., 0]]
        lin = [m for m in self.lidar_decoder.layers if isinstance(m, torch.nn.Linear)]

        def lidar_head(x):
            return be.mlp_fwd(x, [m.weight for m in lin], [m.bias for m in lin]).split(1, dim=-1)

        if intensity_for_cam:
            intensity, ray_drop_logit = lidar_head(features)
        elif lidar_features.numel() > 0:
            intensity, ray_drop_logit = lidar_head(lidar_features)
        else:
            intensity, ray_drop_logit = None, None
        intensity = intensity.sigmoid() if intensity is not None else None
        sd = self.rgb_decoder.state_dict()
        token = (self._b200_uid, tuple(v._version for v in sd.values()), tuple(v.data_ptr() for v in sd.values()))
        if getattr(be, "_dec_owner", None) != token:
            be.set_rgb_decoder(sd, prefix="", bn_eps=self.rgb_decoder[2].main_branch[1].eps)
            be._dec_owner = token
        rgb = be.rgb_decode(cam_features.reshape(-1, *patch_size, cam_features.shape[-1]))  # [B,h,w,C] -> [B,3h,3w,3]
        return rgb, intensity, ray_drop_logit


def _make_spec() -> MethodSpecification:
    cfg = deepcopy(method_configs["neurad"])
    cfg.method_name = "neurad-b200"
    ref = cfg.pipeline.model
    fields = {k: v for k, v in vars(ref).items() if k not in ("_target", "implementation", "eval_num_rays_per_chunk")}
    cfg.pipeline.model = B200NeuRADModelConfig(**fields)
    return MethodSpecification(config=cfg, description="NeuRAD with the B200-native (sm_100a) neural-feature-field backend")


spec = _make_spec()
