"""TEST INFRASTRUCTURE ONLY -- golden vectors of the reference's own "neurad" method recipe (needs the reference tree,
see oracle/ref_import.py):

    python -m oracle.make_golden_reference_recipe      ->  tests/golden/reference_recipe.npz

Builds the model the way `ns-train neurad-b200` does -- the reference's plugin registry finds
`integration/neurad_b200_plugin.py`, the reference's config system sets the model up (shrunken hash tables) -- and runs
the reference's own torch walk on it: `NeuRADModel.get_nff_outputs` on a flat ray batch (outputs and the pixel areas it
leaves in the caller's bundle), and the parts `get_outputs_for_camera_ray_bundle` is made of on a 12 x 9 camera image and a lidar
sweep, and `get_nff_outputs` once more after an in-place update of the static hash table.  Before writing, it runs the
plugin's own overridden entry points (`B200NeuRADModel`, backend = tests/fake_backend.py) on the same inputs and asserts
that they match the reference, dispatch once per call and re-bind only after the update: the plugin subclasses the
reference's classes, so this is the one place it can run.  Stores the hot-path parameters, the rays and the reference's
outputs; the rgb decoder's parameters come from `scene.make_rgb_decoder_params` and are stored as checksums only.
tests/test_reference_recipe.py replays them through the API mirror with no reference installed.
"""
from __future__ import annotations

import dataclasses
import os
import sys
import warnings
from copy import deepcopy

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import neurad_studio_b200 as nsb  # noqa: E402
from neurad_studio_b200 import scene  # noqa: E402
from oracle import ref_import  # noqa: E402
from oracle.make_golden import _save  # noqa: E402

META = dict(n_actors=3, traj_seed=5, log2_main=9, log2_prop=8, decoder_seed=2, flat_rays=96, flat_seed=9,
            image_hw=(12, 9), lidar_rays=40, image_seed=11)


def small_cfg():
    return nsb.small_config(n_actors=META["n_actors"], log2_main=META["log2_main"], log2_prop=META["log2_prop"])


def _methods():
    ref_import.install(full=True)
    warnings.filterwarnings("ignore")
    from oracle.ref_driver import _install_nerfacc_restatements

    _install_nerfacc_restatements()
    import nerfstudio.models.neurad as ref_neurad

    ref_neurad.VGGPerceptualLossPix2Pix = lambda: torch.nn.Identity()
    os.environ["NERFSTUDIO_METHOD_CONFIGS"] = "neurad-b200=integration.neurad_b200_plugin:spec"
    from nerfstudio.plugins.registry import discover_methods

    return discover_methods()[0]


def build_model():
    methods = _methods()
    from nerfstudio.data.scene_box import SceneBox
    from nerfstudio.field_components.field_heads import FieldHeadNames

    from integration.neurad_b200_plugin import config_from_reference

    small = small_cfg()
    mc = deepcopy(methods["neurad-b200"].pipeline.model)
    for f, g in zip(mc.fields, (small.grid, small.proposal_grid_1, small.proposal_grid_2)):
        f.grid.static.log2_hashmap_size, f.grid.actor.log2_hashmap_size = g.static.log2_hashmap_size, g.actor.log2_hashmap_size
    trajs = scene.make_trajectories(META["n_actors"], small.duration, seed=META["traj_seed"])
    scene_box = SceneBox(aabb=torch.tensor([[-100.0, -100.0, -10.0], [100.0, 100.0, 30.0]]))
    metadata = {"duration": small.duration, "sensor_idx_to_name": {i: f"s{i}" for i in range(7)}, "trajectories": trajs}
    torch.manual_seed(META["traj_seed"])  # the reference's default initialisation of everything the tables do not cover
    model = mc.setup(scene_box=scene_box, num_train_data=1, metadata=metadata)
    with torch.no_grad():  # the default 1e-3 table init renders a constant; make the outputs informative
        for k, p in model.named_parameters():
            if k.endswith("hash_table"):
                p.uniform_(-1, 1)
        model.field.mlp_geo.layers[1].bias[0] = 0.5
        model.field.sdf_to_density.beta.fill_(4.0)
    dec = scene.make_rgb_decoder_params(seed=META["decoder_seed"])
    missing, unexpected = model.rgb_decoder.load_state_dict({k[len("rgb_decoder."):]: v for k, v in dec.items()}, strict=False)
    assert not unexpected and all(k.endswith("num_batches_tracked") for k in missing), (missing, unexpected)
    model.eval()
    # the mirror is configured by small_cfg(): it must be what the reference's config tree amounts to
    assert dataclasses.asdict(config_from_reference(model)) == dataclasses.asdict(small), "config drift"

    def _render_weights(self, outputs, ray_samples):  # the reference's CUDA branch (neurad.py:716-717) on CPU tensors
        import nerfacc

        return nerfacc.render_weight_from_alpha(outputs[FieldHeadNames.ALPHA].squeeze(-1))[0]

    model._render_weights = _render_weights.__get__(model)
    params = {k: v.detach().clone() for k, v in model._b200_tensors().items()}
    return model, trajs, small, params, dec


def _bundle(rays, sl=slice(None)):
    from nerfstudio.cameras.rays import RayBundle

    return RayBundle(origins=rays["origins"][sl].clone(), directions=rays["directions"][sl].clone(), pixel_area=rays["pixel_area"][sl].clone(),
                     times=rays["times"][sl].clone(), camera_indices=torch.zeros_like(rays["sensor_idx"][sl]),
                     metadata={"is_lidar": rays["is_lidar"][sl].clone().bool(), "sensor_idxs": rays["sensor_idx"][sl].clone()})


def rel_to_max(a, b):
    return (a - b).abs().max().item() / (b.abs().max().item() + 1e-30)


def _close(ours, ref, what):
    assert ours.shape == ref.shape and rel_to_max(ours, ref) < 1e-4, (what, rel_to_max(ours, ref))


def check_plugin(model, flat_rays, image_rays, arrays, ref_bundle):
    """integration/neurad_b200_plugin.py's overrides (eval mode) against the reference outputs in `arrays`."""
    from integration.neurad_b200_plugin import B200NeuRADModel
    from neurad_studio_b200 import nerfstudio_api
    from tests.fake_backend import FakeBackend

    assert isinstance(model, B200NeuRADModel)
    be = FakeBackend()
    calls, loads = [], []
    render, load_params = be.render, be.load_params
    be.render = lambda *a, **k: (calls.append("render"), render(*a, **k))[1]
    be.load_params = lambda *a, **k: (loads.append(1), load_params(*a, **k))[1]
    nerfstudio_api.get_backend = lambda device: be
    rb = _bundle(flat_rays)
    with torch.no_grad():
        ours = model.get_nff_outputs(rb)
    assert calls == ["render"] and loads == [1]
    assert set(ours) == {k.split("/")[1] for k in arrays if k.startswith("flat_ref/")}
    for k, v in ours.items():
        _close(v, arrays[f"flat_ref/{k}"], k)
    # the same side effects on the caller's bundle as the reference's function
    for k in ("pixel_area", "fars", "nears"):
        assert torch.equal(getattr(rb, k), getattr(ref_bundle, k)), k
    with torch.no_grad():  # untouched parameters are not bound again
        model.get_nff_outputs(_bundle(flat_rays))
    assert loads == [1]
    h, w = META["image_hw"]
    n_cam = h * w
    cam = _bundle(image_rays, slice(0, n_cam)).reshape((h, w))
    cam.metadata.pop("is_lidar")  # camera bundles of the eval path carry no is_lidar (cameras.py generate_rays)
    out = model.get_outputs_for_camera_ray_bundle(cam)
    _close(out["rgb"], arrays["image_ref/rgb"], "rgb")
    for k in ("depth", "intensity"):
        _close(out[k].reshape(-1), arrays[f"image_ref/{k}"].reshape(-1), k)
    out = model.get_outputs_for_camera_ray_bundle(_bundle(image_rays, slice(n_cam, None)))
    for k in ("depth", "intensity", "ray_drop_logits"):
        _close(out[k], arrays[f"lidar_ref/{k}"], f"lidar {k}")
    return be, loads


def main():
    model, trajs, small, params, dec = build_model()
    from nerfstudio.models.neurad import NeuRADModel

    arrays = {f"param/{k}": v for k, v in params.items()}
    arrays.update({f"decoder_sum/{k}": v.double().sum() for k, v in dec.items()})
    # flat batch: get_nff_outputs and the pixel areas it leaves in the caller's bundle
    rays = scene.random_rays(META["flat_rays"], small, seed=META["flat_seed"], trajectories=trajs)
    arrays.update({f"flat_ray/{k}": v for k, v in rays.items()})
    flat_rays = rays
    rb = _bundle(rays)
    with torch.no_grad():
        out = NeuRADModel.get_nff_outputs(model, rb)
    arrays.update({f"flat_ref/{k}": v for k, v in out.items()})
    arrays["flat_bundle/pixel_area"] = rb.pixel_area
    ref_bundle = rb
    # a camera image and a lidar sweep: render at the stride-3 pixels, then the decoders (neurad.py:623-675)
    h, w = META["image_hw"]
    n_cam = h * w
    rays = scene.random_rays(n_cam + META["lidar_rays"], small, seed=META["image_seed"], trajectories=trajs)
    rays["is_lidar"][:n_cam] = 0
    rays["is_lidar"][n_cam:] = 1
    arrays.update({f"image_ray/{k}": v for k, v in rays.items()})
    cam = _bundle(rays, slice(0, n_cam)).reshape((h, w))
    with torch.no_grad():
        sub = cam[1::3, 1::3].reshape((-1,))
        nff = NeuRADModel.get_nff_outputs(model, sub)
        rgb, intensity, _ = NeuRADModel.decode_features(model, nff["features"], patch_size=(h // 3, w // 3), is_lidar=None,
                                                        intensity_for_cam=True)
        arrays.update({"image_ref/rgb": rgb.squeeze(0), "image_ref/depth": nff["depth"], "image_ref/intensity": intensity})
        nff = NeuRADModel.get_nff_outputs(model, _bundle(rays, slice(n_cam, None)))
        _, intensity, drop = NeuRADModel.decode_features(model, nff["features"], patch_size=(1, 1),
                                                         is_lidar=torch.ones(META["lidar_rays"], 1, dtype=torch.bool),
                                                         intensity_for_cam=True)
        arrays.update({"lidar_ref/depth": nff["depth"], "lidar_ref/intensity": intensity, "lidar_ref/ray_drop_logits": drop})
    be, loads = check_plugin(model, flat_rays, rays, arrays, ref_bundle)
    # an in-place update of the static table: the reference's output on the updated parameters, and the plugin's
    with torch.no_grad():
        model.field.hashgrid.static_grid.hash_table.mul_(0.5)
        out = NeuRADModel.get_nff_outputs(model, _bundle(flat_rays))
        arrays.update({f"flat_updated_ref/{k}": v for k, v in out.items()})
        ours = model.get_nff_outputs(_bundle(flat_rays))
    assert loads == [1, 1]
    for k, v in ours.items():
        _close(v, out[k], f"updated {k}")
    assert rel_to_max(out["features"], arrays["flat_ref/features"]) > 1e-3
    print("plugin (B200NeuRADModel on the stand-in backend) == reference: flat batch, image, lidar sweep, after an update")
    _save("reference_recipe.npz", arrays, dict(META, torch=torch.__version__))


if __name__ == "__main__":
    main()
