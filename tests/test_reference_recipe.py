"""The reference's own "neurad" method recipe (the model `ns-train neurad-b200` builds through the reference's plugin
registry and config system, shrunken hash tables) through the API mirror, against what the reference's torch walk
computed on the same parameters and rays: `get_nff_outputs` on a flat batch, and a camera image and a lidar sweep through
`get_outputs_for_camera_ray_bundle` (one backend call each, decoders on the library's operators), and `get_nff_outputs`
again after an in-place parameter update.  The fixture tests/golden/reference_recipe.npz is written by
oracle/make_golden_reference_recipe.py, which also checks integration/neurad_b200_plugin.py against the same reference
outputs (the plugin subclasses the reference's classes and cannot be imported without it).  On the CPU the backend is
tests/fake_backend.py (oracle + host emulation); on the GPU it is the library."""
import pytest
import torch

import neurad_studio_b200 as nsb
from tests.helpers import load_golden


def rel_to_max(a, b):
    return (a.cpu() - b).abs().max().item() / (b.abs().max().item() + 1e-30)


@pytest.fixture
def fake_backend(monkeypatch):
    from neurad_studio_b200 import nerfstudio_api
    from tests.fake_backend import FakeBackend

    be = FakeBackend()
    monkeypatch.setattr(nerfstudio_api, "get_backend", lambda device: be)
    return be


def _recipe(dev):
    from neurad_studio_b200 import scene
    from neurad_studio_b200.nerfstudio_api import NeuRADModel

    meta, g = load_golden("reference_recipe.npz")
    cfg = nsb.small_config(n_actors=meta["n_actors"], log2_main=meta["log2_main"], log2_prop=meta["log2_prop"])
    trajs = scene.make_trajectories(meta["n_actors"], cfg.duration, seed=meta["traj_seed"])
    dec = scene.make_rgb_decoder_params(seed=meta["decoder_seed"])
    for k, v in dec.items():  # the decoder is re-created from its generator, not stored
        ref = g["decoder_sum"][k].item()
        assert abs(v.double().sum().item() - ref) <= 1e-6 * max(1.0, v.double().abs().sum().item()), k
    model = NeuRADModel(cfg, trajs)
    model.load_reference_state_dict(g["param"])
    model.rgb_decoder.load_state_dict({k[len("rgb_decoder."):]: v for k, v in dec.items()}, strict=False)
    return model.to(dev).eval(), meta, g


def _bundle(rays, dev, sl=slice(None)):
    from neurad_studio_b200.nerfstudio_api import RayBundle

    return RayBundle(origins=rays["origins"][sl].to(dev), directions=rays["directions"][sl].to(dev),
                     pixel_area=rays["pixel_area"][sl].to(dev), times=rays["times"][sl].to(dev),
                     metadata={"is_lidar": rays["is_lidar"][sl].to(dev).bool(), "sensor_idxs": rays["sensor_idx"][sl].to(dev)})


def _check_flat_batch(dev, be=None):
    """get_nff_outputs on a flat batch of camera and lidar rays; with `be` (the CPU stand-in) also what reaches the
    backend: one render per call, parameters bound once and again only after they change."""
    model, _, g = _recipe(dev)
    calls, loads = [], []
    if be is not None:
        render, load_params = be.render, be.load_params
        be.render = lambda *a, **k: (calls.append("render"), render(*a, **k))[1]
        be.load_params = lambda *a, **k: (loads.append(1), load_params(*a, **k))[1]
    rb = _bundle(g["flat_ray"], dev)
    with torch.no_grad():
        ours = model.get_nff_outputs(rb)
    ref = g["flat_ref"]
    assert set(ours) == set(ref) == {"features", "depth", "accumulation", "prop_depth_0", "prop_depth_1"}
    for k in ref:
        assert ours[k].shape == ref[k].shape and rel_to_max(ours[k], ref[k]) < 1e-4, (k, rel_to_max(ours[k], ref[k]))
    # the fused path leaves the caller's bundle as it is; _scale_pixel_area (the module walk's first step) gives the pixel
    # areas the reference's function leaves there
    assert torch.equal(model._scale_pixel_area(rb).pixel_area.cpu(), g["flat_bundle"]["pixel_area"])
    with torch.no_grad():
        again = model.get_nff_outputs(rb)
        model._param("field.hashgrid.static_grid.hash_table").mul_(0.5)  # in place, as an optimizer step does
        changed = model.get_nff_outputs(rb)
    assert torch.equal(again["features"], ours["features"])
    if be is not None:
        assert calls == ["render"] * 3 and loads == [1, 1]
    ref = g["flat_updated_ref"]
    for k in ref:
        assert rel_to_max(changed[k], ref[k]) < 1e-4, (k, rel_to_max(changed[k], ref[k]))


def _check_image_and_lidar(dev):
    """get_outputs_for_camera_ray_bundle (neurad.py:623-675), the function the metric is defined on: a 2-D bundle is
    rendered at its [1::3, 1::3] pixels and decoded to a full-resolution rgb image; a 1-D bundle is a lidar sweep."""
    model, meta, g = _recipe(dev)
    h, w = meta["image_hw"]
    rays = g["image_ray"]
    cam = _bundle(rays, dev, slice(0, h * w))._map(lambda t: t.reshape(h, w, -1))
    cam.metadata.pop("is_lidar")  # camera bundles of the eval path carry no is_lidar (cameras.py generate_rays)
    ours = model.get_outputs_for_camera_ray_bundle(cam)
    ref = g["image_ref"]
    assert ours["rgb"].shape == (h, w, 3) and rel_to_max(ours["rgb"], ref["rgb"]) < 1e-4
    assert rel_to_max(ours["depth"].reshape(-1), ref["depth"].reshape(-1)) < 1e-4
    assert rel_to_max(ours["intensity"].reshape(-1), ref["intensity"].reshape(-1)) < 1e-4
    out = model.get_outputs_for_camera_ray_bundle(_bundle(rays, dev, slice(h * w, None)))
    ref = g["lidar_ref"]
    n = meta["lidar_rays"]
    assert out["depth"].shape == (n, 1) and rel_to_max(out["depth"], ref["depth"]) < 1e-4
    assert rel_to_max(out["intensity"], ref["intensity"]) < 1e-4 and rel_to_max(out["ray_drop_logits"], ref["ray_drop_logits"]) < 1e-4


def test_renders_the_reference_recipe_like_the_reference(fake_backend):
    _check_flat_batch("cpu", fake_backend)


def test_image_and_lidar_entry_points_match_the_reference(fake_backend):
    _check_image_and_lidar("cpu")


@pytest.mark.gpu
def test_renders_the_reference_recipe_like_the_reference_on_gpu():
    _check_flat_batch("cuda")


@pytest.mark.gpu
def test_image_and_lidar_entry_points_match_the_reference_on_gpu():
    _check_image_and_lidar("cuda")
