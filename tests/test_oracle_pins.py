"""CPU: the oracle restatement and the host mirrors next to what the unmodified reference computed on fresh seeded
scenes (tests/golden/make_golden_pins.py, which imports the reference through oracle/ref_shim.py).  The scenes are
regenerated from their seeds; a digest of the inputs the reference consumed checks that they are the same scenes."""
import hashlib
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import mvsnerf_oracle as orc
from mvsnerf_b200 import synthetic


def digest(a) -> str:
    """sha256 of an array's dtype, shape and bytes (same definition as in tests/golden/make_golden_pins.py)."""
    a = np.ascontiguousarray(a.detach().cpu().numpy() if torch.is_tensor(a) else a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


def scene_digest(sc) -> str:
    parts = [sc.imgs_raw, sc.imgs_norm, sc.proj_mats, sc.pose_source["w2cs"], sc.pose_source["c2ws"],
             sc.pose_source["intrinsics"], sc.c2w_target, sc.directions, np.array(sc.near_far, dtype=np.float64)]
    return hashlib.sha256("".join(digest(p) for p in parts).encode()).hexdigest()


@pytest.fixture(scope="module")
def pins():
    z = np.load(os.path.join(GOLDEN, "pins_64x96_pad4.npz"))
    return {k: z[k] if z[k].dtype.kind == "U" else torch.from_numpy(z[k]) for k in z.files}


def recorded_scene(pins, tag, seed):
    sc = synthetic.make_scene(64, 96, pad=4, seed=seed)
    assert scene_digest(sc) == str(pins[tag + "/scene_sha256"]), "synthetic.make_scene no longer gives the recorded scene"
    return sc


def test_weights_fixture_matches_checkpoint(pins, weights):
    keys, sha = pins["ckpt_mlp_keys"], pins["ckpt_mlp_sha256"]
    assert len(keys) == sum(1 for k in weights if k.startswith("mlp/")) == 22
    for k, h in zip(keys, sha):
        assert digest(weights["mlp/" + str(k)]) == str(h), k
    n = sum(1 for k in weights if k.startswith("mvs/"))
    assert n == int(pins["ckpt_mvs_count"]) == 110


def test_live_reference_vs_oracle(pins, weights):
    sc = recorded_scene(pins, "s11", 11)                 # h=16,w=24 -> 24x32 padded: legal
    vol = orc.encode_volume(sc.imgs_norm, sc.proj_mats, sc.near_far, sc.pad, weights)
    idx = pins["s11/vox_idx"]
    assert (vol[0].reshape(8, -1)[:, idx] - pins["s11/volume_sub"]).abs().max() < 2e-4
    assert torch.allclose(vol[0].double().sum((1, 2, 3)), pins["s11/volume_chsum"], rtol=1e-4, atol=0.5)
    # the reference rendered this same (oracle) volume: the comparison isolates the renderer
    rays = synthetic.scene_rays(sc)[::5]
    rgb, depth = orc.render_rays(rays, vol, sc.imgs_raw, sc.pose_source, weights, sc.H, sc.W,
                                 sc.near_far, float(sc.pad), n_samples=24)
    assert (rgb - pins["s11/rgb"]).abs().max() < 2e-6
    assert (depth - pins["s11/depth"]).abs().max() < 1e-5


def test_live_reference_eval_mode_vs_oracle(pins, weights):
    """MVSNet.eval() (running-statistics BatchNorm, models.py:661-685 through the InPlaceABN stub) vs the oracle's eval_mode."""
    sc = recorded_scene(pins, "s12", 12)
    # the running statistics of the reference module after the seed-11 train-mode forward, not the checkpoint's: every
    # train-mode forward of the reference updates them in place -- the side effect MVSN_BN_BATCH_UPDATE reproduces
    w = dict(weights)
    w.update({"mvs/" + k[len("s12/stats/"):]: v for k, v in pins.items() if k.startswith("s12/stats/")})
    vol = orc.encode_volume(sc.imgs_norm, sc.proj_mats, sc.near_far, sc.pad, w, eval_mode=True)
    idx, want = pins["s12/vox_idx"], pins["s12/volume_eval_sub"]
    assert (vol[0].reshape(8, -1)[:, idx] - want).abs().max() < 2e-4 * max(1.0, float(want.abs().max()))
    assert torch.allclose(vol[0].double().sum((1, 2, 3)), pins["s12/volume_eval_chsum"], rtol=1e-4, atol=0.5)
    vol_train = orc.encode_volume(sc.imgs_norm, sc.proj_mats, sc.near_far, sc.pad, weights)
    assert (vol - vol_train).abs().max() > 0.1          # the two modes differ grossly with this checkpoint (SURVEY App. D)


def test_host_mirrors_of_ray_marcher_and_ndc_vs_live_reference(pins):
    """mvsnerf_b200.backend.ray_marcher / get_ndc_coordinate (what the fine-tuning step calls before `rendering`) against
    the reference's own data/ray_utils.ray_marcher and utils.get_ndc_coordinate, bit for bit."""
    from mvsnerf_b200 import backend
    sc = recorded_scene(pins, "s13", 13)
    rays = synthetic.scene_rays(sc)[::9].contiguous()
    for lindisp in (False, True):
        tag = f"s13/lindisp{int(lindisp)}/"
        xyz, ro, rd, z = backend.ray_marcher(rays, N_samples=20, lindisp=lindisp)
        assert torch.equal(xyz, pins[tag + "xyz"]) and torch.equal(z, pins[tag + "z"]) and torch.equal(rd, pins[tag + "rd"])
        inv = torch.tensor([sc.W - 1, sc.H - 1])
        b = backend.get_ndc_coordinate(sc.pose_source["w2cs"][0], sc.pose_source["intrinsics"][0].clone(), xyz, inv,
                                       near=sc.near_far[0], far=sc.near_far[1], pad=4.0, lindisp=lindisp)
        assert torch.equal(b, pins[tag + "ndc"])
