"""Generate tests/golden/pins_64x96_pad4.npz from the UNMODIFIED reference.

    MVSNERF_REFERENCE_ROOT=<checkout of apchenstu/mvsnerf> python tests/golden/make_golden_pins.py

Records what tests/test_oracle_pins.py compares the oracle and the host mirrors against, in the order that module
runs: the checkpoint's MLP tensors (as digests); a train-mode volume and 24-sample render of scene seed 11; an
eval-mode volume of scene seed 12 with the running statistics the seed-11 forward left behind; ray_marcher and
get_ndc_coordinate on scene seed 13.  The scenes come from mvsnerf_b200.synthetic; their inputs are stored as digests
(the test regenerates them and checks the digests) because their per-pixel noise does not compress.  The volumes are
stored at a seeded subset of voxels plus per-channel sums; the seed-11 render is of the ORACLE's volume, so that the
test can feed the renderer the same volume without storing it whole.
"""
import hashlib
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import mvsnerf_oracle as orc  # noqa: E402
from oracle import ref_shim  # noqa: E402
from mvsnerf_b200 import synthetic  # noqa: E402


def digest(a) -> str:
    """sha256 of an array's dtype, shape and bytes (same definition as in tests/test_oracle_pins.py)."""
    a = np.ascontiguousarray(a.detach().cpu().numpy() if torch.is_tensor(a) else a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


def scene_digest(sc) -> str:
    parts = [sc.imgs_raw, sc.imgs_norm, sc.proj_mats, sc.pose_source["w2cs"], sc.pose_source["c2ws"],
             sc.pose_source["intrinsics"], sc.c2w_target, sc.directions, np.array(sc.near_far, dtype=np.float64)]
    return hashlib.sha256("".join(digest(p) for p in parts).encode()).hexdigest()


def volume_sample(vol, n, seed):
    g = torch.Generator().manual_seed(seed)
    idx = torch.randperm(vol[0, 0].numel(), generator=g)[:n]
    return idx.numpy(), vol[0].reshape(8, -1)[:, idx].numpy(), vol[0].double().sum((1, 2, 3)).numpy()


def main():
    torch.manual_seed(0)
    torch.set_num_threads(os.cpu_count())
    R = ref_shim.build_reference(N_samples=24)
    ref = R.ref
    weights = orc.load_weights_npz(os.path.join(HERE, "mvsnerf_v0_weights.npz"))
    out = {}

    sd = R.render_kwargs["network_fn"].state_dict()
    out["ckpt_mlp_keys"] = np.array(list(sd.keys()))
    out["ckpt_mlp_sha256"] = np.array([digest(v) for v in sd.values()])
    out["ckpt_mvs_count"] = np.int64(len(R.mvsnet.state_dict()))

    # ---- seed 11: train-mode volume, then the reference renderer on the oracle's volume ----
    sc = synthetic.make_scene(64, 96, pad=4, seed=11)
    with torch.no_grad():
        vol_ref, _, _ = R.mvsnet(sc.imgs_norm, sc.proj_mats, sc.near_far, pad=sc.pad)
    vol = orc.encode_volume(sc.imgs_norm, sc.proj_mats, sc.near_far, sc.pad, weights)
    rays = synthetic.scene_rays(sc)[::5]
    with torch.no_grad():
        xyz, ro, rd, z = ref.ray_utils.ray_marcher(rays, N_samples=24)
        ndc = ref.utils.get_ndc_coordinate(sc.pose_source["w2cs"][0], sc.pose_source["intrinsics"][0].clone(),
                                           xyz, torch.tensor([sc.W - 1, sc.H - 1]), near=sc.near_far[0],
                                           far=sc.near_far[1], pad=sc.pad * 1.0)
        rgb_ref, _, _, depth_ref, _, _ = ref.renderer.rendering(
            R.args, sc.pose_source, xyz, ndc, z, ro, rd, vol, sc.imgs_raw, **R.render_kwargs)
    idx, sub, chsum = volume_sample(vol_ref, 8192, 11)
    out.update({"s11/scene_sha256": np.array(scene_digest(sc)), "s11/vox_idx": idx, "s11/volume_sub": sub,
                "s11/volume_chsum": chsum, "s11/rgb": rgb_ref.numpy(), "s11/depth": depth_ref.numpy()})
    rgb_o, _ = orc.render_rays(rays, vol, sc.imgs_raw, sc.pose_source, weights, sc.H, sc.W, sc.near_far,
                               float(sc.pad), n_samples=24)
    print("s11: volume Linf oracle vs reference", (vol - vol_ref).abs().max().item(),
          "rgb Linf on the oracle's volume", (rgb_o - rgb_ref).abs().max().item())

    # ---- seed 12: eval mode with the running statistics the seed-11 train-mode forward left behind ----
    sc = synthetic.make_scene(64, 96, pad=4, seed=12)
    R.mvsnet.eval()
    with torch.no_grad():
        vol_ref, _, _ = R.mvsnet(sc.imgs_norm, sc.proj_mats, sc.near_far, pad=sc.pad)
    R.mvsnet.train()
    idx, sub, chsum = volume_sample(vol_ref, 8192, 12)
    out.update({"s12/scene_sha256": np.array(scene_digest(sc)), "s12/vox_idx": idx, "s12/volume_eval_sub": sub,
                "s12/volume_eval_chsum": chsum})
    for k, v in R.mvsnet.state_dict().items():
        if k.endswith(("running_mean", "running_var", "num_batches_tracked")):
            out["s12/stats/" + k] = v.numpy()

    # ---- seed 13: ray_marcher / get_ndc_coordinate, bit for bit ----
    sc = synthetic.make_scene(64, 96, pad=4, seed=13)
    rays = synthetic.scene_rays(sc)[::9].contiguous()
    out["s13/scene_sha256"] = np.array(scene_digest(sc))
    for lindisp in (False, True):
        xyz, ro, rd, z = ref.ray_utils.ray_marcher(rays, N_samples=20, lindisp=lindisp)
        ndc = ref.utils.get_ndc_coordinate(sc.pose_source["w2cs"][0], sc.pose_source["intrinsics"][0].clone(), xyz,
                                           torch.tensor([sc.W - 1, sc.H - 1]), near=sc.near_far[0],
                                           far=sc.near_far[1], pad=4.0, lindisp=lindisp)
        tag = f"s13/lindisp{int(lindisp)}/"
        out.update({tag + "xyz": xyz.numpy(), tag + "rd": rd.numpy(), tag + "z": z.numpy(), tag + "ndc": ndc.numpy()})

    path = os.path.join(HERE, "pins_64x96_pad4.npz")
    np.savez_compressed(path, **out)
    print(os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
