"""Drop-in check of this ``KeypointNeRF`` as the reference's ``KeypointNeRFLightningModule`` drives it, against the
reference's own renderings (``tests/golden/dropin_sweep.npz``, written by ``tests/golden/make_golden.py``).

The golden holds the names and shapes of the reference module's ``state_dict``, the checksum of a checkpoint made from seeds
for exactly those names, the checksum of the sweep's seeded inputs, and the 8-bit renderings of a two-camera sweep that the reference's ``render_novel_views``
(``src/model.py:474-507``) made with that checkpoint.  Here the same checkpoint goes through a strict ``load_state_dict`` of a
module that holds this class as ``model`` (what the reference's ``load_ckpt``, ``src/model.py:113-117``, does), and the sweep
makes the same calls: ``attach_im_feat`` once, then ``render_pifu_nerf`` per camera with the reference's keyword arguments
(``src/model.py:453-473``), ``tex_fg_fine`` clamped to [0, 1] and scaled to 8 bits.  There is no GPU here, so the CUDA
marcher is replaced by a stand-in that answers ``set_scene`` / ``render`` with the CPU oracle: what is under test is everything
ABOVE the C ABI -- state_dict keys, encoders, feature caching, argument marshalling, output dict -- and the images must agree
with the reference's.
"""
import json
import math
import os

import numpy as np
import torch

from tests.util import GOLDEN, seeded_checkpoint, state_dict_checksum, sweep_checksum, sweep_inputs


class OracleMarcher:
    """Stand-in for ``RayMarcher`` (same ``set_scene`` / ``render`` keywords) that shades with the CPU oracle."""

    def __init__(self, weights):
        from oracle import kpnerf_oracle as O
        self.O, self.fw = O, O.fold_weights(weights)
        self.scene_binds = 0

    def set_scene(self, *, KRT, extrin, kpt3d, bounds, feat64, feat8, feat_tex, img, fg, width, height, znear, zfar, nml_scale):
        n = lambda t: t.detach().float().contiguous().numpy()
        V = img.shape[0]
        self.scene = {"n_views": V, "KRT": n(KRT).reshape(V, 4, 4), "extrin": n(extrin).reshape(V, 4, 4), "kpt3d": n(kpt3d)[None],
                      "bounds": n(bounds).reshape(1, 2, 3), "feat64": n(feat64), "feat8": n(feat8), "feat_tex": n(feat_tex),
                      "img": n(img), "fg": fg.reshape(V, 1, *fg.shape[-2:]).numpy().astype(bool), "width": float(width),
                      "height": float(height), "znear": float(znear), "zfar": float(zfar), "nml_scale": float(nml_scale)}
        self.scene_binds += 1

    def render(self, *, K, RT, znear, zfar, x0, y0, step, nx, ny, S_c, S_f=0, fine=False, out_device=None, engine=0, ert_eps=0.0,
               step_y=0):
        O = self.O
        target = {"K": K.reshape(-1, 4, 4).numpy(), "RT": RT.reshape(-1, 4, 4).numpy(), "znear": znear, "zfar": zfar}
        ys = torch.arange(ny) * (step_y or step) + y0
        xs = torch.arange(nx) * step + x0
        yy, xx = torch.meshgrid(ys, xs, indexing="ij")
        pix = torch.stack([xx, yy], -1).reshape(-1, 2).float()
        flat = O.render_pixels(self.scene, self.fw, target, pix, S_c, S_f, fine)
        img = lambda v: v.reshape(ny, nx, 3).permute(2, 0, 1).contiguous()
        res = {"tex_fg": img(flat["tex_fg"]), "depth": flat["depth"].reshape(ny, nx), "alpha": flat["alpha"].reshape(ny, nx)}
        if fine:
            res.update({"tex_fg_fine": img(flat["tex_fg_fine"]), "depth_fine": flat["depth_fine"].reshape(ny, nx),
                        "alpha_fine": flat["alpha_fine"].reshape(ny, nx), "sdf": flat["sdf"].reshape(ny, nx)})
        return res


def test_novel_view_sweep_matches_reference_renderings(tmp_path):
    from keypointnerf_b200 import synthetic as syn
    from keypointnerf_b200.config import default_cfg
    from keypointnerf_b200.model import KeypointNeRF
    g = np.load(os.path.join(GOLDEN, "dropin_sweep.npz"))
    meta = json.loads(bytes(g["meta"]).decode())
    want = g["renderings"]
    n_kpt = meta["n_kpt"]
    cfg = default_cfg(n_kpt)
    cfg["models"]["KeypointNeRF"]["dr_kwargs"].update(sample_per_ray_c=meta["S_c"], sample_per_ray_f=meta["S_f"])

    class Module(torch.nn.Module):   # the reference's LightningModule holds the network as `model`
        def __init__(self):
            super().__init__()
            self.model = KeypointNeRF(cfg)

    mine = Module().eval()
    shapes = {k: list(v.shape) for k, v in mine.state_dict().items()}
    ref_shapes = {k: s for k, s in meta["state_dict"]}
    assert shapes == ref_shapes, f"state_dict differs from the reference's: {sorted(set(shapes.items()) ^ set(ref_shapes.items()))[:8]}"
    sd = seeded_checkpoint(meta["state_dict"], syn.make_weights(n_kpt))
    assert state_dict_checksum(sd) == bytes(g["ckpt_sha256"]).decode(), "the seeded checkpoint is not the one the golden was made with"
    sd["model.vgg_loss.vgg.slice1.0.weight"] = np.zeros(4, np.float32)   # the real model owns a frozen VGG19 (src/model.py:608)
    path = tmp_path / "latest.ckpt"
    torch.save({"state_dict": {k: torch.from_numpy(v) for k, v in sd.items()}, "epoch": 3, "global_step": 7}, path)
    mine.load_state_dict(torch.load(path)["state_dict"])             # strict, as the reference's load_ckpt
    net = mine.model
    fake = OracleMarcher({k: v.numpy() for k, v in net.state_dict().items() if not k.startswith(("geo_", "tex_", "sp_"))})
    net.marcher = lambda: fake

    # the reference's decode_batch (src/model.py:309-409): index 0 of the batch is the target view, 1.. the source views
    batch, cams = sweep_inputs(n_kpt)
    assert sweep_checksum(batch, cams) == bytes(g["input_sha256"]).decode(), "seeded inputs drifted from the ones the golden run used"
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    im = t(batch["images"][0, 1:])
    V, s = im.shape[0], im.shape[-1]
    extrin = torch.eye(4).repeat(V, 1, 1)
    extrin[:, :3, :4] = t(batch["Rt"][0, 1:])
    intrin = torch.eye(4).repeat(V, 1, 1)
    intrin[:, :3, :3] = t(batch["K"][0, 1:])
    cam = {"KRT": intrin @ extrin, "K": intrin, "Rt": t(batch["Rt"][0, 1:]), "extrin": extrin, "znear": 2.0, "zfar": 5.0,
           "width": s, "height": s, "nml_scale": 100.0}
    kpt3d = t(batch["kpt3d"])
    sp_data = {"extrin": extrin, "kpt3d": kpt3d}
    dr = net.kwargs["dr_kwargs"]
    got = []
    with torch.no_grad():
        net.attach_im_feat(im)
        for c in cams:
            K, RT = t(c["intrinsics"]), t(c["w2cs"])[None]
            cam_tar = {"K": K, "RT": RT, "KRT": K @ RT, "width": c["im_w"], "height": c["im_h"], "nml_scale": 100.0,
                       "znear": c["znear"], "zfar": c["zfar"]}
            out = net.render_pifu_nerf(net=net, img_in=im, cam_in=cam, cam_tar=cam_tar, tar_img=None, sp_data=sp_data,
                                       objcenter=kpt3d[:, 0, :], fine=dr["fine"], uniform=True, objrad=250., blur=3,
                                       level=max(0, int(math.log(c["im_h"], 2)) - 5), sample_per_ray_c=dr["sample_per_ray_c"],
                                       sample_per_ray_f=dr["sample_per_ray_f"], src_foreground_mask=t(batch["images_masks"][:, 1:]),
                                       bounds=t(batch["bounds"]), mask_at_box=t(batch["mask_at_box"]))
            got.append(out["tex_fg_fine"].clamp(min=0.0, max=1.0).permute(1, 2, 0).numpy())
    got = (np.stack(got) * 255.).astype(np.uint8)
    assert got.shape == want.shape == (2, 64, 64, 3) and want.dtype == np.uint8
    assert fake.scene_binds == 1, "the source-image set must be bound (and encoded) once per sweep, not once per camera"
    d = np.abs(got.astype(np.int32) - want.astype(np.int32))
    assert want.max() > 30, "the test scene renders nothing"
    assert d.max() <= 1, f"8-bit renderings differ by up to {d.max()}"
