"""Generate golden vectors by running the UNMODIFIED reference (/root/reference) on CPU.

Run in the build container only (the GPU box has no /root/reference):
    python tests/golden/make_golden.py
Writes tests/golden/<case>.npz for every entry of CASES and dropin_sweep.npz (or only the cases named
on the command line).  Inputs are regenerated from seeds by keypointnerf_b200.synthetic; the .npz files hold the
reference's outputs (and, for the tiny cases, per-sample intermediates captured with forward
hooks), plus an input checksum so that drift in the seeded generators is detected.  To keep every
file under 1 MB, per-sample arrays are stored for a fixed, seeded subset: the tiny cases keep every
valid query point and a sample of the invalid ones (``query_*``, positions ``sel`` of the stage
intermediates index into that subset); the config-size passes with ``rays`` set keep that many rays
of the pass (``rays`` = their row-major indices) for ``contrib_coarse``, ``z_coarse`` and ``z_fine``.

Scenes: "hull" = ellipsoid-silhouette foreground masks (every ray's last sample is invalid, so no
ray sits on the reference's final-sample discontinuity and every ray is compared); "ones" = the
SURVEY.md section 8d recipe the bench runs (kept for the config-1/2 passes of the bench scene).

Harness = SURVEY.md Appendix C: stub modules for kornia / pytorch_lightning / skimage /
imageio, VGGLoss patched out, Tensor.cuda made the identity.
"""
import hashlib
import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))
from keypointnerf_b200 import synthetic as syn  # noqa: E402


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


class _LightningModule(torch.nn.Module):
    def save_hyperparameters(self, *a, **k):
        pass

    def log(self, *a, **k):
        pass

    @property
    def device(self):
        return torch.device("cpu")


def import_reference():
    k = _stub("kornia")
    k.utils = _stub("kornia.utils", tensor_to_image=lambda x: x.permute(0, 2, 3, 1).cpu().numpy())
    k.metrics = _stub("kornia.metrics")
    kg = _stub("kornia.geometry")
    kg.conversions = _stub("kornia.geometry.conversions", convert_points_to_homogeneous=lambda x: x)
    k.geometry = kg
    _stub("pytorch_lightning", LightningModule=_LightningModule)
    _stub("pytorch_lightning.utilities")
    _stub("pytorch_lightning.utilities.apply_func", move_data_to_device=lambda b, d: b)
    _stub("skimage")
    _stub("skimage.metrics", structural_similarity=None)
    _stub("imageio")
    torch.Tensor.cuda = lambda self, *a, **kw: self
    sys.path.insert(0, "/root/reference")
    import src.model as M
    M.VGGLoss = lambda: None
    return M


def build_net(M, n_kpt, weights):
    cfg = json.load(open("/root/reference/configs/zju.json"))
    cfg["models"]["KeypointNeRF"]["sp_args"]["n_kpt"] = n_kpt
    net = M.KeypointNeRF(cfg).eval()
    sd = {k: torch.from_numpy(np.asarray(v)) for k, v in weights.items()}
    res = net.load_state_dict(sd, strict=False)
    assert not res.unexpected_keys, res.unexpected_keys
    bad = [k for k in res.missing_keys if not k.startswith(("geo_encoder", "tex_encoder", "sp_encoder"))]
    assert not bad, bad
    return net


def ref_inputs(scene, target):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    cam = {"KRT": t(scene["KRT"]), "K": t(scene["K"]), "Rt": t(scene["extrin"]), "extrin": t(scene["extrin"]),
           "znear": scene["znear"], "zfar": scene["zfar"], "width": scene["width"], "height": scene["height"],
           "nml_scale": scene["nml_scale"]}
    cam_tar = {"K": t(target["K"]), "RT": t(target["RT"]), "KRT": t(target["KRT"]), "width": target["width"],
               "height": target["height"], "znear": target["znear"], "zfar": target["zfar"],
               "nml_scale": target["nml_scale"]}
    sp_data = {"extrin": t(scene["extrin"]), "kpt3d": t(scene["kpt3d"])}
    feat_geo = [t(scene["feat64"]), t(scene["feat8"])]
    return cam, cam_tar, sp_data, feat_geo, t(scene["feat_tex"]), t(scene["img"]), t(scene["fg"]), t(scene["bounds"])


def checksum(scene, weights):
    h = hashlib.sha256()
    for k in ("feat64", "feat8", "feat_tex", "img", "fg", "kpt3d", "KRT", "extrin"):
        h.update(np.ascontiguousarray(scene[k]).tobytes())
    for k in sorted(weights):
        h.update(np.ascontiguousarray(weights[k]).tobytes())
    return h.hexdigest()


def run_tile(M, net, scene, target, level, x_off, y_off, S_c, S_f, fine, capture=False, keep=128, keep_pts=None):
    cam, cam_tar, sp_data, feat_geo, feat_tex, img, fg, bounds = ref_inputs(scene, target)
    cap = {}
    hooks = []
    if capture:
        calls = {"q": 0}
        # (hook outputs of the first (coarse) query only)
        def h_sp(mod, args, kwargs, out):
            if "enc" not in cap:
                cap["enc"] = out.detach().clone()
        def h_geo(mod, args, out):
            if "x_view" not in cap:
                cap["geo_out"] = out[0].detach().clone()
                cap["x_view"] = out[2].detach().clone()
                cap["x_pool"] = out[3].detach().clone()
                cap["pw"] = args[3].detach().clone()
                cap["f64"] = args[1][0].detach().clone()
                cap["f8"] = args[1][1].detach().clone()
        def h_tex(mod, args, out):
            if "ibr_rgb" not in cap:
                cap["ibr_feat"] = args[0].detach().clone()
                cap["ibr_raydiff"] = args[1].detach().clone()
                cap["ibr_mask"] = args[2].detach().clone()
                cap["ibr_rgb"] = out.detach().clone()
        hooks.append(net.sp_encoder.register_forward_hook(h_sp, with_kwargs=True))
        hooks.append(net.mlp_geo.register_forward_hook(h_geo))
        hooks.append(net.mlp_tex.register_forward_hook(h_tex))
        orig_q = net.query
        def q_wrap(*a, **kw):
            out, valid = orig_q(*a, **kw)
            if "query_out" not in cap:
                cap["query_pts"] = a[0].detach().clone()
                cap["query_view"] = kw["view"].detach().clone()
                cap["query_out"] = out.detach().clone()
                cap["query_valid"] = valid.detach().clone()
            return out, valid
        net.query = q_wrap
        orig_imp = M.KeypointNeRF.importance_sample
        orig_r2o = M.KeypointNeRF.rgba2out
        def r2o(rgba, z):
            res = orig_r2o(rgba, z)
            key = "coarse" if "contrib_coarse" not in cap else "fine"
            cap["contrib_" + key] = res[3].detach().clone()
            cap["z_" + key] = z.detach().clone()
            cap["rgba_" + key] = rgba.detach().clone()
            return res
        net.rgba2out = r2o
    with torch.no_grad():
        out = M.KeypointNeRF.batch_render_pifu_nerf(
            net, img, cam, scene["n_views"], cam_tar, level, torch.Tensor([[x_off, y_off]]), None,
            feat_geo, feat_tex, dict(sp_data), torch.from_numpy(scene["kpt3d"][:, 0, :]),
            sample_per_ray_c=S_c, sample_per_ray_f=S_f, fine=fine, uniform=True,
            src_foreground_mask=fg, bounds=bounds)
    for h in hooks:
        h.remove()
    res = {k: v.numpy() for k, v in out.items() if torch.is_tensor(v)}
    if capture:
        del net.query
        del net.rgba2out
        N = cap["query_pts"].shape[1]
        # stored query points (keep_pts set): every valid one and a seeded sample of the invalid ones (whose outputs are zero)
        valid = cap["query_valid"][0, :, 0].numpy()
        pts = np.arange(N)
        if keep_pts is not None:
            assert valid.sum() <= keep_pts
            invalid = np.flatnonzero(~valid)
            extra = np.random.default_rng(0).choice(invalid, min(len(invalid), keep_pts - int(valid.sum())), replace=False)
            pts = np.sort(np.concatenate([np.flatnonzero(valid), extra]))
        sel = np.linspace(0, len(pts) - 1, num=min(keep, len(pts))).astype(np.int64)   # positions in pts
        at = pts[sel]                                                                  # indices into the N query points
        V = scene["n_views"]
        res["sel"] = sel
        res["query_pts"] = cap["query_pts"][0].numpy()[pts]
        res["query_view"] = cap["query_view"][0].numpy()[pts]
        res["query_out"] = cap["query_out"][0].numpy()[pts]
        res["query_valid"] = valid[pts]
        res["enc"] = cap["enc"].numpy()[:, at]                        # (V,sel,7K)
        res["pw"] = cap["pw"][0].numpy()[:, pts, 0]                    # (V,pts)
        res["f64"] = cap["f64"][0].numpy()[:, at]
        res["f8"] = cap["f8"][0].numpy()[:, at]
        res["x_view"] = cap["x_view"][0].numpy()[:, at]
        res["x_pool"] = cap["x_pool"][0].numpy()[at]
        res["geo_out"] = cap["geo_out"][0].numpy()[pts]
        res["ibr_feat"] = cap["ibr_feat"].reshape(N, V, -1).numpy()[at]       # (sel,V,35)
        res["ibr_raydiff"] = cap["ibr_raydiff"].reshape(N, V, -1).numpy()[at]
        res["ibr_rgb"] = cap["ibr_rgb"].reshape(N, 3).numpy()[pts]
        for k in ("contrib_coarse", "z_coarse", "rgba_coarse", "z_fine"):
            if k in cap:
                res[k] = cap[k][0].numpy()
    return res


# name -> dict(src, tgt, az, zoom, level, off, S_c, S_f, fine, n_kpt, seeds, fg_mode, fg_hole, capture, keep)
def _c(**kw):
    d = dict(src_size=512, tgt_size=512, azimuth=1.0, zoom=1.0, level=4, x_off=0, y_off=0, S_c=32, S_f=0, fine=False,
             n_kpt=18, scene_seed=2, w_seed=26, fg_mode="hull", fg_hole=False, capture="none", rays=None)
    d.update(kw)
    return d


PI4 = float(np.pi / 4)
CASES = {
    # tiny cases: small maps, every per-sample intermediate (capture="all")
    "tiny": _c(src_size=64, tgt_size=32, zoom=2.0, level=1, S_c=16, S_f=16, fine=True, capture="all"),
    "tiny_fg": _c(src_size=64, tgt_size=64, zoom=2.0, level=2, x_off=1, y_off=0, S_c=16, S_f=16, fine=True, fg_hole=True,
                  capture="all"),
    "tiny_k24": _c(src_size=64, tgt_size=32, zoom=2.0, azimuth=2.5, level=1, S_c=12, S_f=8, fine=True, n_kpt=24,
                   scene_seed=3, w_seed=5, capture="all"),
    # BASELINE config 1: one 64x64 strided pass, 32 samples/ray, 512^2 sources (hull scene and the bench scene)
    "cfg1_tile": _c(),
    "cfg1_ones": _c(fg_mode="ones", capture="some"),
    # BASELINE config 2 at config size: one strided pass of the 512x512x128 frame (hull scene and the bench scene)
    "cfg2_pass": _c(x_off=3, y_off=5, S_c=128, capture="some", rays=1024),
    "cfg2_pass_ones": _c(x_off=3, y_off=5, S_c=128, fg_mode="ones", capture="some", rays=1024),
    # BASELINE config 3 at config size: 64 coarse + 64 fine
    "cfg3_pass": _c(x_off=3, y_off=5, S_c=64, S_f=64, fine=True, capture="some", rays=1024),
    # BASELINE config 4: 1024^2 target, one level-5 pass (64x64 rays), 128 samples
    "cfg4_pass": _c(tgt_size=1024, level=5, x_off=7, y_off=9, S_c=128),
    # BASELINE config 5: second novel view of the sweep (azimuth 1.0 + pi/4)
    "cfg5_view": _c(azimuth=1.0 + PI4, x_off=2, y_off=6, S_c=128),
}


def dropin_sweep(M):
    """dropin_sweep.npz: the reference's KeypointNeRFLightningModule loads a seeded checkpoint with its strict
    load_state_dict and renders a two-camera sweep through render_novel_views (src/model.py:474-507).  Stores the module's
    state_dict names and shapes, the checksums of the checkpoint and of the sweep's inputs, and the 8-bit renderings."""
    from keypointnerf_b200.config import default_cfg
    from tests.util import seeded_checkpoint, state_dict_checksum, sweep_checksum, sweep_inputs
    n_kpt, S_c, S_f = 18, 12, 8
    cfg = default_cfg(n_kpt)
    cfg["models"]["KeypointNeRF"]["dr_kwargs"].update(sample_per_ray_c=S_c, sample_per_ray_f=S_f)
    cfg.update(expname="t", out_dir=HERE, training={})
    ref = M.KeypointNeRFLightningModule(cfg, None).eval()
    shapes = [(k, list(v.shape)) for k, v in ref.state_dict().items()]
    sd = seeded_checkpoint(shapes, syn.make_weights(n_kpt))
    ref.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    batch, cams = sweep_inputs(n_kpt)
    input_sha = sweep_checksum(batch, cams)
    batch = {k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in batch.items()}
    cams = [{k: torch.from_numpy(v) if isinstance(v, np.ndarray) else v for k, v in c.items()} for c in cams]
    with torch.no_grad():
        want = ref.render_novel_views(cams, batch, only_renderings=True)[0]
    meta = {"n_kpt": n_kpt, "S_c": S_c, "S_f": S_f, "state_dict": shapes}
    np.savez_compressed(os.path.join(HERE, "dropin_sweep.npz"), renderings=want,
                        ckpt_sha256=np.frombuffer(state_dict_checksum(sd).encode(), dtype=np.uint8),
                        input_sha256=np.frombuffer(input_sha.encode(), dtype=np.uint8),
                        meta=np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8))
    print("dropin_sweep", want.shape, want.dtype, "max", int(want.max()), flush=True)


def main():
    M = import_reference()
    torch.set_num_threads(8)
    names = sys.argv[1:] or list(CASES) + ["dropin_sweep"]
    nets = {}
    for name in names:
        if name == "dropin_sweep":
            dropin_sweep(M)
            continue
        c = CASES[name]
        scene = syn.make_scene(src_size=c["src_size"], n_views=3, n_kpt=c["n_kpt"], seed=c["scene_seed"],
                               fg_mode=c["fg_mode"], fg_hole=c["fg_hole"])
        weights = syn.make_weights(c["n_kpt"], seed=c["w_seed"])
        target = syn.make_target(size=c["tgt_size"], azimuth=c["azimuth"], zoom=c["zoom"])
        key = (c["n_kpt"], c["w_seed"])
        if key not in nets:
            nets[key] = build_net(M, c["n_kpt"], weights)
        res = run_tile(M, nets[key], scene, target, level=c["level"], x_off=c["x_off"], y_off=c["y_off"], S_c=c["S_c"],
                       S_f=c["S_f"], fine=c["fine"], capture=c["capture"] != "none",
                       keep_pts=3072 if c["capture"] == "all" else None)
        if c["capture"] == "some":   # outputs + what the compositing / resampling tests need, not the per-sample tensors
            keys = ["tex_fg", "depth", "alpha", "tex_fg_fine", "depth_fine", "alpha_fine", "sdf", "z_fine", "contrib_coarse",
                    "z_coarse"]
            valid_frac = float(res["query_valid"].mean())
            res = {k: res[k] for k in keys if k in res}
            if c["rays"]:
                rays = np.sort(np.random.default_rng(0).choice(res["tex_fg"][0, 0].size, c["rays"], replace=False))
                for k in ("z_fine", "contrib_coarse", "z_coarse"):
                    if k in res:
                        res[k] = res[k][rays]
                res["rays"] = rays
        else:
            valid_frac = float(res["query_valid"].mean()) if "query_valid" in res else float("nan")
        meta = {k: v for k, v in c.items() if k not in ("capture", "rays")}
        res["input_sha256"] = np.frombuffer(checksum(scene, weights).encode(), dtype=np.uint8)
        res["meta"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **res)
        print(name, res["tex_fg"].shape, "valid frac", valid_frac, "alpha mean", float(res["alpha"].mean()),
              "alpha max", float(res["alpha"].max()), flush=True)


if __name__ == "__main__":
    main()
