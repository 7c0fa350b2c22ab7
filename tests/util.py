"""Shared helpers for the tests: golden loading and scene reconstruction from fixture metadata."""
import hashlib
import json
import os
import zlib

import numpy as np

from keypointnerf_b200 import synthetic as syn

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    g = {k: z[k] for k in z.files}
    meta = json.loads(bytes(g.pop("meta")).decode())
    sha = bytes(g.pop("input_sha256")).decode()
    return g, meta, sha


def scene_from_meta(meta):
    scene = syn.make_scene(src_size=meta["src_size"], n_views=3, n_kpt=meta["n_kpt"], seed=meta["scene_seed"],
                           fg_hole=meta["fg_hole"], fg_mode=meta.get("fg_mode", "ones"))
    weights = syn.make_weights(meta["n_kpt"], seed=meta["w_seed"])
    target = syn.make_target(size=meta["tgt_size"], azimuth=meta["azimuth"], zoom=meta.get("zoom", 1.0))
    return scene, weights, target


def checksum(scene, weights):
    h = hashlib.sha256()
    for k in ("feat64", "feat8", "feat_tex", "img", "fg", "kpt3d", "KRT", "extrin"):
        h.update(np.ascontiguousarray(scene[k]).tobytes())
    for k in sorted(weights):
        h.update(np.ascontiguousarray(weights[k]).tobytes())
    return h.hexdigest()


def psnr(a, b):
    mse = float(np.mean((np.asarray(a, np.float64) - np.asarray(b, np.float64)) ** 2))
    return 99.0 if mse == 0 else 10.0 * np.log10(1.0 / mse)


def seeded_checkpoint(shapes, weights, seed=0):
    """A full state_dict from seeds, for the (name, shape) list of a checkpoint: the hot-path networks from ``weights``
    (``synthetic.make_weights``, names without the ``model.`` prefix), every other tensor drawn per name (independent of the
    order of the list) like torch's default layer init: matrices and kernels uniform in +-1/sqrt(fan_in), norm scales
    1 +- 0.1, biases +-0.1, other vectors (``sp_encoder.center``) zero."""
    sd = {}
    for name, shape in shapes:
        short = name.split(".", 1)[1] if name.startswith("model.") else name
        if short in weights:
            v = np.asarray(weights[short], np.float32)
            assert v.shape == tuple(shape), name
        else:
            rng = np.random.default_rng([seed, zlib.crc32(name.encode())])
            if len(shape) >= 2:
                b = 1.0 / np.sqrt(np.prod(shape[1:]))
                v = rng.uniform(-b, b, shape)
            elif name.endswith(".weight"):
                v = 1.0 + rng.uniform(-0.1, 0.1, shape)
            elif name.endswith(".bias"):
                v = rng.uniform(-0.1, 0.1, shape)
            else:
                v = np.zeros(shape)
        sd[name] = np.ascontiguousarray(v, np.float32)
    return sd


def state_dict_checksum(sd):
    h = hashlib.sha256()
    for k in sorted(sd):
        h.update(k.encode())
        h.update(np.ascontiguousarray(sd[k]).tobytes())
    return h.hexdigest()


def sweep_checksum(batch, cams):
    h = hashlib.sha256()
    for k in sorted(batch):
        h.update(np.ascontiguousarray(batch[k]).tobytes())
    for c in cams:
        for k in sorted(c):
            h.update(np.ascontiguousarray(c[k]).tobytes())
    return h.hexdigest()


def sweep_inputs(n_kpt=18):
    """The camera sweep of the drop-in test: one ZJUDataset-style batch (index 0 = target view, 1.. = source views,
    reference ``src/zju_dataset.py:217-343``) and two 64x64 cameras as ``render_novel_views`` takes them."""
    scene = syn.make_scene(src_size=128, n_kpt=n_kpt, fg_mode="hull")
    tgt = syn.make_target(size=64, azimuth=1.0, zoom=2.0)
    s = scene["src_size"]
    Rt = np.concatenate([tgt["RT"][:, :3, :4], scene["extrin"][:, :3, :4]], 0)[None]
    Ks = np.concatenate([tgt["K"][:, :3, :3], scene["K"][:, :3, :3]], 0)[None]
    imgs = np.concatenate([np.zeros((1, 3, s, s), np.float32), scene["img"]], 0)[None]
    msk = np.concatenate([np.ones((1, 1, s, s), np.float32), scene["fg"].astype(np.float32)], 0)[None]
    batch = {"images": imgs, "images_masks": msk, "Rt": Rt, "K": Ks, "kpt3d": scene["kpt3d"], "bounds": scene["bounds"],
             "mask_at_box": np.ones((1, s * s), np.float32)}
    cams = []
    for az in (1.0, 2.5):
        t = syn.make_target(64, az, zoom=2.0)
        cams.append({"intrinsics": t["K"], "w2cs": t["RT"][0], "im_h": 64, "im_w": 64, "znear": 2.0, "zfar": 5.0})
    return batch, cams
