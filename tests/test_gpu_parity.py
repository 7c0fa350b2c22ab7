"""GPU parity tests: the CUDA path (through the reference-facing Python API -> ctypes -> C ABI)
against (a) golden vectors produced by the reference itself and (b) the CPU oracle on the same
seeded inputs.

Gate (BASELINE.json north_star): RGB within 1e-3 abs of the reference, PSNR delta < 0.01 dB.
  * engines 0 and 4 (tcgen05, fp16 operands with two-term weights, fp32 accumulate; 0 runs the view-sequential geometry kernel at
    18 keypoints, 4 the row-per-view one everywhere) are held to exactly that on RGB, on EVERY ray;
    accumulated alpha / per-sample compositing weights / depth are looser by the factors below (they are
    not averaged by colours in [0,1] and the density head has a x30 gain in the synthetic recipe);
  * engine 1 (fp32 CUDA cores) is held to fp32 round-off.
Scenes: the goldens use silhouette ("hull") foreground masks, for which the last sample of every ray is invalid, so that no
ray sits on the reference's final-sample step (dist[-1] = 1e10, src/model.py:1166) and no ray is excluded from any
comparison (SURVEY.md section 7.4).  The bench scene (all-ones masks, SURVEY.md section 8d) does have such rays (0.9 %): its
config-size passes compare everything in front of the last sample strictly on every ray and the images statistically.
The hierarchical resampling (searchsorted + sort) is discontinuous: the free-running fine pass is gated by PSNR and a high
quantile; pointwise only with the reference's own z_fine injected (SURVEY.md section 7, hard parts 3-4).
"""
import numpy as np
import pytest
import torch

from keypointnerf_b200 import synthetic as syn
from keypointnerf_b200.testing import build_model, scene_tensors
from oracle import kpnerf_oracle as O  # checker only
from tests.util import checksum, load_golden, psnr, scene_from_meta

pytestmark = pytest.mark.gpu

ENGINES = [0, 1, 4]   # default (view-sequential geometry kernel at 18 keypoints), fp32 CUDA cores, row-per-view geometry kernel
TOL = {
    0: dict(rgb=1e-3, alpha=3e-3, contrib=3e-3, depth=3e-2, sdf=3e-2, q99_fine=2.5e-3, psnr=70.0),
    1: dict(rgb=1e-4, alpha=1e-4, contrib=1e-4, depth=2e-3, sdf=2e-3, q99_fine=1e-3, psnr=80.0),
}
TOL[4] = TOL[0]
ALL = np.ones((), dtype=bool)   # every ray


def last_sample_rad(scene, weights, target, meta):
    step = 2 ** (meta["level"] - 1)
    pix = O.pixel_lattice(meta["tgt_size"], meta["tgt_size"], step, meta["x_off"], meta["y_off"])
    o, d, n_r, f_r = O.ray_setup(pix, target["K"], target["RT"], float(target["znear"]), float(target["zfar"]))
    near, far, hit = O.ray_bbox(scene["bounds"], o, d)
    n_r, f_r = O.clip_near_far(n_r, f_r, near, far, hit)
    out, valid = O.query(scene, O.fold_weights(weights), o + d * f_r, d)
    n = meta["tgt_size"] // step
    return out[:, 1].reshape(n, n).numpy(), valid.reshape(n, n).numpy()


def max_err(actual, desired, mask):
    err = np.abs(np.asarray(actual, np.float64) - np.asarray(desired, np.float64))
    m = np.broadcast_to(mask, err.shape)
    return float(err[m].max()) if m.any() else 0.0


def check(report, what, actual, desired, mask, tol):
    e = max_err(actual, desired, mask)
    report.append(f"{what}: {e:.2e} (tol {tol:.0e})")
    return e <= tol


def masked_psnr(a, b, mask):
    e = (np.asarray(a, np.float64) - np.asarray(b, np.float64))[np.broadcast_to(mask, np.shape(a))]
    mse = float(np.mean(e ** 2))
    return 120.0 if mse == 0 else 10.0 * np.log10(1.0 / mse)


def _render_tile(net, meta, scene, target, dev="cuda:0", engine=0, fine=None, debug=False, z_override=None):
    a = scene_tensors(scene, target, dev)
    net.engine = engine
    fine = meta["fine"] if fine is None else fine
    m = net._bind_scene(a["cam"], a["feat_geo"], a["feat_tex"], a["sp_data"], a["img"], a["fg"], a["bounds"])
    step = 2 ** (meta["level"] - 1)
    n = meta["tgt_size"] // step
    res = m.render(K=a["cam_tar"]["K"], RT=a["cam_tar"]["RT"], znear=target["znear"], zfar=target["zfar"],
                   x0=meta["x_off"], y0=meta["y_off"], step=step, nx=n, ny=n, S_c=meta["S_c"], S_f=meta["S_f"],
                   fine=fine, engine=engine, debug=debug, z_fine_override=z_override)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in res.items()}


@pytest.fixture(scope="module", params=["tiny", "tiny_fg", "tiny_k24"])
def case(request):
    g, meta, sha = load_golden(request.param)
    scene, weights, target = scene_from_meta(meta)
    assert checksum(scene, weights) == sha
    net = build_model(weights, meta["n_kpt"], "cuda:0")
    return g, meta, scene, weights, target, net


@pytest.mark.parametrize("engine", ENGINES)
def test_query_matches_reference(case, engine):
    """KeypointNeRF.query on the reference's own sample points."""
    g, meta, scene, weights, target, net = case
    a = scene_tensors(scene, target, "cuda:0")
    net.engine = engine
    pts = torch.from_numpy(g["query_pts"]).cuda()[None]
    view = torch.from_numpy(g["query_view"]).cuda()[None]
    with torch.no_grad():
        out, valid = net.query(pts, a["cam"], a["feat_geo"], a["feat_tex"], n_views=3, sp_data=a["sp_data"],
                               tx_data={"img": a["img"]}, view=view, src_foreground_mask=a["fg"], bounds=a["bounds"])
    torch.cuda.synchronize()
    out, valid = out[0].cpu().numpy(), valid[0, :, 0].cpu().numpy()
    assert np.array_equal(valid, g["query_valid"])
    v = g["query_valid"]
    t = TOL[engine]
    e_rgb = np.abs(out[v][:, 2:] - g["query_out"][v][:, 2:]).max()
    e_sdf = np.abs(out[v][:, 0] - g["query_out"][v][:, 0]).max()
    e_rad = np.abs(out[v][:, 1] - g["query_out"][v][:, 1]).max()   # density row carries the x30 gain
    print(f"query engine {engine}: rgb {e_rgb:.2e} sdf_raw {e_sdf:.2e} rad {e_rad:.2e}")
    assert e_rgb <= t["rgb"] and e_sdf <= 10 * t["rgb"] and e_rad <= (5e-2 if engine != 1 else 3e-3)
    assert np.all(out[~v] == 0.0)


@pytest.mark.parametrize("engine", ENGINES)
def test_tile_coarse_matches_reference(case, engine):
    g, meta, scene, weights, target, net = case
    r = _render_tile(net, meta, scene, target, engine=engine, debug=True)
    t = TOL[engine]
    ok = ALL
    rep = []
    good = check(rep, "tex_fg", r["tex_fg"], g["tex_fg"][0], ok, t["rgb"])
    good &= check(rep, "alpha", r["alpha"], g["alpha"][0], ok, t["alpha"])
    good &= check(rep, "contrib", r["contrib"], g["contrib_coarse"], ok, t["contrib"])
    good &= check(rep, "depth", r["depth"], g["depth"][0], ok, t["depth"])
    p = masked_psnr(r["tex_fg"], g["tex_fg"][0], ok)
    print(f"coarse engine {engine}: " + "; ".join(rep) + f"; psnr (all rays) {p:.1f} dB")
    assert good and p > t["psnr"], rep


@pytest.mark.parametrize("engine", ENGINES)
def test_tile_fine_with_reference_depths(case, engine):
    """Fine pass evaluated on the reference's own sorted z_fine: pointwise gate."""
    g, meta, scene, weights, target, net = case
    r = _render_tile(net, meta, scene, target, engine=engine, z_override=torch.from_numpy(g["z_fine"]))
    t = TOL[engine]
    ok = ALL
    rep = []
    good = check(rep, "tex_fg_fine", r["tex_fg_fine"], g["tex_fg_fine"][0], ok, t["rgb"])
    good &= check(rep, "alpha_fine", r["alpha_fine"], g["alpha_fine"][0], ok, t["alpha"])
    good &= check(rep, "sdf", r["sdf"], g["sdf"][0], ok, t["sdf"])
    good &= check(rep, "depth_fine", r["depth_fine"], g["depth_fine"][0], ok, t["depth"])
    print(f"fine@ref-z engine {engine}: " + "; ".join(rep))
    assert good, rep


@pytest.mark.parametrize("engine", ENGINES)
def test_tile_fine_free_running(case, engine):
    g, meta, scene, weights, target, net = case
    r = _render_tile(net, meta, scene, target, engine=engine, debug=True)
    t = TOL[engine]
    ok = ALL
    dz = np.abs(r["z_fine"] - g["z_fine"])
    e = np.abs(r["tex_fg_fine"] - g["tex_fg_fine"][0]).reshape(-1)
    p = masked_psnr(r["tex_fg_fine"], g["tex_fg_fine"][0], ok)
    print(f"fine free engine {engine}: z q99 {np.quantile(dz, 0.99):.2e} rgb q99 {np.quantile(e, 0.99):.2e} max {e.max():.2e} psnr {p:.1f}")
    assert np.quantile(dz, 0.99) < 1e-3
    assert p > 50.0
    assert np.quantile(e, 0.99) < t["q99_fine"]


def rays(g):
    """The rays of a pass whose per-sample arrays the golden stores (tests/golden/make_golden.py): all when it has no `rays`."""
    return g.get("rays", slice(None))


def _golden_case(name):
    g, meta, sha = load_golden(name)
    scene, weights, target = scene_from_meta(meta)
    assert checksum(scene, weights) == sha
    return g, meta, scene, weights, target, build_model(weights, meta["n_kpt"], "cuda:0")


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("name", ["cfg1_tile", "cfg2_pass", "cfg4_pass", "cfg5_view"])
def test_config_size_pass_matches_reference(name, engine):
    """One strided pass of BASELINE configs 1 (32 samples), 2 (512^2 x 128), 4 (1024^2 target, level 5) and 5 (second view of
    the sweep) at config size against the reference's own output of that pass; every ray is compared."""
    g, meta, scene, weights, target, net = _golden_case(name)
    r = _render_tile(net, meta, scene, target, engine=engine, debug="contrib_coarse" in g)
    t = TOL[engine]
    rep = []
    good = check(rep, "tex_fg", r["tex_fg"], g["tex_fg"][0], ALL, t["rgb"])
    good &= check(rep, "alpha", r["alpha"], g["alpha"][0], ALL, t["alpha"])
    good &= check(rep, "depth", r["depth"], g["depth"][0], ALL, t["depth"])
    if "contrib_coarse" in g:
        good &= check(rep, "contrib", r["contrib"][rays(g)], g["contrib_coarse"], ALL, t["contrib"])
    p = psnr(r["tex_fg"], g["tex_fg"][0])
    print(f"{name} engine {engine}: " + "; ".join(rep) + f"; psnr (all rays) {p:.1f} dB")
    assert good and p > t["psnr"], rep


@pytest.mark.parametrize("engine", ENGINES)
def test_cfg3_pass_matches_reference(engine):
    """BASELINE config 3 at config size (64 coarse + 64 fine samples) on one pass: coarse image and compositing weights,
    the fine image on the reference's own resampled depths (pointwise, on the rays whose depths the golden stores) and
    free-running (PSNR over every ray + resampled-depth quantile)."""
    g, meta, scene, weights, target, net = _golden_case("cfg3_pass")
    r = _render_tile(net, meta, scene, target, engine=engine, debug=True)
    t = TOL[engine]
    sub = rays(g)
    px = lambda a: a.reshape(*a.shape[:-2], -1)[..., sub]   # (.., h, w) image -> the stored rays
    rep = []
    good = check(rep, "tex_fg", r["tex_fg"], g["tex_fg"][0], ALL, t["rgb"])
    good &= check(rep, "contrib", r["contrib"][sub], g["contrib_coarse"], ALL, t["contrib"])
    p_free = psnr(r["tex_fg_fine"], g["tex_fg_fine"][0])
    dz = np.abs(r["z_fine"][sub] - g["z_fine"])
    z_ref = r["z_fine"].copy()
    z_ref[sub] = g["z_fine"]
    r2 = _render_tile(net, meta, scene, target, engine=engine, z_override=torch.from_numpy(z_ref))
    good &= check(rep, "tex_fg_fine@ref-z", px(r2["tex_fg_fine"]), px(g["tex_fg_fine"][0]), ALL, t["rgb"])
    good &= check(rep, "alpha_fine@ref-z", px(r2["alpha_fine"]), px(g["alpha_fine"][0]), ALL, t["alpha"])
    good &= check(rep, "sdf@ref-z", px(r2["sdf"]), px(g["sdf"][0]), ALL, t["sdf"])
    p_ref = psnr(px(r2["tex_fg_fine"]), px(g["tex_fg_fine"][0]))
    print(f"cfg3 engine {engine}: " + "; ".join(rep) + f"; fine psnr @ref-z {p_ref:.1f} dB, free-running {p_free:.1f} dB, "
          f"z_fine q99 {np.quantile(dz, 0.99):.2e}")
    assert good and p_ref > t["psnr"] and p_free > 55.0 and np.quantile(dz, 0.99) < 1e-3, rep


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("name", ["cfg1_ones", "cfg2_pass_ones"])
def test_bench_scene_pass_matches_reference(name, engine):
    """The bench scene (all-ones foreground masks, 46 % of the samples valid) at config size.  About 1 % of its rays end on a
    valid sample whose density is within rounding of 0, which the reference's dist[-1] = 1e10 turns into alpha 0 or 1; so the
    compositing weights of every sample IN FRONT of the last one are compared strictly on every ray, and the image by the
    fraction of rays beyond the gate and by the PSNR over all rays."""
    g, meta, scene, weights, target, net = _golden_case(name)
    r = _render_tile(net, meta, scene, target, engine=engine, debug=True)
    t = TOL[engine]
    rep = []
    good = check(rep, "contrib[:, :-1]", r["contrib"][rays(g), :-1], g["contrib_coarse"][:, :-1], ALL, t["contrib"])
    e = np.abs(r["tex_fg"] - g["tex_fg"][0]).max(0)
    frac = float((e > t["rgb"]).mean())
    p = psnr(r["tex_fg"], g["tex_fg"][0])
    print(f"{name} engine {engine}: " + "; ".join(rep) + f"; rays beyond the rgb gate {frac:.4%} (final-sample step); "
          f"rgb q99 {np.quantile(e, 0.99):.2e}; psnr (all rays) {p:.1f} dB")
    assert good and frac < 0.015 and np.quantile(e, 0.98) < t["rgb"] and p > 40.0, rep


def test_last_sample_step_semantics():
    """The reference's step at the final sample (dist[-1] = 1e10) is reproduced: on rays of the bench scene whose last-sample
    density is clearly positive the accumulated alpha is 1, for the reference and for both engines."""
    g, meta, scene, weights, target, net = _golden_case("cfg1_ones")
    rad, valid = last_sample_rad(scene, weights, target, meta)
    opaque = valid & (rad > 0.15)
    assert opaque.sum() > 100
    assert np.abs(g["alpha"][0][opaque] - 1.0).max() < 1e-5
    for engine in ENGINES:
        r = _render_tile(net, meta, scene, target, engine=engine)
        assert np.abs(r["alpha"][opaque] - 1.0).max() < 1e-5


def test_engines_agree_per_sample():
    """200k random points (many tiles per CTA slot): tensor-core engine vs fp32 engine, per sample."""
    scene = syn.make_scene(src_size=512, n_kpt=18)
    weights = syn.make_weights(18)
    target = syn.make_target(size=512)
    net = build_model(weights, 18, "cuda:0")
    a = scene_tensors(scene, target, "cuda:0")
    m = net._bind_scene(a["cam"], a["feat_geo"], a["feat_tex"], a["sp_data"], a["img"], a["fg"], a["bounds"])
    g = torch.Generator().manual_seed(0)
    n = 200000
    pts = ((torch.rand(n, 3, generator=g) - 0.5) * torch.tensor([0.8, 1.8, 0.6])).cuda()
    view = torch.nn.functional.normalize(torch.randn(n, 3, generator=g), dim=-1).cuda()
    o1, v1 = m.query(pts, view, engine=1)
    o0, v0 = m.query(pts, view, engine=0)
    o0b, _ = m.query(pts, view, engine=0)
    torch.cuda.synchronize()
    assert torch.equal(v0, v1) and torch.equal(o0, o0b)   # same validity; bit-deterministic run to run
    d = (o0 - o1).abs()[v1]
    print(f"engines per-sample: rgb {float(d[:, 2:].max()):.2e} rad {float(d[:, 1].max()):.2e} sdf {float(d[:, 0].max()):.2e}")
    assert float(d[:, 2:].max()) < 5e-4 and float(d[:, 1].max()) < 5e-2 and float(d[:, 0].max()) < 5e-3


def test_api_shapes_and_host_path_equal_device_path():
    """batch_render_pifu_nerf / render_pifu_nerf return what the reference returns (shapes, devices), and
    the KPN_MEM_HOST path (host buffers in, host buffers out) is bit-identical to the device path."""
    scene = syn.make_scene(src_size=64, n_kpt=18, fg_hole=True)
    weights = syn.make_weights(18)
    target = syn.make_target(size=32)
    net = build_model(weights, 18, "cuda:0")
    cfg = dict(sample_per_ray_c=8, sample_per_ray_f=8, fine=True, uniform=True)
    outs = []
    for dev in ("cuda:0", "cpu"):
        a = scene_tensors(scene, target, dev, pin=True)
        tar = torch.rand(1, 3, 32, 32, device=a["img"].device)
        with torch.no_grad():
            o = net.batch_render_pifu_nerf(net, a["img"], a["cam"], 3, a["cam_tar"], 2, torch.Tensor([[1, 1]]), tar,
                                           a["feat_geo"], a["feat_tex"], a["sp_data"], None,
                                           src_foreground_mask=a["fg"], bounds=a["bounds"], **cfg)
        torch.cuda.synchronize()
        assert o["tex_fg"].shape == (1, 3, 16, 16) and o["depth"].shape == (1, 16, 16)
        assert o["tex_fg_fine"].shape == (1, 3, 16, 16) and o["sdf"].shape == (1, 16, 16)
        assert torch.equal(o["tar_img"].cpu(), tar[:, :, 1::2, 1::2].cpu())
        outs.append({k: v.cpu() for k, v in o.items()})
    for k in ("tex_fg", "alpha", "tex_fg_fine", "sdf"):
        assert torch.equal(outs[0][k], outs[1][k]), k
    a = scene_tensors(scene, target, "cuda:0")
    with torch.no_grad():
        full = net.render_pifu_nerf(net, a["img"], a["cam"], a["cam_tar"], level=2, sp_data=a["sp_data"],
                                    feat_geo=a["feat_geo"], feat_tex=a["feat_tex"],
                                    src_foreground_mask=a["fg"], bounds=a["bounds"], mask_at_box=None, **cfg)
    assert full["tex_fg_fine"].shape == (3, 32, 32) and full["depth"].shape == (1, 32, 32)
    assert not full["tex_fg"].is_cuda
    # the frame equals the reference's assembly of strided passes (pixel_shuffle), reference src/model.py:916-938
    assert torch.equal(full["tex_fg"][:, 1::2, 1::2], outs[0]["tex_fg"][0])
    assert torch.equal(full["tex_fg_fine"][:, 1::2, 1::2], outs[0]["tex_fg_fine"][0])


def test_edge_cases():
    scene = syn.make_scene(src_size=64, n_kpt=18)
    weights = syn.make_weights(18)
    net = build_model(weights, 18, "cuda:0")
    for az, size in ((0.0, 16), (3.3, 24)):
        target = syn.make_target(size=size, azimuth=az)
        a = scene_tensors(scene, target, "cuda:0")
        m = net._bind_scene(a["cam"], a["feat_geo"], a["feat_tex"], a["sp_data"], a["img"], a["fg"], a["bounds"])
        r = m.render(K=a["cam_tar"]["K"], RT=a["cam_tar"]["RT"], znear=2.0, zfar=5.0, x0=0, y0=0, step=1, nx=size, ny=size,
                     S_c=3, S_f=1, fine=True)
        torch.cuda.synchronize()
        for k, v in r.items():
            assert torch.isfinite(v).all(), k
    # all-background foreground masks: no sample is valid -> exact zeros, and the stats say so
    target = syn.make_target(size=16, azimuth=1.0)
    a = scene_tensors(scene, target, "cuda:0")
    m = net._bind_scene(a["cam"], a["feat_geo"], a["feat_tex"], a["sp_data"], a["img"], torch.zeros_like(a["fg"]), a["bounds"])
    r = m.render(K=a["cam_tar"]["K"], RT=a["cam_tar"]["RT"], znear=2.0, zfar=5.0, x0=0, y0=0, step=1, nx=16, ny=16, S_c=8)
    torch.cuda.synchronize()
    assert float(r["tex_fg"].abs().max()) == 0.0 and float(r["alpha"].abs().max()) == 0.0
    st = m.stats()
    assert st["samples_valid"] == 0 and st["samples_total"] == 16 * 16 * 8
    # near > far (target znear beyond the bbox exit): depths run backwards exactly as in the reference; still finite
    m = net._bind_scene(a["cam"], a["feat_geo"], a["feat_tex"], a["sp_data"], a["img"], a["fg"], a["bounds"])
    r = m.render(K=a["cam_tar"]["K"], RT=a["cam_tar"]["RT"], znear=50.0, zfar=60.0, x0=0, y0=0, step=1, nx=16, ny=16, S_c=8)
    torch.cuda.synchronize()
    assert torch.isfinite(r["tex_fg"]).all()
    # a single sample per ray
    r = m.render(K=a["cam_tar"]["K"], RT=a["cam_tar"]["RT"], znear=2.0, zfar=5.0, x0=0, y0=0, step=1, nx=16, ny=16, S_c=1)
    torch.cuda.synchronize()
    assert torch.isfinite(r["tex_fg"]).all()
    # two source views: the tensor-core engine does not cover it and says so (no silent 25x cliff); the fp32 engine,
    # requested explicitly, renders it (still CUDA)
    from keypointnerf_b200._lib import KpnError
    s2 = syn.make_scene(src_size=64, n_views=2, n_kpt=18)
    a2 = scene_tensors(s2, target, "cuda:0")
    m2 = net._bind_scene(a2["cam"], a2["feat_geo"], a2["feat_tex"], a2["sp_data"], a2["img"], a2["fg"], a2["bounds"])
    kw2 = dict(K=a2["cam_tar"]["K"], RT=a2["cam_tar"]["RT"], znear=2.0, zfar=5.0, x0=0, y0=0, step=1, nx=16, ny=16, S_c=8)
    with pytest.raises(KpnError, match="engine = 1"):
        m2.render(**kw2)
    r2 = m2.render(engine=1, **kw2)
    torch.cuda.synchronize()
    ref2 = O.render_pixels(s2, O.fold_weights(weights), target, O.pixel_lattice(16, 16, 1, 0, 0), 8)
    assert np.abs(r2["tex_fg"].cpu().numpy().reshape(3, -1).T - ref2["tex_fg"].numpy()).max() < 1e-4
    # bad arguments fail loudly
    with pytest.raises(KpnError):
        m.render(K=a["cam_tar"]["K"], RT=a["cam_tar"]["RT"], znear=2.0, zfar=5.0, x0=0, y0=0, step=1, nx=16, ny=16, S_c=0)
    with pytest.raises(KpnError):
        m.render(K=a["cam_tar"]["K"], RT=a["cam_tar"]["RT"], znear=2.0, zfar=5.0, x0=0, y0=0, step=1, nx=0, ny=16, S_c=4)


def test_full_frame_properties_at_baseline_size():
    """BASELINE config 2 (512x512, 128 samples, 512^2 sources): size-independent properties.
    (1) any strided pass equals the corresponding pixels of the one-shot frame bit-for-bit (rays are
    independent; this is the reference's pixel_shuffle assembly); (2) chunking does not matter;
    (3) alpha in [0,1], colours inside the convex hull of the source colours; (4) the tensor-core frame is
    within the RGB gate of the fp32-engine frame on robust rays and > 50 dB PSNR overall."""
    scene = syn.make_scene(src_size=512, n_kpt=18)
    weights = syn.make_weights(18)
    target = syn.make_target(size=512)
    net = build_model(weights, 18, "cuda:0")
    a = scene_tensors(scene, target, "cuda:0")
    m = net._bind_scene(a["cam"], a["feat_geo"], a["feat_tex"], a["sp_data"], a["img"], a["fg"], a["bounds"])
    kw = dict(K=a["cam_tar"]["K"], RT=a["cam_tar"]["RT"], znear=2.0, zfar=5.0, S_c=128)
    frame = m.render(x0=0, y0=0, step=1, nx=512, ny=512, **kw)
    st = m.stats()
    assert st["samples_total"] == 512 * 512 * 128 and 0.2 < st["samples_valid"] / st["samples_total"] < 0.8
    tile = m.render(x0=3, y0=5, step=8, nx=64, ny=64, **kw)
    torch.cuda.synchronize()
    assert torch.equal(frame["tex_fg"][:, 5::8, 3::8], tile["tex_fg"])
    assert torch.equal(frame["alpha"][5::8, 3::8], tile["alpha"])
    # BASELINE config 4's partition: a row band rendered on its own (what one rank of a row-sharded frame does) is the
    # corresponding slice of the frame, and the sharded entry point with world = 1 is the frame itself
    from keypointnerf_b200 import distributed as D
    y0, ny = D.row_shard(512, 3, 8)
    band = m.render(x0=0, y0=y0, step=1, nx=512, ny=ny, **kw)
    assert torch.equal(frame["tex_fg"][:, y0:y0 + ny], band["tex_fg"]) and torch.equal(frame["alpha"][y0:y0 + ny], band["alpha"])
    whole = D.render_frame_row_sharded(m, width=512, height=512, rank=0, world=1, **kw)
    assert torch.equal(whole["tex_fg"], frame["tex_fg"])
    # BASELINE config 4's partition: the 8 lattice phases (2 x 4), each rendered on its own as one rank would, interleave to
    # the frame bit-for-bit
    phases = []
    for r in range(8):
        py, px, sy, sx = D.lattice_phase(r, 8)
        phases.append(m.render(x0=px, y0=py, step=sx, step_y=sy, nx=512 // sx, ny=512 // sy, **kw)["tex_fg"])
    assert torch.equal(D.interleave_lattice(torch.stack(phases), 8), frame["tex_fg"])
    m.check_health()
    al = frame["alpha"]
    assert float(al.min()) >= 0.0 and float(al.max()) <= 1.0 + 1e-5
    assert float(frame["tex_fg"].min()) >= -1e-6 and float(frame["tex_fg"].max()) <= 1.0 + 1e-5
    assert float(al.mean()) > 0.2  # the synthetic scene is not empty
    ref = m.render(x0=0, y0=0, step=1, nx=512, ny=512, engine=1, **kw)
    torch.cuda.synchronize()
    err = (frame["tex_fg"] - ref["tex_fg"]).abs().amax(0)
    # rays not hit by the final-sample step: both engines agree on alpha to 0.5 there or are both opaque
    flipped = (frame["alpha"] - ref["alpha"]).abs() > 0.05
    frac_flipped = float(flipped.float().mean())
    e_rob = float(err[~flipped].max())
    mse = float(((frame["tex_fg"] - ref["tex_fg"]) ** 2)[:, ~flipped].mean())
    p = 10 * np.log10(1.0 / mse)
    print(f"512^2x128 frame, tcgen05 vs fp32 engine: max rgb err {e_rob:.2e} on {1 - frac_flipped:.4f} of rays, psnr {p:.1f} dB; "
          f"final-sample step flips on {frac_flipped:.4%} of rays")
    assert e_rob < 1e-3 and p > 60.0 and frac_flipped < 0.01


def test_24_keypoint_frame_many_tiles_per_slot():
    """24 keypoints (configs/zju.json's n_kpt) take the tensor-core path WITHOUT the next-tile staging buffer (shared-memory
    budget); a 192x192x96 frame gives every tile slot several tiles, i.e. the persistent loop, the ghost tiles and the
    inline gathers of that path.  Checked against the fp32 engine like the baseline-size frame, and the device watchdog
    (kpn_debug_timing) must report that no barrier wait gave up."""
    import ctypes as C
    scene = syn.make_scene(src_size=256, n_kpt=24)
    weights = syn.make_weights(24)
    target = syn.make_target(size=192)
    net = build_model(weights, 24, "cuda:0")
    a = scene_tensors(scene, target, "cuda:0")
    m = net._bind_scene(a["cam"], a["feat_geo"], a["feat_tex"], a["sp_data"], a["img"], a["fg"], a["bounds"])
    kw = dict(K=a["cam_tar"]["K"], RT=a["cam_tar"]["RT"], znear=2.0, zfar=5.0, S_c=96, x0=0, y0=0, step=1, nx=192, ny=192)
    frame = m.render(engine=0, **kw)
    st = m.stats()
    assert st["samples_valid"] > 148 * 2 * 40 * 4, "scene too empty to give every slot several tiles"
    ref = m.render(engine=1, **kw)
    torch.cuda.synchronize()
    wd = (C.c_ulonglong * 16)()
    assert m.lib.kpn_debug_timing(m.ctx, 1, wd) == 0 and wd[0] == 0, f"device watchdog fired: {list(wd)[:5]}"
    flipped = (frame["alpha"] - ref["alpha"]).abs() > 0.05
    err = (frame["tex_fg"] - ref["tex_fg"]).abs().amax(0)
    e_rob = float(err[~flipped].max())
    print(f"24-keypoint 192^2x96 frame, tcgen05 vs fp32 engine: max rgb err {e_rob:.2e}, flipped {float(flipped.float().mean()):.4%}")
    assert e_rob < 1e-3 and float(flipped.float().mean()) < 0.01


@pytest.mark.parametrize("engine", ENGINES)
def test_early_ray_termination(engine):
    """ert_eps > 0 (BASELINE config 3): the front half of every ray is composited first and rays that are already opaque
    skip their back half.  Dense scene (density gain x600) so that many rays saturate early.  Properties: (1) every output
    stays within ert_eps (+ round-off) of the exact render, coarse and fine; (2) fewer samples are shaded; (3) ert_eps = 0
    is the exact path (bit-identical to not passing it)."""
    eps = 1e-3
    scene = syn.make_scene(src_size=256, n_kpt=18)
    weights = syn.make_weights(18, density_gain=600.0)
    target = syn.make_target(size=128)
    net = build_model(weights, 18, "cuda:0")
    a = scene_tensors(scene, target, "cuda:0")
    m = net._bind_scene(a["cam"], a["feat_geo"], a["feat_tex"], a["sp_data"], a["img"], a["fg"], a["bounds"])
    kw = dict(K=a["cam_tar"]["K"], RT=a["cam_tar"]["RT"], znear=2.0, zfar=5.0, x0=0, y0=0, step=1, nx=128, ny=128, S_c=48, S_f=32,
              fine=True, engine=engine)
    exact = m.render(**kw)
    n_exact = m.stats()["samples_valid"]
    zero = m.render(ert_eps=0.0, **kw)
    ert = m.render(ert_eps=eps, **kw)
    n_ert = m.stats()["samples_valid"]
    torch.cuda.synchronize()
    for k in ("tex_fg", "alpha", "tex_fg_fine", "alpha_fine"):
        assert torch.equal(exact[k], zero[k])
    saturated = float((exact["alpha"] > 1.0 - eps).float().mean())
    d_c = float((ert["tex_fg"] - exact["tex_fg"]).abs().max())
    d_a = float((ert["alpha"] - exact["alpha"]).abs().max())
    print(f"ERT engine {engine}: coarse rgb diff {d_c:.2e} alpha diff {d_a:.2e}; shaded samples {n_ert}/{n_exact} "
          f"({n_ert / n_exact:.3f}); opaque rays {saturated:.3f}")
    assert saturated > 0.05, "scene not dense enough to exercise early termination"
    assert d_c <= eps * 1.05 + 1e-5 and d_a <= eps * 1.05 + 1e-5
    assert n_ert < 0.97 * n_exact
    # the fine pass resamples from the (slightly different) coarse weights: robust comparison as for the free-running fine pass
    q = float(torch.quantile((ert["tex_fg_fine"] - exact["tex_fg_fine"]).abs().flatten().float().cpu(), 0.99))
    assert q <= 5e-3


def test_encoders_feed_the_kernels_in_place():
    """attach_im_feat path (SURVEY.md 8f.1): the channels-last encoders' outputs are gathered from in place (NHWC, no re-layout
    pass) and give bit-identical images to the same maps passed as ordinary NCHW tensors; the maps are cached per source-image
    set (the second camera of a sweep does not re-run the encoders), and match the fp32 NCHW encoders to conv round-off."""
    from keypointnerf_b200 import encoders as E
    torch.manual_seed(0)
    scene = syn.make_scene(src_size=256, n_kpt=18, fg_mode="hull")
    weights = syn.make_weights(18)
    net = build_model(weights, 18, "cuda:0")
    target = syn.make_target(size=64, zoom=2.0)
    a = scene_tensors(scene, target, "cuda:0")
    cfg = dict(sample_per_ray_c=24, sample_per_ray_f=0, fine=False, uniform=True, src_foreground_mask=a["fg"], bounds=a["bounds"],
               mask_at_box=None)
    with torch.no_grad():
        net.attach_im_feat(a["img"])
        fg0, ft0 = net.feat_geo, net.feat_tex
        assert fg0[0].shape == (3, 64, 32, 32) and fg0[1].shape == (3, 8, 128, 128) and ft0.shape == (3, 8, 64, 64)
        assert E.is_nhwc(fg0[0]) and E.is_nhwc(fg0[1]) and E.is_nhwc(ft0)
        out_nhwc = net.render_pifu_nerf(net, a["img"], a["cam"], a["cam_tar"], level=1, sp_data=a["sp_data"], **cfg)
        net.attach_im_feat(a["img"])
        assert net.feat_geo[0] is fg0[0] and net.feat_tex is ft0, "feature maps of the same source images must be cached"
        nchw = lambda t: t.contiguous(memory_format=torch.contiguous_format)
        out_nchw = net.render_pifu_nerf(net, a["img"], a["cam"], a["cam_tar"], level=1, sp_data=a["sp_data"],
                                        feat_geo=[nchw(fg0[0]), nchw(fg0[1])], feat_tex=nchw(ft0), **cfg)
    assert torch.equal(out_nhwc["tex_fg"], out_nchw["tex_fg"]) and torch.equal(out_nhwc["alpha"], out_nchw["alpha"])
    assert torch.equal(out_nhwc["tex_fg_fine"], out_nhwc["tex_fg"])   # fine=False: alias the reference's caller reads
    assert float(out_nhwc["alpha"].max()) > 0.05
    # the same encoders in plain NCHW fp32 without TF32: the channels-last run agrees to convolution round-off
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            x = torch.nn.functional.avg_pool2d(a["img"], 2, stride=2) * 2.0 - 1.0
            ref = net.geo_encoder(x.contiguous())
            got = net.geo_encoder(x.contiguous(memory_format=torch.channels_last))
        assert float((ref[0] - got[0]).abs().max()) < 1e-3 * float(ref[0].abs().max())
    finally:
        torch.backends.cudnn.allow_tf32 = prev


@pytest.mark.parametrize("engine", ENGINES)
def test_odd_sizes_against_oracle(engine):
    """Sizes that are multiples of nothing: 37 coarse + 53 fine samples, a 19 x 23 pixel lattice with step 3 / step_y 2 and offsets,
    against the CPU oracle (coarse pointwise; fine on the oracle's own resampled depths)."""
    scene = syn.make_scene(src_size=128, n_kpt=18, fg_mode="hull", fg_hole=True)
    weights = syn.make_weights(18)
    target = syn.make_target(size=96, azimuth=0.7, zoom=1.6)
    net = build_model(weights, 18, "cuda:0")
    a = scene_tensors(scene, target, "cuda:0")
    m = net._bind_scene(a["cam"], a["feat_geo"], a["feat_tex"], a["sp_data"], a["img"], a["fg"], a["bounds"])
    nx, ny, step, step_y, x0, y0, S_c, S_f = 19, 23, 3, 2, 5, 7, 37, 53
    ys, xs = torch.arange(ny) * step_y + y0, torch.arange(nx) * step + x0
    yy, xx = torch.meshgrid(ys, xs, indexing="ij")
    pix = torch.stack([xx, yy], -1).reshape(-1, 2).float()
    ref = O.render_pixels(scene, O.fold_weights(weights), target, pix, S_c, S_f, True)
    kw = dict(K=a["cam_tar"]["K"], RT=a["cam_tar"]["RT"], znear=2.0, zfar=5.0, x0=x0, y0=y0, step=step, step_y=step_y, nx=nx, ny=ny,
              S_c=S_c, S_f=S_f, fine=True, engine=engine)
    r = m.render(debug=True, **kw)
    r2 = m.render(z_fine_override=ref["z_fine"], **kw)
    torch.cuda.synchronize()
    t = TOL[engine]
    img = lambda v: v.reshape(ny, nx, 3).permute(2, 0, 1).numpy()
    rep = []
    good = check(rep, "tex_fg", r["tex_fg"].cpu().numpy(), img(ref["tex_fg"]), ALL, t["rgb"])
    good &= check(rep, "contrib", r["contrib"].cpu().numpy(), ref["contrib"].numpy(), ALL, t["contrib"])
    good &= check(rep, "tex_fg_fine@oracle-z", r2["tex_fg_fine"].cpu().numpy(), img(ref["tex_fg_fine"]), ALL, t["rgb"])
    good &= check(rep, "alpha_fine@oracle-z", r2["alpha_fine"].cpu().numpy(), ref["alpha_fine"].reshape(ny, nx).numpy(), ALL, t["alpha"])
    dz = (r["z_fine"].cpu() - ref["z_fine"]).abs()
    print(f"odd sizes engine {engine}: " + "; ".join(rep) + f"; z_fine q99 {float(torch.quantile(dz.flatten(), 0.99)):.2e}")
    assert good and float(ref["alpha"].max()) > 0.05 and float(torch.quantile(dz.flatten(), 0.99)) < 1e-3, rep


def test_config3_early_ray_termination_on_the_bench_scene():
    """BASELINE config 3 as benched (512 x 512, 64 + 64 samples, ert_eps = 1e-4, bench scene): every output stays within ert_eps
    (+ round-off) of the exact render of the same engine; the coarse image pointwise, the fine image (resampled from slightly
    different coarse weights) by quantile."""
    scene = syn.make_scene(src_size=512, n_kpt=18)
    weights = syn.make_weights(18)
    target = syn.make_target(size=512)
    net = build_model(weights, 18, "cuda:0")
    a = scene_tensors(scene, target, "cuda:0")
    m = net._bind_scene(a["cam"], a["feat_geo"], a["feat_tex"], a["sp_data"], a["img"], a["fg"], a["bounds"])
    kw = dict(K=a["cam_tar"]["K"], RT=a["cam_tar"]["RT"], znear=2.0, zfar=5.0, x0=0, y0=0, step=1, nx=512, ny=512, S_c=64, S_f=64, fine=True)
    exact = m.render(**kw)
    n_exact = m.stats()["samples_valid"]
    ert = m.render(ert_eps=1e-4, **kw)
    n_ert = m.stats()["samples_valid"]
    torch.cuda.synchronize()
    d_c = float((ert["tex_fg"] - exact["tex_fg"]).abs().max())
    d_a = float((ert["alpha"] - exact["alpha"]).abs().max())
    q = float(torch.quantile((ert["tex_fg_fine"] - exact["tex_fg_fine"]).abs().amax(0).flatten()[::4].float(), 0.999))
    print(f"config 3 ERT 1e-4: coarse rgb diff {d_c:.2e} alpha diff {d_a:.2e}; fine rgb q99.9 {q:.2e}; shaded samples {n_ert}/{n_exact} "
          f"({n_ert / n_exact:.4f})")
    assert d_c <= 1.05e-4 + 1e-5 and d_a <= 1.05e-4 + 1e-5 and q <= 2e-3 and n_ert <= n_exact


def test_front_kernel_validity_is_exact():
    """The front kernel skips, per ray, every sample outside a conservative depth interval (frustum + foreground bounding box of
    every view) and takes the exact test inside it: the number of valid samples must equal the oracle's count EXACTLY, for
    all-foreground, silhouette and holed masks (incl. masks touching the image border), zoomed / wide / off-axis targets and
    the fine pass' resampled depths."""
    weights = syn.make_weights(18)
    net = build_model(weights, 18, "cuda:0")
    cases = [dict(fg_mode="ones", fg_hole=False, size=48, az=1.0, zoom=1.0), dict(fg_mode="hull", fg_hole=False, size=64, az=2.0, zoom=1.5),
             dict(fg_mode="hull", fg_hole=True, size=40, az=0.3, zoom=3.0), dict(fg_mode="ones", fg_hole=True, size=56, az=4.4, zoom=0.6)]
    for c in cases:
        scene = syn.make_scene(src_size=128, n_kpt=18, fg_mode=c["fg_mode"], fg_hole=c["fg_hole"])
        target = syn.make_target(size=c["size"], azimuth=c["az"], zoom=c["zoom"])
        a = scene_tensors(scene, target, "cuda:0")
        m = net._bind_scene(a["cam"], a["feat_geo"], a["feat_tex"], a["sp_data"], a["img"], a["fg"], a["bounds"])
        n, S_c, S_f = c["size"], 24, 16
        r = m.render(K=a["cam_tar"]["K"], RT=a["cam_tar"]["RT"], znear=2.0, zfar=5.0, x0=0, y0=0, step=1, nx=n, ny=n, S_c=S_c, S_f=S_f,
                     fine=True, engine=1, debug=True)
        got = m.stats()["samples_valid"]
        pix = O.pixel_lattice(n, n, 1, 0, 0)
        o, d, n_r, f_r = O.ray_setup(pix, target["K"], target["RT"], 2.0, 5.0)
        near, far, hit = O.ray_bbox(scene["bounds"], o, d)
        n_r, f_r = O.clip_near_far(n_r, f_r, near, far, hit)
        want = 0
        for zz in (O.coarse_z(n_r, f_r, S_c), r["z_fine"].cpu()):   # the fine pass tests the GPU's own merged depths
            P = (o[:, None, :] + d[:, None, :] * zz[..., None]).reshape(-1, 3)
            xy, zc = O.project(scene, P)
            want += int(O.validity(scene, xy, zc).sum())
        print(f"front validity {c}: valid samples {got} (oracle {want})")
        assert got == want and want > 0, c


def test_camera_sweep_equals_per_camera_calls():
    """render_views (one source set, many cameras; async device-to-host copies on a side stream, one sync) returns exactly what
    per-camera render_pifu_nerf calls return, and binds / encodes the source set once."""
    scene = syn.make_scene(src_size=128, n_kpt=18, fg_mode="hull")
    weights = syn.make_weights(18)
    net = build_model(weights, 18, "cuda:0")
    a = scene_tensors(scene, syn.make_target(64, zoom=2.0), "cuda:0")
    cams = []
    for az in (0.3, 1.0, 2.2, 3.9, 5.1):
        t = syn.make_target(64, az, zoom=2.0)
        cams.append({"K": torch.from_numpy(t["K"]).cuda(), "RT": torch.from_numpy(t["RT"]).cuda(), "width": 64, "height": 64,
                     "znear": 2.0, "zfar": 5.0, "nml_scale": 100.0})
    cfg = dict(sample_per_ray_c=24, sample_per_ray_f=16, fine=True, uniform=True, src_foreground_mask=a["fg"], bounds=a["bounds"],
               mask_at_box=None)
    with torch.no_grad():
        sweep = net.render_views(net, a["img"], a["cam"], cams, sp_data=a["sp_data"], **cfg)
        launches = net.marcher().stats()["kernel_launches"]
        solo = [net.render_pifu_nerf(net, a["img"], a["cam"], c, level=1, sp_data=a["sp_data"], **cfg) for c in cams]
    assert len(sweep) == 5
    for f, g in zip(sweep, solo):
        for k in ("tex_fg", "alpha", "depth", "tex_fg_fine", "alpha_fine", "sdf"):
            assert not f[k].is_cuda and torch.equal(f[k], g[k]), k
    assert float(sweep[1]["alpha_fine"].max()) > 0.05
    part = net.render_views(net, a["img"], a["cam"], cams, sp_data=a["sp_data"], rank=1, world=2, **cfg)
    assert len(part) == 2 and torch.equal(part[0]["tex_fg_fine"], solo[1]["tex_fg_fine"]) and torch.equal(part[1]["tex_fg"], solo[3]["tex_fg"])
    assert launches > 0


def test_multi_gpu_equals_single_gpu():
    """BASELINE configs 4 and 5 on 2 GPUs (NCCL): the lattice-sharded frame and the gathered views are bit-identical to the
    single-GPU renders.  Needs >= 2 devices (skipped on the single-GPU test box; run with `gpurun --gpus 2`)."""
    import os
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29631", os.path.join(root, "tools", "multi_gpu_check.py")]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    print(p.stdout[-2000:], p.stderr[-2000:])
    assert p.returncode == 0 and "MULTI_GPU_OK" in p.stdout
