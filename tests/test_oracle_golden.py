"""Pin the CPU oracle (oracle/kpnerf_oracle.py) against outputs of the reference itself.

The golden files were produced by tests/golden/make_golden.py running the unmodified
reference on CPU in the build container.  Tolerances are fp32 round-off level: the
oracle is an independent restatement, not a bit-copy (different summation order).
"""
import numpy as np
import pytest
import torch

from oracle import kpnerf_oracle as O
from tests.util import checksum, load_golden, scene_from_meta, psnr


@pytest.fixture(scope="module", params=["tiny", "tiny_fg", "tiny_k24"])
def case(request):
    g, meta, sha = load_golden(request.param)
    scene, weights, target = scene_from_meta(meta)
    assert checksum(scene, weights) == sha, "seeded inputs drifted from the ones the golden run used"
    return g, meta, scene, weights, target


def test_query_stages_match_reference(case):
    g, meta, scene, weights, target = case
    fw = O.fold_weights(weights)
    pts = torch.from_numpy(g["query_pts"])
    view = torch.from_numpy(g["query_view"])
    out, valid, parts = O.query(scene, fw, pts, view, return_parts=True)
    sel = g["sel"]
    assert np.array_equal(valid.numpy(), g["query_valid"])
    np.testing.assert_allclose(parts["pw"][..., 0].numpy(), g["pw"], atol=2e-6)
    np.testing.assert_allclose(parts["f64"].numpy()[:, sel], g["f64"], atol=1e-5)
    np.testing.assert_allclose(parts["f8"].numpy()[:, sel], g["f8"], atol=1e-5)
    np.testing.assert_allclose(parts["enc"].numpy()[:, sel], g["enc"], atol=2e-5)
    np.testing.assert_allclose(parts["x_view"].numpy()[:, sel], g["x_view"], atol=1e-4)
    np.testing.assert_allclose(parts["x_pool"].numpy()[sel], g["x_pool"], atol=1e-4)
    np.testing.assert_allclose(out[:, :2].numpy(), g["geo_out"], atol=2e-3, rtol=1e-4)  # density row has gain 30
    f = torch.cat([parts["rgb_src"], parts["tex"], parts["lat"][None].expand(3, -1, -1)], -1)
    np.testing.assert_allclose(f.permute(1, 0, 2).numpy()[sel], g["ibr_feat"], atol=1e-4)
    np.testing.assert_allclose(parts["ray_diff"].permute(1, 0, 2).numpy()[sel], g["ibr_raydiff"], atol=2e-5)
    v = g["query_valid"]
    np.testing.assert_allclose(out[:, 2:].numpy()[v], g["ibr_rgb"][v], atol=2e-4)
    np.testing.assert_allclose(out.numpy()[v], g["query_out"][v], atol=2e-3, rtol=1e-4)


def test_tile_coarse_matches_reference(case):
    g, meta, scene, weights, target = case
    fw = O.fold_weights(weights)
    r = O.render_tile(scene, fw, target, meta["level"], meta["x_off"], meta["y_off"], meta["S_c"], meta["S_f"], True)
    np.testing.assert_allclose(r["z"].numpy(), g["z_coarse"], atol=2e-6)
    np.testing.assert_allclose(r["rgba"].numpy(), g["rgba_coarse"], atol=2e-3, rtol=1e-4)
    np.testing.assert_allclose(r["contrib"].numpy(), g["contrib_coarse"], atol=2e-5)
    np.testing.assert_allclose(r["tex_fg"].numpy(), g["tex_fg"][0], atol=2e-5)
    np.testing.assert_allclose(r["alpha"].numpy(), g["alpha"][0], atol=2e-5)
    np.testing.assert_allclose(r["depth"].numpy(), g["depth"][0], atol=2e-4)


def test_tile_fine_matches_reference(case):
    g, meta, scene, weights, target = case
    fw = O.fold_weights(weights)
    r = O.render_tile(scene, fw, target, meta["level"], meta["x_off"], meta["y_off"], meta["S_c"], meta["S_f"], True)
    # free-running hierarchical pass: inverse-CDF is discontinuous (SURVEY.md section 7 hard part 3), so
    # compare the resampled depths loosely and the image by PSNR ...
    dz = np.abs(r["z_fine"].numpy() - g["z_fine"])
    assert np.quantile(dz, 0.99) < 1e-4
    assert psnr(r["tex_fg_fine"].numpy(), g["tex_fg_fine"][0]) > 60.0
    # ... and tightly with the reference's own z_fine injected.
    r2 = O.render_tile(scene, fw, target, meta["level"], meta["x_off"], meta["y_off"], meta["S_c"], meta["S_f"], True,
                       z_fine_override=g["z_fine"])
    np.testing.assert_allclose(r2["tex_fg_fine"].numpy(), g["tex_fg_fine"][0], atol=3e-5)
    np.testing.assert_allclose(r2["alpha_fine"].numpy(), g["alpha_fine"][0], atol=3e-5)
    np.testing.assert_allclose(r2["sdf"].numpy(), g["sdf"][0], atol=2e-4)
    np.testing.assert_allclose(r2["depth_fine"].numpy(), g["depth_fine"][0], atol=3e-4)


def test_importance_sample_matches_reference(case):
    g, meta, scene, weights, target = case
    z = torch.from_numpy(g["z_coarse"])
    c = torch.from_numpy(g["contrib_coarse"])
    zf = O.importance_sample(c[:, 1:-1], 0.5 * (z[:, 1:] + z[:, :-1]), meta["S_f"])
    z_all = torch.sort(torch.cat([z, zf], -1), -1).values
    np.testing.assert_allclose(z_all.numpy(), g["z_fine"], atol=1e-6)


PASSES = ["cfg1_tile", "cfg1_ones", "cfg2_pass", "cfg2_pass_ones", "cfg3_pass", "cfg4_pass", "cfg5_view"]


@pytest.mark.parametrize("name", PASSES)
def test_config_size_pass_matches_reference(name):
    """One strided pass of every BASELINE config at config size (512^2 / 1024^2 targets, 32 / 128 / 64+64 samples,
    512^2 sources) against the reference's own output for that pass."""
    g, meta, sha = load_golden(name)
    scene, weights, target = scene_from_meta(meta)
    assert checksum(scene, weights) == sha
    fw = O.fold_weights(weights)
    sub = g.get("rays", slice(None))   # the rays of the pass whose per-sample arrays are stored (all when absent)
    r = O.render_tile(scene, fw, target, meta["level"], meta["x_off"], meta["y_off"], meta["S_c"], meta["S_f"], meta["fine"])
    if meta["fg_mode"] == "hull":
        # the property the hull scenes exist for: no ray's last sample is valid, so nothing sits on the final-sample step
        assert float(r["rgba"][:, -1, 0].abs().max()) == 0.0
        np.testing.assert_allclose(r["tex_fg"].numpy(), g["tex_fg"][0], atol=3e-5)
        np.testing.assert_allclose(r["alpha"].numpy(), g["alpha"][0], atol=3e-5)
    else:
        # bench scene: a few rays end on a valid sample whose density is within round-off of 0 (dist[-1] = 1e10 turns that into
        # alpha 0 or 1); everything in front of the last sample is compared strictly, the images statistically
        np.testing.assert_allclose(r["contrib"].numpy()[sub, :-1], g["contrib_coarse"][:, :-1], atol=3e-5)
        e = np.abs(r["tex_fg"].numpy() - g["tex_fg"][0]).max(0)
        assert (e > 3e-5).mean() < 0.002, f"{(e > 3e-5).mean():.4f} of the rays differ"
    np.testing.assert_allclose(r["depth"].numpy(), g["depth"][0], atol=3e-4)
    if meta["fine"]:
        # free-running fine pass over every ray by PSNR; pointwise on the reference's own z_fine for the stored rays
        assert psnr(r["tex_fg_fine"].numpy(), g["tex_fg_fine"][0]) > 60.0
        step = 2 ** (meta["level"] - 1)
        pix = O.pixel_lattice(meta["tgt_size"], meta["tgt_size"], step, meta["x_off"], meta["y_off"])[sub]
        f = O.render_pixels(scene, fw, target, pix, meta["S_c"], meta["S_f"], True, z_fine_override=g["z_fine"])
        np.testing.assert_allclose(f["tex_fg_fine"].numpy(), g["tex_fg_fine"][0].reshape(3, -1)[:, sub].T, atol=3e-5)
        np.testing.assert_allclose(f["alpha_fine"].numpy(), g["alpha_fine"][0].reshape(-1)[sub], atol=3e-5)
        zf = O.importance_sample(torch.from_numpy(g["contrib_coarse"])[:, 1:-1],
                                 0.5 * (torch.from_numpy(g["z_coarse"])[:, 1:] + torch.from_numpy(g["z_coarse"])[:, :-1]), meta["S_f"])
        z_all = torch.sort(torch.cat([torch.from_numpy(g["z_coarse"]), zf], -1), -1).values
        np.testing.assert_allclose(z_all.numpy(), g["z_fine"], atol=1e-6)
