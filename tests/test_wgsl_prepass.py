"""The ray-cast G-buffer held against the reference's RASTER prepass (SURVEY 8(a) rows P0 / T8; DESIGN.md 2, deviation 1).

The reference rasterises its G-buffer (src/prepass.rs + src/shaders/prepass.wgsl); oracle and CUDA path cast one primary ray per pixel.
oracle/wgsl/raster_prepass.py executes prepass.wgsl's `vertex` and `fragment` as written (translated like the compute shaders) behind a
software rasteriser that does what a GPU's fixed-function stages do (near-plane clipping, 1/256-pixel vertex snapping, top-left fill
rule, perspective-correct interpolation, GreaterEqual depth test, fine quad derivatives, the five target formats).  What that produces
for three sequences is committed (tests/golden/wgsl_prepass_*.npz, tools/make_wgsl_golden.py --prepass); here

  * the oracle's G-buffer agrees with it: the SAME pixels are covered and show the same (instance, material) except for a handful where
    an edge passes within the rasteriser's snapping of a pixel centre; on those pixels world position agrees to a few percent of the
    pixel's own footprint, NDC depth to 1e-3 relative, the packed normal to 1 snorm8 step, the depth gradient to 2 %, screen-space
    velocity to 5e-6 + 3e-4 of its magnitude and texture coordinates to 2e-3 — on all but the <= 2 % of pixels where the two methods hit different triangles of
    one instance (an edge inside a mesh, coplanar faces) or where a ground plane recedes to the horizon;
  * in the build container the fixtures are regenerated from the shader text and must be identical;
  * four more scenes (a quad through the near plane, the sampler scene, examples/scene.rs with 120 k triangles, the city at twice the
    size) against a window of what the rasteriser made of them (tests/golden/wgsl_prepass_<case>.npz, same tool);
  * `-m gpu`: the CUDA path's G-buffer against the same fixtures with the same bounds (tests/test_gpu_wgsl_golden.py)."""
import os
import sys

import numpy as np
import pytest

from bevy_hikari_b200 import layout as L
from tests import wgsl_cases as WC
from tests.conftest import ROOT

GOLDEN = os.path.join(ROOT, "tests", "golden")
IN_CONTAINER = os.path.isdir("/root/reference/src/shaders")

# bounds: (tolerance, largest allowed fraction of the commonly covered pixels beyond it)
BOUNDS = {"coverage_mismatch": 0.002, "id_mismatch": 0.005, "outliers": 0.02,
          "position_per_footprint": 0.05, "depth_relative": 1e-3, "normal_snorm8": 1, "gradient_relative": 0.02, "gradient_floor": 1e-3,
          "velocity": 5e-6, "velocity_relative": 3e-4, "uv": 2e-3}


def fixture(case):
    z = np.load(os.path.join(GOLDEN, f"wgsl_prepass_{case}.npz"))
    return {k: z[k] for k, _ in WC.PREPASS_PLANES}


def compare(raster, gbuffer, width, height, what):
    """`raster`: the five planes as the rasterised prepass.wgsl wrote them; `gbuffer`: {plane id: array} of the implementation under test"""
    H, W = height, width
    pos_r = raster["position"].reshape(H, W, 4)
    pos_o = np.ascontiguousarray(gbuffer[L.OUT_GBUFFER_POSITION]).reshape(H, W, 4)
    im_r = raster["instance_material"].reshape(H, W, 2)
    im_o = np.ascontiguousarray(gbuffer[L.OUT_GBUFFER_INSTANCE_MATERIAL]).reshape(H, W, 2)
    cov_r, cov_o = pos_r[..., 3] > 0, pos_o[..., 3] > 0
    n_cov = max(int(cov_r.sum()), 1)
    assert (cov_r != cov_o).sum() <= BOUNDS["coverage_mismatch"] * n_cov, (what, "coverage", int((cov_r != cov_o).sum()), n_cov)
    both = cov_r & cov_o
    same = both & (im_r[..., 0] == im_o[..., 0]) & (im_r[..., 1] == im_o[..., 1])
    assert both.sum() - same.sum() <= max(BOUNDS["id_mismatch"] * n_cov, 8), (what, "instance / material", int(both.sum() - same.sum()), n_cov)
    n = int(same.sum())
    assert n > 0.5 * n_cov
    # a pixel's footprint in world units: distance to the nearest neighbour pixel of the same instance
    fp = np.full((H, W), np.inf, np.float32)
    for dy, dx in ((0, 1), (1, 0), (0, -1), (-1, 0)):
        sh, shi, shc = (np.roll(a, (-dy, -dx), axis=(0, 1)) for a in (pos_r, im_r[..., 0], cov_r))
        d = np.linalg.norm(sh[..., :3] - pos_r[..., :3], axis=2)
        fp = np.where(shc & (shi == im_r[..., 0]), np.minimum(fp, d), fp)
    have_fp = same & np.isfinite(fp) & (fp > 0)
    nrm_r = raster["normal"].view(np.int8).reshape(H, W, 4).astype(np.int32)
    nrm_o = np.ascontiguousarray(gbuffer[L.OUT_GBUFFER_NORMAL]).view(np.int8).reshape(H, W, 4).astype(np.int32)
    dg_r = raster["depth_gradient"].reshape(H, W, 2)
    dg_o = np.ascontiguousarray(gbuffer[L.OUT_GBUFFER_DEPTH_GRADIENT]).reshape(H, W, 2)
    vu_r = raster["velocity_uv"].reshape(H, W, 4)
    vu_o = np.ascontiguousarray(gbuffer[L.OUT_GBUFFER_VELOCITY_UV]).reshape(H, W, 4)
    grad_scale = float(np.abs(dg_r[same]).max()) if n else 0.0
    beyond = {
        "position": have_fp & (np.linalg.norm(pos_r[..., :3] - pos_o[..., :3], axis=2) > BOUNDS["position_per_footprint"] * np.where(have_fp, fp, 1.0)),
        "depth": same & (np.abs(pos_r[..., 3] - pos_o[..., 3]) > BOUNDS["depth_relative"] * np.abs(pos_r[..., 3])),
        "normal": same & (np.abs(nrm_r - nrm_o).max(axis=2) > BOUNDS["normal_snorm8"]),
        "gradient": same & (np.abs(dg_r - dg_o).max(axis=2) > BOUNDS["gradient_relative"] * np.abs(dg_r).max(axis=2) + BOUNDS["gradient_floor"] * grad_scale),
        # the two projections of a pixel's velocity share the world position, so its snapping error enters only in proportion to the motion
        "velocity": same & (np.abs(vu_r - vu_o)[..., :2].max(axis=2) > BOUNDS["velocity"] + BOUNDS["velocity_relative"] * np.abs(vu_r[..., :2]).max(axis=2)),
        "uv": same & (np.abs(vu_r - vu_o)[..., 2:].max(axis=2) > BOUNDS["uv"]),
    }
    report = {k: int(v.sum()) for k, v in beyond.items()}
    for k, v in report.items():
        assert v <= BOUNDS["outliers"] * n, (what, k, f"{v} of {n} pixels beyond the bound", report)
    return dict(report, covered=n_cov, compared=n, coverage_mismatch=int((cov_r != cov_o).sum()), id_mismatch=int(both.sum() - same.sum()))


def render_gbuffer(case, make_renderer, update_scene):
    r = None
    for bench, inp, previous_models, animated in WC.prepass_sequence(case):
        if r is None:
            r = make_renderer(bench)
        if animated:
            update_scene(r, bench)
        r.prepass(inp)
    return bench, {which: np.ascontiguousarray(r.readback(which)) for _, which in WC.PREPASS_PLANES}


FIXTURE_CASES = sorted(c for c, v in WC.PREPASS_CASES.items() if v[7])


@pytest.mark.parametrize("case", FIXTURE_CASES)
def test_oracle_gbuffer_agrees_with_the_rasterised_prepass(case):
    bench, g = render_gbuffer(case, lambda b: b.oracle(), lambda r, b: r.update_instances_desc(b.world.scene_desc()))
    rep = compare(fixture(case), g, bench.width, bench.height, case)
    assert rep["coverage_mismatch"] == 0           # on these sequences not one pixel is covered by one method and not the other


@pytest.mark.skipif(not IN_CONTAINER, reason="the reference's shader sources exist only in the build container")
@pytest.mark.parametrize("case", sorted(WC.PREPASS_CASES))
def test_committed_prepass_fixtures_are_what_the_shader_text_rasterises_today(case):
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    sys.path.insert(0, os.path.join(ROOT, "oracle", "wgsl"))
    import make_wgsl_golden
    r = make_wgsl_golden.prepass_fixture(case)
    z = np.load(os.path.join(GOLDEN, f"wgsl_prepass_{case}.npz"))
    for k, _ in WC.PREPASS_PLANES:
        assert np.array_equal(np.ascontiguousarray(r[k]).view(np.uint8), np.ascontiguousarray(z[k]).view(np.uint8)), (case, k)
    if "skipped_triangles" in z:
        assert int(r["skipped_triangles"]) == int(z["skipped_triangles"])


@pytest.mark.parametrize("case", sorted(WC.PREPASS_WINDOWS))
def test_more_scenes_against_a_window_of_the_rasterised_prepass(case):
    """what the rasteriser made of these scenes is stored for a window of the frame (WC.PREPASS_WINDOWS); the oracle's G-buffer is
    compared on the same window"""
    z = np.load(os.path.join(GOLDEN, f"wgsl_prepass_{case}.npz"))
    assert int(z["skipped_triangles"]) == 0 or case == "town"      # degenerate clipped slivers only
    bench, g = render_gbuffer(case, lambda b: b.oracle(), lambda r, b: r.update_instances_desc(b.world.scene_desc()))
    x0, x1, y0, y1 = WC.PREPASS_WINDOWS[case]
    compare({k: z[k] for k, _ in WC.PREPASS_PLANES}, {which: WC.prepass_window(case, a, bench.width, bench.height) for which, a in g.items()},
            x1 - x0, y1 - y0, case)
