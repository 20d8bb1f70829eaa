#!/usr/bin/env python
"""Randomised campaign for the WGSL pin (build container only): random scene, frame size, HikariSettings, upscalers, camera motion and
instance animation; every frame is computed twice — by the reference's own shader text (oracle/wgsl/: light / denoise / tone mapping /
SMAA / TAA WGSL and the FSR 1.0 GLSL, translated and executed with the wiring of light.rs / post_process.rs) and by the CPU oracle — and
every buffer and texture of every frame must be identical, bit for bit.  The committed fixtures (tests/golden/wgsl_*.npz) are 23 chosen
sequences; this walks the space between them.  The reference's planes of FIXED_SEEDS are committed too (tests/golden/wgsl_pin_seeds.npz),
so tests/test_wgsl_reference.py runs the oracle side of those (oracle_digests) anywhere.

usage: tools/fuzz_wgsl_pin.py FIRST_SEED COUNT

Render widths are kept multiples of 8 (tests/wgsl_cases.py explains the reference's race for other widths, DESIGN.md 2 deviation 5)."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle", "wgsl"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bevy_hikari_b200 import layout as L  # noqa: E402
from bevy_hikari_b200 import plugin  # noqa: E402
from tests import wgsl_cases as WC  # noqa: E402
from tests.conftest import Bench, cornell_animation  # noqa: E402

SCENES = [("cornell", "cornell_1080p"), ("cornell", "cornell_256"), ("simple", "cornell_1080p"), ("samplers", "cornell_1080p"),
          ("city", "city_4k"), ("city", "city_8k"), ("minimal", "cornell_1080p")]


def random_case(rng):
    scene, config = SCENES[rng.integers(len(SCENES))]
    upscalers = rng.random() < 0.4
    kind = plugin.UPSCALE_SMAA_TU4X if rng.random() < 0.6 else plugin.UPSCALE_FSR1
    ratio = float(rng.choice([1.0, 1.0, 2.0, 1.6])) if (upscalers or rng.random() < 0.3) else 1.0
    rw = int(rng.choice([8, 16, 24, 32, 40, 48]))                               # render width: a multiple of 8
    w = {1.0: rw, 2.0: 2 * rw - int(rng.integers(2)), 1.6: int(np.floor(rw * 1.6))}[ratio]
    h = int(rng.integers(9, 56))
    while int(np.ceil(np.float32(1.0) / np.float32(ratio) * np.float32(w))) != rw:
        w -= 1
    settings = dict(indirect_bounces=int(rng.integers(0, 5)), temporal_reuse=int(rng.random() < 0.85),
                    emissive_spatial_reuse=int(rng.random() < 0.5), indirect_spatial_reuse=int(rng.random() < 0.6), denoise=int(rng.random() < 0.6),
                    direct_validate_interval=int(rng.integers(1, 5)), emissive_validate_interval=int(rng.integers(1, 6)),
                    max_temporal_reuse_count=int(rng.choice([2, 20, 50, 200])), max_spatial_reuse_count=int(rng.choice([3, 10, 800])),
                    max_reservoir_lifetime=float(rng.choice([0.5, 1.0, 8.0, 32.0])), solar_angle=float(rng.choice([0.0, 0.046, 0.5])),
                    max_indirect_luminance=float(rng.choice([0.5, 10.0, 1e6])),
                    taa=plugin.TAA_JASMINE if (upscalers and rng.random() < 0.6) else plugin.TAA_NONE,
                    upscale_kind=kind, upscale_ratio=ratio, upscale_sharpness=float(rng.choice([0.0, 0.2, 1.0])))
    step = tuple(float(x) for x in (rng.uniform(-0.04, 0.04, 3) if rng.random() < 0.6 else np.zeros(3)))
    animated = scene == "cornell" and rng.random() < 0.3
    frames = int(rng.integers(3, 7))
    return scene, config, (w, h), settings, upscalers, step, animated, frames


# the seeds whose reference planes are committed (tests/golden/wgsl_pin_seeds.npz, tools/make_wgsl_golden.py --pin-seeds)
FIXED_SEEDS = list(range(5000, 5010))


class Case:
    """the random case of `seed`: bench, planes compared, frame inputs"""

    def __init__(self, seed):
        rng = np.random.default_rng(seed)
        scene, config, (w, h), settings, self.upscalers, self.step, animated, self.frames = random_case(rng)
        self.bench = bench = Bench(scene, w, h, config=config, **settings)
        self.anim = cornell_animation(bench) if animated else None
        self.smaa = self.upscalers and bench.settings.upscale_kind == plugin.UPSCALE_SMAA_TU4X
        self.taa = self.upscalers and bench.settings.taa == plugin.TAA_JASMINE
        self.fsr = self.upscalers and bench.settings.upscale_kind == plugin.UPSCALE_FSR1
        planes = list(WC.PLANES) + (WC.DENOISED[:3 if bench.settings.indirect_bounces else 2] if bench.settings.denoise else [])
        planes += ([("upscaled", L.OUT_UPSCALED)] if self.smaa else []) + ([("taa", L.OUT_TAA)] if self.taa else [])
        planes += [("fsr_easu", L.OUT_UPSCALED), ("fsr_rcas", L.OUT_FSR_SHARPENED)] if self.fsr else []
        self.planes = planes
        self.what = (f"{scene}/{config} {w}x{h} {self.frames} frames upscalers={self.upscalers} step={tuple(round(s, 3) for s in self.step)} "
                     f"animated={animated} {settings}")

    def inputs(self, f):
        inp = self.bench.moving_inputs(f, self.step) if any(self.step) else self.bench.inputs(f)
        if self.upscalers:
            inp.temporal_upscalers = 1
        return inp


def reference_digests(seed):
    """{f<frame>_<plane>: digest} of every plane of every frame as the reference's shader text computes them (G-buffer: the oracle's)"""
    import make_wgsl_golden as G
    import run_reference as R
    c = Case(seed)
    bench = c.bench
    w, h = bench.width, bench.height
    textures = [(np.ascontiguousarray(t["rgba"]), t["address_mode_u"], t["address_mode_v"], t["filter_linear"], t["srgb"]) for t in bench.scene.textures]
    ref = R.WgslReference(bench.world.buffers(), textures, plugin.load_noise(), w, h, bench.settings.upscale_ratio)
    orc_g = bench.oracle()
    out = {}
    for f in range(1, c.frames + 1):
        if c.anim:
            c.anim.step(f)
            orc_g.update_instances_desc(bench.world.scene_desc())
            ref.scene = {k: np.ascontiguousarray(v) for k, v in bench.world.buffers().items()}
        inp = c.inputs(f)
        orc_g.prepass(inp)
        ref.set_gbuffer(*[np.ascontiguousarray(orc_g.readback(k)) for k in WC.GBUFFER])
        ref.light_node(inp)
        ref.post_process_node(inp, bool(bench.settings.denoise))
        if c.smaa or c.taa:
            ref.upscale_node(inp, c.smaa, c.taa)
        if c.fsr:
            ref.fsr_node(inp, c.taa, bench.settings.upscale_sharpness)
        got = G.reference_planes(ref, bench)
        for name, _ in c.planes:
            out[f"f{f}_{name}"] = WC.digest(got[name])
    return out, c.what


def oracle_digests(seed):
    """the same planes as the CPU oracle renders them"""
    c = Case(seed)
    orc = c.bench.oracle()
    out = {}
    for f in range(1, c.frames + 1):
        if c.anim:
            c.anim.step(f)
            orc.update_instances_desc(c.bench.world.scene_desc())
        orc.render_frame(c.inputs(f))
        for name, which in c.planes:
            out[f"f{f}_{name}"] = WC.digest(orc.readback(which))
    return out, c.what


def run(seed):
    ref, what = reference_digests(seed)
    orc, _ = oracle_digests(seed)
    bad = [k for k in ref if orc[k] != ref[k]]
    return bad, what


def main():
    import run_reference as R
    if not R.available():
        raise SystemExit("needs /root/reference and g++ (build container only)")
    first, count = int(sys.argv[1]), int(sys.argv[2])
    failures = 0
    for seed in range(first, first + count):
        bad, what = run(seed)
        if bad:
            failures += 1
            print(f"seed {seed}: {what}\n   -> {len(bad)} planes differ, first {bad[:6]}")
    print(f"{count} cases, {failures} failures")
    return 1 if failures else 0


if __name__ == "__main__":
    sys.exit(main())
