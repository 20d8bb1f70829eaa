"""Sequences shared by tools/make_wgsl_golden.py (which runs them through the reference's own WGSL, translated and executed on the CPU —
oracle/wgsl/) and by the tests that hold the oracle and the CUDA path against what that produced (tests/golden/wgsl_*.npz).

Each case: a scene, a benchmark configuration's settings, a frame size, a number of frames from zeroed temporal state, a camera
translation per frame and optionally animated instances.  Per frame and per plane the fixture stores a SHA-256 of the plane's bytes in
the reference's texture / buffer format (the compared implementations must be bit-identical), plus the last frame's tone-mapped image
in full for diagnostics.

Render widths are multiples of 8 here, as they are in every BASELINE configuration (1920, 3840, 7680 and their halves).  For other widths
the reference's shaders have a second data race that only a GPU can "resolve": the dispatch covers ceil(w / 8) * 8 columns, the extra
invocations read a zero G-buffer (robust access), take the background branch and STORE a reservoir at index x + w * y — which, for
x >= w, is a pixel at the start of the next row (light.wgsl:1057-1066 with the linear index of :1063; found by executing the shader
text at 60 x 34).  The oracle and the CUDA path run no out-of-range invocations; DESIGN.md 2 lists this with the other deviations."""
import hashlib

import numpy as np

from bevy_hikari_b200 import layout as L
from bevy_hikari_b200 import plugin as _P

CASES = {
    # name: (scene, config, (W, H), frames, camera step per frame, animation or None, settings overrides)
    "cornell_cfg1": ("cornell", "cornell_256", (64, 64), 8, (0.0, 0.0, 0.0), None, {}),                 # BASELINE configs[0] settings
    "cornell_cfg2_moving": ("cornell", "cornell_1080p", (80, 48), 9, (0.03, 0.01, -0.02), None, {}),     # configs[1] settings, moving camera
    "cornell_animated": ("cornell", "cornell_1080p", (72, 48), 7, (0.0, 0.0, 0.0), "cornell", {}),       # instances move every frame
    "city_cfg4_moving": ("city", "city_4k", (80, 45), 7, (0.05, 0.0, -0.04), None, {}),                  # textures, sun, 13 textures
    "city_cfg5": ("city", "city_8k", (64, 36), 6, (0.0, 0.0, 0.0), None, {}),                            # 4 bounces, both spatial reuses
    "town_cfg3": ("town", "scene_1080p", (64, 40), 5, (0.04, 0.0, -0.03), None, {}),                        # configs[2]: examples/scene.rs, 120 k triangles, 3 bounces
    "simple_two_lights": ("simple", "cornell_1080p", (72, 48), 7, (0.02, 0.0, 0.0), None, {}),           # two emissives: light BVH + alias
    "samplers": ("samplers", "cornell_1080p", (64, 40), 6, (0.0, 0.0, 0.0), None, {}),                   # wrap modes, nearest / bilinear, textured light
    "no_denoise_one_bounce": ("simple", "cornell_256", (56, 40), 6, (0.0, 0.02, 0.0), None, {}),
    # HikariSettings away from the BASELINE configurations (the corners tests/test_gpu_variants.py walks on the device)
    "settings_no_bounces": ("simple", "cornell_1080p", (56, 40), 5, (0.02, 0.0, 0.0), None, {"indirect_bounces": 0}),     # ambient-only indirect pass, two denoised signals
    "settings_no_temporal_reuse": ("cornell", "cornell_1080p", (56, 40), 5, (0.02, 0.01, 0.0), None, {"temporal_reuse": 0, "denoise": 0}),
    "settings_lifetime_and_validation": ("cornell", "cornell_1080p", (56, 40), 7, (0.0, 0.0, 0.0), "cornell",
                                         {"max_reservoir_lifetime": 1.0, "direct_validate_interval": 1, "emissive_validate_interval": 2, "denoise": 0}),
    "settings_clamps": ("city", "city_8k", (64, 36), 6, (0.03, 0.0, -0.02), None,
                        {"max_temporal_reuse_count": 2, "max_spatial_reuse_count": 3, "max_indirect_luminance": 0.5}),
    "settings_sun_disc_and_clear_color": ("city", "city_4k", (64, 36), 5, (0.0, 0.0, 0.0), None,
                                          {"solar_angle": 0.5, "clear_color": (0.1, 0.2, 0.3, 1.0), "indirect_bounces": 1}),
    # scaled rendering (Upscale ratio > 1: light / denoise planes at ceil(size / ratio), jittered_deferred_uv / _coords look-ups)
    "cornell_ratio2": ("cornell", "cornell_1080p", (96, 64), 7, (0.02, 0.0, -0.01), None, {"upscale_ratio": 2.0}),
    "city_ratio1p5": ("city", "city_4k", (96, 54), 6, (0.0, 0.0, 0.0), None, {"upscale_ratio": 1.5}),
    # the temporal upscalers after tone mapping (smaa.wgsl: smaa_tu4x + smaa_tu4x_extrapolate, taa.wgsl: taa_jasmine), jittered prepass
    "cornell_default_upscalers": ("cornell", "cornell_1080p", (96, 64), 9, (0.03, 0.01, -0.02), None,        # HikariSettings::default():
                                  {"taa": _P.TAA_JASMINE, "upscale_kind": _P.UPSCALE_SMAA_TU4X, "upscale_ratio": 2.0}),   # SMAA_TU_2_0 + Jasmine
    "cornell_smaa_ratio1_taa": ("cornell", "cornell_1080p", (72, 48), 8, (0.02, 0.0, -0.01), "cornell",
                                {"taa": _P.TAA_JASMINE, "upscale_kind": _P.UPSCALE_SMAA_TU4X, "upscale_ratio": 1.0}),
    "city_smaa_only_ratio1p5": ("city", "city_4k", (96, 54), 7, (0.04, 0.0, -0.03), None,
                                {"taa": _P.TAA_NONE, "upscale_kind": _P.UPSCALE_SMAA_TU4X, "upscale_ratio": 1.5}),
    "simple_taa_only": ("simple", "cornell_1080p", (80, 48), 8, (0.02, 0.01, 0.0), None,
                        {"taa": _P.TAA_JASMINE, "upscale_kind": _P.UPSCALE_FSR1, "upscale_ratio": 1.0}),      # TAA on the tone-mapped image
    # default settings on an odd window: 127 x 63 renders 64 x 32, and upscale_output = ceil(size * (0.5 * 2)) is 127 x 63, not 128 x 64 —
    # stores of the last column / row fall outside the texture, every uv of smaa.wgsl / taa.wgsl is computed from the odd extent
    "cornell_default_upscalers_odd_window": ("cornell", "cornell_1080p", (127, 63), 7, (0.03, 0.01, -0.02), None,
                                             {"taa": _P.TAA_JASMINE, "upscale_kind": _P.UPSCALE_SMAA_TU4X, "upscale_ratio": 2.0}),
    # Upscale::Fsr1: EASU + RCAS (src/shaders/fsr/source.zip: the GLSL of the reference's SPIR-V blobs) after tone mapping / TAA
    "cornell_fsr_ratio1p5": ("cornell", "cornell_1080p", (96, 64), 6, (0.03, 0.01, -0.02), None,
                             {"taa": _P.TAA_NONE, "upscale_kind": _P.UPSCALE_FSR1, "upscale_ratio": 1.5, "upscale_sharpness": 0.0}),
    "city_taa_fsr_ratio2": ("city", "city_4k", (128, 72), 6, (0.04, 0.0, -0.03), None,
                            {"taa": _P.TAA_JASMINE, "upscale_kind": _P.UPSCALE_FSR1, "upscale_ratio": 2.0, "upscale_sharpness": 0.5}),
}
# cases whose frames run with HikariInputs::temporal_upscalers (the passes of post_process.rs:1236-1277 after tone mapping)
UPSCALER_CASES = {"cornell_default_upscalers", "cornell_smaa_ratio1_taa", "city_smaa_only_ratio1p5", "simple_taa_only",
                  "cornell_default_upscalers_odd_window", "cornell_fsr_ratio1p5", "city_taa_fsr_ratio2"}

# cases added after the round's last full device run (call 17): the device suite runs them LAST, in a file of their own
# (tests/test_gpu_zzz_wgsl_late_cases.py; green on a B200 in call 18, the round's last 70 GPU-seconds)
LATE_CASES = {"town_cfg3", "settings_no_bounces", "settings_no_temporal_reuse", "settings_lifetime_and_validation", "settings_clamps",
              "settings_sun_disc_and_clear_color"}

PLANES = ([("albedo", L.OUT_ALBEDO)] + [(f"render{i}", L.OUT_RENDER_DIRECT + i) for i in range(3)] +
          [(f"variance{i}", L.OUT_VARIANCE_DIRECT + i) for i in range(3)] + [(f"reservoir{i}", L.OUT_RESERVOIR_0 + i) for i in range(10)] +
          [("tone_mapped", L.OUT_TONE_MAPPED)])
DENOISED = [(f"denoised{i}", L.OUT_DENOISED_DIRECT + i) for i in range(3)]
GBUFFER = [L.OUT_GBUFFER_POSITION, L.OUT_GBUFFER_NORMAL, L.OUT_GBUFFER_DEPTH_GRADIENT, L.OUT_GBUFFER_INSTANCE_MATERIAL, L.OUT_GBUFFER_VELOCITY_UV]


def digest(array):
    return hashlib.sha256(np.ascontiguousarray(array).tobytes()).hexdigest()


def load_digests(path):
    """{name: hex digest} of a digest fixture (tools/make_wgsl_golden.py: `names` + raw SHA-256 `digests`)"""
    z = np.load(path)
    return {str(n): bytes(d).hex() for n, d in zip(z["names"], z["digests"])}


def save_digests(path, digests, **extra):
    names = sorted(digests)
    np.savez_compressed(path, names=np.array(names), digests=np.array([np.frombuffer(bytes.fromhex(digests[n]), np.uint8) for n in names]),
                        **extra)


# ------------------------------------------------------------------------------------------------ pass by pass
# Every pass of the reference's shader text run FROM THE ORACLE'S STATE (before each pass the reference's planes are overwritten with the
# oracle's): scene, config, size; PER_PASS_FRAMES frames, the camera translating by PER_PASS_STEP per frame.  The digest of every plane
# after every pass is stored in tests/golden/wgsl_per_pass_<scene>.npz (a per-pass diagnosis of any drift).
PER_PASS_CASES = [("cornell", "cornell_1080p", (48, 40)), ("city", "city_4k", (64, 36)), ("simple", "city_8k", (48, 32))]
PER_PASS_FRAMES, PER_PASS_STEP = 6, (0.02, 0.0, -0.01)
PASS_PLANES = PLANES[:-1]          # albedo, render and variance of the three signals, the ten reservoir buffers


def light_passes(inp):
    """the passes of LightNode::run in order; the spatial reuses when the frame enables them"""
    from oracle import oracle as O
    return ([O.PASS_ALBEDO, O.PASS_DIRECT, O.PASS_EMISSIVE] + ([O.PASS_EMISSIVE_SPATIAL] if inp.frame.emissive_spatial_reuse else []) +
            [O.PASS_INDIRECT] + ([O.PASS_INDIRECT_SPATIAL] if inp.frame.indirect_spatial_reuse else []))


def make_bench(case):
    from tests.conftest import Bench
    scene, config, (w, h), frames, step, animation, overrides = CASES[case]
    return Bench(scene, w, h, config=config, **overrides)


def frame_inputs(bench, case, frame):
    step = CASES[case][4]
    inp = bench.moving_inputs(frame, step) if any(step) else bench.inputs(frame)
    if case in UPSCALER_CASES:
        inp.temporal_upscalers = 1
    return inp


def upscalers_of(case, bench):
    """(smaa, taa) as PostProcessNode::run decides them (post_process.rs:1236,1260)"""
    if case not in UPSCALER_CASES:
        return False, False
    return bench.settings.upscale_kind == _P.UPSCALE_SMAA_TU4X, bench.settings.taa == _P.TAA_JASMINE


def fsr_of(case, bench):
    """Upscale::Fsr1 passes run (post_process.rs:1279)"""
    return case in UPSCALER_CASES and bench.settings.upscale_kind == _P.UPSCALE_FSR1


def animate(bench, case, frame):
    """moves the case's animated instances to their pose of `frame` (host mirror: transforms, previous transforms, prepare_instances);
    returns True when the scene changed"""
    if CASES[case][5] is None:
        return False
    from tests.conftest import cornell_animation
    if not hasattr(bench, "_wgsl_anim"):
        bench._wgsl_anim = cornell_animation(bench)
    bench._wgsl_anim.step(frame)
    return True


def planes_of(case, bench):
    denoise = bool(bench.settings.denoise)
    signals = 3 if bench.settings.indirect_bounces else 2
    smaa, taa = upscalers_of(case, bench)
    return (PLANES + (DENOISED[:signals] if denoise else []) + ([("upscaled", L.OUT_UPSCALED)] if smaa else []) +
            ([("taa", L.OUT_TAA)] if taa else []) +
            ([("fsr_easu", L.OUT_UPSCALED), ("fsr_rcas", L.OUT_FSR_SHARPENED)] if fsr_of(case, bench) else []))


# ------------------------------------------------------------------------------------------------ the raster prepass (G-buffer)
# prepass.wgsl executed through the software rasteriser of oracle/wgsl/raster_prepass.py: scene, config, size, frame compared, camera
# step, animation, TAA jitter.  The ray-cast G-buffer of oracle and CUDA path is held against it within the bounds of
# tests/test_wgsl_prepass.py (coverage / ids exact up to edge pixels, values within the sub-pixel snapping of a rasteriser).
PREPASS_CASES = {
    # name: (scene, config, (W, H), frame, camera step, animation, taa jitter, fixture committed)
    "cornell_moving": ("cornell", "cornell_1080p", (96, 64), 3, (0.03, 0.01, -0.02), None, False, True),
    "cornell_animated_jittered": ("cornell", "cornell_1080p", (96, 64), 4, (0.02, 0.0, 0.0), "cornell", True, True),
    "city_moving": ("city", "city_4k", (128, 72), 2, (0.05, 0.0, -0.04), None, False, True),
    "simple_ground_plane": ("simple", "cornell_1080p", (96, 64), 2, (0.02, 0.0, 0.0), None, False, False),      # a quad through the near plane
    "samplers": ("samplers", "cornell_1080p", (96, 64), 1, (0.0, 0.0, 0.0), None, False, False),
    "town": ("town", "scene_1080p", (128, 72), 1, (0.0, 0.0, 0.0), None, False, False),                       # examples/scene.rs, 120 k triangles
    "city_larger": ("city", "city_4k", (256, 144), 2, (0.05, 0.0, -0.04), None, False, False),
}
# the cases without a committed full-frame fixture: their fixtures hold this window (x0, x1, y0, y1) of the compared frame, which keeps
# each file small.  The oracle against the rasterised G-buffer, full frame -> window (tools/make_wgsl_golden.py --prepass prints both):
#   simple_ground_plane  covered pixels 4550 -> 1442; beyond a bound: position 76 -> 15, depth 17 -> 4, gradient 1 -> 1
#   samplers             the whole frame (3630 covered, none beyond any bound)
#   town                 covered 8903 -> 2304; id mismatches 6 -> 2, normal 14 -> 5, gradient 27 -> 8; position 136, depth 54, uv 3 -> 0
#   city_larger          covered 26177 -> 2223; id mismatches 1 -> 1, gradient 40 -> 8; normal 15, position 3, depth 2, velocity 2, uv 2 -> 0
PREPASS_WINDOWS = {"simple_ground_plane": (24, 72, 16, 48), "samplers": (0, 96, 0, 64), "town": (32, 96, 18, 54),
                   "city_larger": (96, 160, 54, 90)}
PREPASS_PLANES = [("position", L.OUT_GBUFFER_POSITION), ("normal", L.OUT_GBUFFER_NORMAL), ("depth_gradient", L.OUT_GBUFFER_DEPTH_GRADIENT),
                  ("instance_material", L.OUT_GBUFFER_INSTANCE_MATERIAL), ("velocity_uv", L.OUT_GBUFFER_VELOCITY_UV)]


def prepass_window(case, plane, width, height):
    """`plane` (a full frame of `case`) cut to the case's PREPASS_WINDOWS entry"""
    x0, x1, y0, y1 = PREPASS_WINDOWS[case]
    return np.ascontiguousarray(np.ascontiguousarray(plane).reshape(height, width, -1)[y0:y1, x0:x1])


def prepass_sequence(case):
    """yields (bench, frame inputs, previous models or None) for frames 1 .. the compared frame of a PREPASS case; the caller renders
    the G-buffer of every frame (the prepass keeps the previous frame's planes) and compares the last"""
    from tests.conftest import Bench, cornell_animation
    scene, config, (w, h), frame, step, animation, taa, _ = PREPASS_CASES[case]
    kw = dict(taa=_P.TAA_JASMINE, upscale_kind=_P.UPSCALE_FSR1, upscale_ratio=1.0) if taa else {}
    bench = Bench(scene, w, h, config=config, **kw)
    anim = cornell_animation(bench) if animation else None
    for f in range(1, frame + 1):
        previous_models = None
        if anim:
            previous_models = bench.world.buffers()["instances"]["model"].reshape(-1, 16).copy()
            anim.step(f)
        inp = bench.moving_inputs(f, step) if any(step) else bench.inputs(f)
        if taa:
            inp.temporal_upscalers = 1
        yield bench, inp, previous_models, anim is not None
