#!/usr/bin/env python
"""Golden vectors from the reference's OWN shaders.  Runs every sequence of tests/wgsl_cases.py through the reference's WGSL
(/root/reference/src/shaders/{light,denoise,tone_mapping,smaa,taa}.wgsl translated to C++ by oracle/wgsl/wgsl2cpp.py and executed on the CPU by
oracle/wgsl/run_reference.py, wired as src/light.rs and src/post_process.rs wire the passes) and writes per-frame, per-plane SHA-256
digests of every buffer and texture the passes produce to tests/golden/wgsl_<case>.npz.

Only in the build container (needs /root/reference + g++).  The G-buffer of each frame is the oracle's (the reference rasterises it:
a render pipeline, not part of the translated compute path); everything downstream — albedo, both direct_lit pipelines, both
spatial_reuse pipelines, indirect_lit_ambient (single / multiple bounces), demodulation, the four denoise levels with and without
firefly filtering, tone mapping, SMAA TU4x (+ extrapolation) and TAA, over free-running sequences with validation frames, camera motion and moving instances — is computed
by the reference's shader text from its own state of the previous frames.

  --prepass [CASE ...]   tests/golden/wgsl_prepass_<case>.npz: the G-buffer prepass.wgsl rasterises (a window of it for WC.PREPASS_WINDOWS)
  --per-pass             tests/golden/wgsl_per_pass_<scene>.npz: every pass run from the oracle's state (WC.PER_PASS_CASES)
  --pin-seeds            tests/golden/wgsl_pin_seeds.npz: the reference's planes of tools/fuzz_wgsl_pin.py's FIXED_SEEDS
  --layouts              tests/golden/wgsl_struct_layouts.json: the struct layouts the translator derives from light.wgsl"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle", "wgsl"))

from bevy_hikari_b200 import layout as L  # noqa: E402
from bevy_hikari_b200 import plugin  # noqa: E402
from tests import wgsl_cases as WC  # noqa: E402
import run_reference as R  # noqa: E402


def reference_planes(ref, bench):
    out = {"albedo": ref.albedo, "tone_mapped": ref.tone_mapped}
    for i in range(3):
        out[f"render{i}"], out[f"variance{i}"], out[f"denoised{i}"] = ref.render[i], ref.variance[i], ref.denoise_render[i]
    for i in range(10):
        out[f"reservoir{i}"] = ref.reservoir[i][:ref.rw * ref.rh]      # the records the passes index (render size)
    if ref.upscale_output is not None:
        out["upscaled"] = ref.upscale_output
    if ref.taa_output is not None:
        out["taa"] = ref.taa_output[ref.head]
    if ref.fsr_output is not None:
        out["fsr_easu"], out["fsr_rcas"] = ref.fsr_output
    return out


def run_case(case):
    bench = WC.make_bench(case)
    w, h = bench.width, bench.height
    textures = [(np.ascontiguousarray(t["rgba"]), t["address_mode_u"], t["address_mode_v"], t["filter_linear"], t["srgb"]) for t in bench.scene.textures]
    ref = R.WgslReference(bench.world.buffers(), textures, plugin.load_noise(), w, h, bench.settings.upscale_ratio)
    orc = bench.oracle()
    frames = WC.CASES[case][3]
    digests = {}
    for f in range(1, frames + 1):
        if WC.animate(bench, case, f):
            orc.update_instances_desc(bench.world.scene_desc())
            ref.scene = {k: np.ascontiguousarray(v) for k, v in bench.world.buffers().items()}
        inp = WC.frame_inputs(bench, case, f)
        orc.prepass(inp)                                    # the raster prepass: G-buffer only
        ref.set_gbuffer(*[np.ascontiguousarray(orc.readback(k)) for k in WC.GBUFFER])
        ref.light_node(inp)
        ref.post_process_node(inp, bool(bench.settings.denoise))
        smaa, taa = WC.upscalers_of(case, bench)
        if smaa or taa:
            ref.upscale_node(inp, smaa, taa)
        if WC.fsr_of(case, bench):
            ref.fsr_node(inp, taa, bench.settings.upscale_sharpness)
        planes = reference_planes(ref, bench)
        for name, _ in WC.planes_of(case, bench):
            digests[f"f{f}_{name}"] = WC.digest(planes[name])
    return digests, ref.tone_mapped.copy()


def run_per_pass(scene, config, size):
    """one sequence of WC.PER_PASS_CASES: before each pass the reference's planes are overwritten with the oracle's, the pass runs on
    both.  Returns the digests of the reference's planes after every pass and the names of those the oracle does not reproduce."""
    from oracle import oracle as O
    from tests.conftest import Bench
    W, H = size
    b = Bench(scene, W, H, config=config)
    orc = b.oracle()
    tex = [(np.ascontiguousarray(t["rgba"]), t["address_mode_u"], t["address_mode_v"], t["filter_linear"], t["srgb"]) for t in b.scene.textures]
    ref = R.WgslReference(b.world.buffers(), tex, plugin.load_noise(), W, H)

    def raw(a):
        return np.ascontiguousarray(a).view(np.uint8).reshape(-1)

    def sync():
        for i in range(10):
            ref.reservoir[i][:] = raw(orc.readback(L.OUT_RESERVOIR_0 + i)).view(np.uint32).reshape(-1, 16)
        for s in range(3):
            ref.render[s][:] = raw(orc.readback(L.OUT_RENDER_DIRECT + s)).view(np.uint16).reshape(H, W, 4)
            ref.variance[s][:] = raw(orc.readback(L.OUT_VARIANCE_DIRECT + s)).view(np.float32).reshape(H, W)
        ref.albedo[:] = raw(orc.readback(L.OUT_ALBEDO)).view(np.uint16).reshape(H, W, 4)

    digests, differ = {}, []

    def record(name, mine, which):
        digests[name] = WC.digest(raw(mine))
        if not np.array_equal(raw(mine), raw(orc.readback(which))):
            differ.append(name)

    run = {O.PASS_ALBEDO: lambda inp: ref.full_screen_albedo(inp), O.PASS_DIRECT: lambda inp: ref.direct_lit(inp, False),
           O.PASS_EMISSIVE: lambda inp: ref.direct_lit(inp, True), O.PASS_EMISSIVE_SPATIAL: lambda inp: ref.spatial_reuse(inp, True),
           O.PASS_INDIRECT: lambda inp: ref.indirect_lit_ambient(inp), O.PASS_INDIRECT_SPATIAL: lambda inp: ref.spatial_reuse(inp, False)}
    for f in range(1, WC.PER_PASS_FRAMES + 1):
        inp = b.moving_inputs(f, WC.PER_PASS_STEP)
        orc.prepass(inp)
        ref.set_gbuffer(*[np.ascontiguousarray(orc.readback(k)) for k in WC.GBUFFER])
        for pid in WC.light_passes(inp):
            sync()
            run[pid](inp)
            orc.run_pass(inp, pid)
            planes = reference_planes(ref, b)
            for name, which in WC.PASS_PLANES:
                record(f"f{f}_p{pid}_{name}", planes[name], which)
        sync()
        for s in range(3):
            orc.run_pass(inp, O.PASS_DENOISE, s)
            ref.denoise_signal(inp, s)
            record(f"f{f}_denoised{s}", ref.denoise_render[s], L.OUT_DENOISED_DIRECT + s)
        orc.run_pass(inp, O.PASS_TONE_MAPPING)
        ref.tone_mapping(inp, True)
        record(f"f{f}_tone_mapped", ref.tone_mapped, L.OUT_TONE_MAPPED)
    return digests, differ


def pin_seed_digests():
    """{s<seed>_f<frame>_<plane>: digest} of the reference's planes for tools/fuzz_wgsl_pin.py's FIXED_SEEDS, and each seed's case"""
    import fuzz_wgsl_pin
    digests, cases = {}, []
    for seed in fuzz_wgsl_pin.FIXED_SEEDS:
        d, what = fuzz_wgsl_pin.reference_digests(seed)
        digests.update({f"s{seed}_{k}": v for k, v in d.items()})
        cases.append(what)
    return digests, cases


# the structs of light.wgsl (and the modules it imports) whose layouts include/hk_layout.h restates
LAYOUT_STRUCTS = ["Node", "Primitive", "Vertex", "Instance", "Material", "AliasEntry", "Emissive", "PackedReservoir", "Frame",
                  "PreviousView", "View"]


def struct_layouts():
    """{struct: {"align", "size", "offsets": {member: byte offset}}} as oracle/wgsl/wgsl2cpp.py derives them from WGSL's alignment rules"""
    import wgsl2cpp
    tr = wgsl2cpp.Translator(wgsl2cpp.preprocess(os.path.join(wgsl2cpp.REF_SHADERS, "light.wgsl"), set()))
    tr.module()
    out = {}
    for name in LAYOUT_STRUCTS:
        align, size, members = tr.struct_layout(name)
        out[name] = {"align": align, "size": size, "offsets": {m[0]: m[2] for m in members}}
    return out


def run_prepass_case(case):
    """the G-buffer of the case's compared frame as prepass.wgsl rasterises it (oracle/wgsl/raster_prepass.py)"""
    import raster_prepass as RP
    taa = WC.PREPASS_CASES[case][6]
    rp = RP.RasterPrepass(taa=taa)
    out = None
    for bench, inp, previous_models, _ in WC.prepass_sequence(case):
        out = rp.render(inp, bench.width, bench.height, bench.scene.meshes, bench.scene.inst_mesh, bench.world.buffers()["instances"], previous_models)
    return out


def prepass_fixture(case, r=None):
    """what tests/golden/wgsl_prepass_<case>.npz holds: the five planes of run_prepass_case (`r`, computed when None), cut to the case's
    window for WC.PREPASS_WINDOWS, and the number of triangles the rasteriser skipped"""
    r = run_prepass_case(case) if r is None else r
    planes = {k: r[k] for k, _ in WC.PREPASS_PLANES}
    if case in WC.PREPASS_WINDOWS:
        w, h = WC.PREPASS_CASES[case][2]
        planes = {k: WC.prepass_window(case, v, w, h) for k, v in planes.items()}
    return dict(planes, skipped_triangles=np.array(r["skipped_triangles"]))


def window_reports(case, r):
    """tests/test_wgsl_prepass.py's comparison of the oracle's G-buffer with the rasterised one `r`: on the full frame and on the window"""
    from tests.test_wgsl_prepass import compare, render_gbuffer
    bench, g = render_gbuffer(case, lambda b: b.oracle(), lambda o, b: o.update_instances_desc(b.world.scene_desc()))
    w, h = bench.width, bench.height
    x0, x1, y0, y1 = WC.PREPASS_WINDOWS[case]
    cut = prepass_fixture(case, r)
    return (compare({k: r[k] for k, _ in WC.PREPASS_PLANES}, g, w, h, case),
            compare(cut, {k: WC.prepass_window(case, v, w, h) for k, v in g.items()}, x1 - x0, y1 - y0, case))


def main():
    if not R.available():
        raise SystemExit("needs /root/reference and g++ (build container only)")
    out_dir = os.path.join(ROOT, "tests", "golden")
    if sys.argv[1:2] == ["--prepass"]:
        for case in (sys.argv[2:] or [c for c, v in WC.PREPASS_CASES.items() if v[7]]):
            r = run_prepass_case(case)
            np.savez_compressed(os.path.join(out_dir, f"wgsl_prepass_{case}.npz"), **prepass_fixture(case, r))
            print(f"prepass {case}: {r['fragments']} fragments shaded, {int((r['position'][..., 3] > 0).sum())} pixels covered")
            if case in WC.PREPASS_WINDOWS:
                full, window = window_reports(case, r)
                print(f"  the oracle against it, full frame: {full}\n  window {WC.PREPASS_WINDOWS[case]}: {window}")
        return
    if sys.argv[1:2] == ["--per-pass"]:
        for scene, config, size in WC.PER_PASS_CASES:
            digests, differ = run_per_pass(scene, config, size)
            WC.save_digests(os.path.join(out_dir, f"wgsl_per_pass_{scene}.npz"), digests)
            print(f"per pass {scene}: {len(digests)} plane digests; the oracle differs on {len(differ)} {differ[:6]}")
        return
    if sys.argv[1:2] == ["--pin-seeds"]:
        import fuzz_wgsl_pin
        digests, cases = pin_seed_digests()
        for seed, what in zip(fuzz_wgsl_pin.FIXED_SEEDS, cases):
            print(f"seed {seed}: {sum(k.startswith(f's{seed}_') for k in digests)} plane digests; {what}")
        WC.save_digests(os.path.join(out_dir, "wgsl_pin_seeds.npz"), digests, seeds=np.array(fuzz_wgsl_pin.FIXED_SEEDS), cases=np.array(cases))
        return
    if sys.argv[1:2] == ["--layouts"]:
        import json
        with open(os.path.join(out_dir, "wgsl_struct_layouts.json"), "w") as f:
            json.dump(struct_layouts(), f, indent=1)
            f.write("\n")
        return
    for case in (sys.argv[1:] or WC.CASES):
        digests, last = run_case(case)
        names = sorted(digests)
        np.savez_compressed(os.path.join(out_dir, f"wgsl_{case}.npz"), names=np.array(names), digests=np.array([digests[n] for n in names]),
                            last_tone_mapped=last)
        print(f"{case}: {len(names)} plane digests over {WC.CASES[case][3]} frames")


if __name__ == "__main__":
    main()
