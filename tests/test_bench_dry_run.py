"""bench.py's single-GPU flow (replays, the two timed arms, the one-kernel ring timing, the JSON line) dry-run on the kernel-logic
emulation with a stand-in for the sliver of torch it touches: a Python error in bench.py must not cost a GPU call.  The numbers of
such a run mean nothing and are not looked at; the keys of the contract are."""
import json
import os
import subprocess
import sys

import numpy as np

from tests.conftest import ROOT

# frames 1 .. N of cornell_256 through render_frame on the library argv[1]; saves frames N - 1 and N, read back as a caller would
RENDER_FRAMES = """
import sys
import numpy as np
import bench
from bevy_hikari_b200 import _ffi, layout as L, plugin
_ffi.LIB_PATH = sys.argv[1]
cfg, scene, world, W, H, view, pview, lights, settings = bench.make_bench("cornell_256")
dev = plugin.HikariPlugin(W, H, cuda_device=0)
dev.upload_scene(world)
out = []
for n in range(1, int(sys.argv[2]) + 1):
    dev.render_frame(plugin.make_frame_inputs(settings, n, view, pview, lights))
    out = (out + [dev.readback(L.OUT_TONE_MAPPED).astype(np.float32)])[-2:]
np.save(sys.argv[3], np.stack(out))
"""


def test_bench_line_has_the_contract_keys_on_the_emulated_kernels(tmp_path):
    sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
    import build_emu
    lib = build_emu.build()
    env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, "tests", "emu", "fake_torch"))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--lib", lib, "--config", "cornell_256", "--steps", "3", "--warmup", "3",
                        "--no-cpu-baseline", "--print-frame-hash", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, env=env,
                       timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
                "data", "config", "e2e", "gpu_launches", "roofline", "clocks", "frame_ms", "value_vs_e2e", "kernel_ms"):
        assert key in d, key
    assert d["steps"] == 3 and d["n_gpus"] == 1 and d["gpu_launches"] > 0
    assert d["roofline"]["kernel_ms_source"] == "live, timed region" and d["roofline"]["kernel"] in d["kernel_ms"]
    assert set(d["e2e"]) >= {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} and d["e2e"]["d2h_bytes_per_step"] == 256 * 256 * 8
    assert len(d["frame_check"]["unsharded_sha256"]) == 64
    # animated-scene block: the host path and the device-side rebuild (hk_scene_update_transforms) were both exercised
    assert d["scene_update"]["device_path_taken"] is True and d["scene_update"]["device_rebuild_done_ms"] > 0
    img = np.load(tmp_path / "tone_mapped.npy")         # --dump-outputs: the last timed frame, as a caller reads it back
    assert img.dtype == np.float32 and img.shape == (256, 256, 4) and np.isfinite(img).all() and img[..., :3].mean() > 0.05
    # ... and that frame is frame W + K = 6 of the sequence, not any other
    r = subprocess.run([sys.executable, "-c", RENDER_FRAMES, lib, "6", str(tmp_path / "frames.npy")], capture_output=True, text=True,
                       env=dict(env, PYTHONPATH=os.pathsep.join([env["PYTHONPATH"], ROOT])), timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    before_last, last = np.load(tmp_path / "frames.npy")
    assert np.array_equal(img, last) and not np.array_equal(img, before_last)


def test_dump_outputs_stays_within_its_limit(tmp_path):
    """a 1080p frame is written whole; a 4K frame (133 MB as float32) becomes a pixel sample, and no file exceeds DUMP_LIMIT"""
    import bench
    rng = np.random.default_rng(1)
    for (h, w), name in (((1080, 1920), "tone_mapped"), ((2160, 3840), "tone_mapped_sample")):
        frame = rng.random((h, w, 4), np.float32).astype(np.float16)
        out = tmp_path / f"{h}p"
        bench.dump_outputs(str(out), frame)
        assert [f.name for f in out.iterdir()] == [name + ".npy"]
        assert (out / (name + ".npy")).stat().st_size <= bench.DUMP_LIMIT
        got = np.load(out / (name + ".npy"))
        if name == "tone_mapped":
            assert np.array_equal(got, frame.astype(np.float32))
        else:       # sampled pixels are pixels of the frame, in pixel order
            assert got.shape[1] == 4 and got.nbytes > 0.99 * (bench.DUMP_LIMIT - bench.NPY_HEADER)
            px = frame.reshape(-1, 4).astype(np.float32)
            keep = np.sort(np.random.default_rng(0).choice(px.shape[0], got.shape[0], replace=False))
            assert np.array_equal(got, px[keep])


def test_reference_arm_never_maps_the_cuda_library():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "cornell_256", "--steps", "1",
                        "--warmup", "3"], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert d["impl"] == "reference" and d["mapped_cuda_library"] is False
    assert d["config"]["rendered_width"] == 256 and d["config"]["rendered_pixel_fraction"] == 1.0
