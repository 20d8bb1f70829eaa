"""SURVEY 8(f) rank 4 — run-time scene ingest of the host mirror (host/gltf_ingest.cpp: hikari_world_load_gltf, hikari_decode_png).

  * scenes/cornell.glb (the reference's data asset assets/models/cornell.glb, 9.7 KB, examples/cornell.rs:40) loaded at run time gives
    the SAME nine scene buffers, record for record, as the offline-converted scenes/cornell.npz the benchmark uses;
  * a synthetic .gltf with data: URIs — TRS and matrix nodes three levels deep, two primitives on one mesh, strided / normalised
    accessors, five texture slots over PNG and JPEG images, all three wrap modes, a primitive without material — against the offline
    converter tools/make_assets.py (an independent Python reading of the same rules);
  * triangle strips (mod.rs:433-450) against the equivalent list;
  * the PNG decoder against Pillow over colour types, bit depths and all five scanline filters; malformed files are refused."""
import base64
import ctypes as C
import hashlib
import io
import json
import os
import struct
import sys
import zlib

import numpy as np
import pytest

from bevy_hikari_b200 import layout as L
from bevy_hikari_b200 import plugin, scenes
from bevy_hikari_b200._ffi import host_lib
from tests.conftest import ROOT

PIL = pytest.importorskip("PIL.Image")


def same_records(a, b, what):
    assert a.shape == b.shape, (what, a.shape, b.shape)
    for field in (a.dtype.names or [None]):
        x = a[field] if field else a
        y = b[field] if field else b
        assert np.ascontiguousarray(x).tobytes() == np.ascontiguousarray(y).tobytes(), (what, field)


def same_worlds(w1, w2):
    b1, b2 = w1.buffers(), w2.buffers()
    for name in b1:
        same_records(b1[name], b2[name], name)


def textures_of(world):
    d = world.scene_desc()
    out = []
    arr = C.cast(d.textures, C.POINTER(L.TextureDesc))
    for i in range(d.texture_count):
        t = arr[i]
        out.append((np.frombuffer(C.string_at(t.rgba8, t.width * t.height * 4), np.uint8).reshape(t.height, t.width, 4).copy(),
                    t.address_mode_u, t.address_mode_v, t.filter_linear, t.srgb))
    return out


def test_cornell_glb_at_run_time_equals_the_offline_converted_scene():
    runtime = plugin.World()
    counts = runtime.load_gltf(os.path.join(ROOT, "scenes", "cornell.glb"))
    assert (counts.mesh_count, counts.material_count, counts.instance_count, counts.texture_count) == (8, 8, 8, 0)
    runtime.prepare()
    offline = scenes.cornell().populate(plugin.World())
    same_worlds(runtime, offline)
    assert runtime.buffers()["emissives"].shape == (1,)          # the ceiling light


# ------------------------------------------------------------------------------------------------ a synthetic document
def png_bytes(img, **kw):
    b = io.BytesIO()
    img.save(b, "PNG", **kw)
    return b.getvalue()


def data_uri(raw, mime="application/octet-stream"):
    return f"data:{mime};base64," + base64.b64encode(raw).decode()


def synthetic_gltf(tmp_path, strip=False):
    rng = np.random.default_rng(5)
    # mesh 0 primitive 0: a 3 x 3 grid of quads (interleaved buffer: position | normal, stride 24); primitive 1: one triangle, u16 UVs
    n = 4
    gx, gz = np.meshgrid(np.arange(n, dtype=np.float32), np.arange(n, dtype=np.float32))
    pos = np.stack([gx.ravel(), 0.1 * rng.random(n * n).astype(np.float32), gz.ravel()], 1).astype(np.float32)
    nrm = np.tile(np.array([[0, 1, 0]], np.float32), (n * n, 1))
    uv = (pos[:, [0, 2]] / (n - 1)).astype(np.float32)
    idx = []
    for z in range(n - 1):
        for x in range(n - 1):
            a = z * n + x
            idx += [a, a + n, a + 1, a + 1, a + n, a + n + 1]
    idx = np.array(idx, np.uint16)
    inter = np.concatenate([pos, nrm], 1).astype(np.float32).tobytes()
    tri_pos = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)
    tri_nrm = np.tile(np.array([[0, 0, 1]], np.float32), (3, 1))
    tri_uv = np.array([[0, 0], [65535, 0], [0, 65535]], np.uint16)
    strip_idx = np.array([0, 4, 1, 5, 2, 6, 3, 7], np.uint32)       # one strip over the first two grid rows
    blob = bytearray()

    def add(raw):
        while len(blob) % 4:
            blob.append(0)
        off = len(blob)
        blob.extend(raw)
        return off
    o_inter, o_uv, o_idx = add(inter), add(uv.tobytes()), add(idx.tobytes())
    o_tp, o_tn, o_tuv, o_strip = add(tri_pos.tobytes()), add(tri_nrm.tobytes()), add(tri_uv.tobytes()), add(strip_idx.tobytes())
    # images: RGB PNG, RGBA PNG, palette PNG, a JPEG, a grey PNG as a side-car file
    im_rgb = PIL.fromarray(rng.integers(0, 256, (8, 16, 3), dtype=np.uint8), "RGB")
    im_rgba = PIL.fromarray(rng.integers(0, 256, (5, 7, 4), dtype=np.uint8), "RGBA")
    im_pal = PIL.fromarray(rng.integers(0, 256, (6, 6, 3), dtype=np.uint8), "RGB").quantize(16)
    im_jpg = PIL.fromarray((np.add.outer(np.arange(16), np.arange(16)) * 8).astype(np.uint8), "L").convert("RGB")
    jb = io.BytesIO(); im_jpg.save(jb, "JPEG", quality=90)
    im_l16 = PIL.fromarray(rng.integers(0, 256, (4, 4), dtype=np.uint8), "L")      # grey side-car file
    o_img0 = add(png_bytes(im_rgb)); l_img0 = len(blob) - o_img0
    doc = {
        "asset": {"version": "2.0"}, "scene": 0,
        "scenes": [{"nodes": [0, 3]}],
        "nodes": [
            {"translation": [1.5, 0.25, -2.0], "rotation": [0.0, 0.3826834, 0.0, 0.9238795], "scale": [1.0, 2.0, 0.5], "children": [1]},
            {"matrix": [0.5, 0, 0, 0, 0, 0.5, 0, 0, 0, 0, 0.5, 0, 3, 1, 2, 1], "mesh": 0, "children": [2]},
            {"rotation": [0.7071068, 0.0, 0.0, 0.7071068], "mesh": 1},
            {"translation": [-4.0, 0.0, 1.0], "mesh": 1},
        ],
        "meshes": [
            {"primitives": [{"attributes": {"POSITION": 0, "NORMAL": 1, "TEXCOORD_0": 2}, "indices": 3, "material": 1},
                            {"attributes": {"POSITION": 4, "NORMAL": 5, "TEXCOORD_0": 6}, "material": 0}]},
            {"primitives": [{"attributes": {"POSITION": 4, "NORMAL": 5, "TEXCOORD_0": 6}}
                            if not strip else {"attributes": {"POSITION": 0, "NORMAL": 1, "TEXCOORD_0": 2}, "indices": 7, "mode": 5, "material": 0}]},
        ],
        "buffers": [{"byteLength": 0, "uri": ""}],
        "bufferViews": [
            {"buffer": 0, "byteOffset": o_inter, "byteLength": len(inter), "byteStride": 24},
            {"buffer": 0, "byteOffset": o_uv, "byteLength": uv.nbytes},
            {"buffer": 0, "byteOffset": o_idx, "byteLength": idx.nbytes},
            {"buffer": 0, "byteOffset": o_tp, "byteLength": tri_pos.nbytes},
            {"buffer": 0, "byteOffset": o_tn, "byteLength": tri_nrm.nbytes},
            {"buffer": 0, "byteOffset": o_tuv, "byteLength": tri_uv.nbytes},
            {"buffer": 0, "byteOffset": o_strip, "byteLength": strip_idx.nbytes},
            {"buffer": 0, "byteOffset": o_img0, "byteLength": l_img0},
        ],
        "accessors": [
            {"bufferView": 0, "byteOffset": 0, "componentType": 5126, "count": n * n, "type": "VEC3"},
            {"bufferView": 0, "byteOffset": 12, "componentType": 5126, "count": n * n, "type": "VEC3"},
            {"bufferView": 1, "componentType": 5126, "count": n * n, "type": "VEC2"},
            {"bufferView": 2, "componentType": 5123, "count": len(idx), "type": "SCALAR"},
            {"bufferView": 3, "componentType": 5126, "count": 3, "type": "VEC3"},
            {"bufferView": 4, "componentType": 5126, "count": 3, "type": "VEC3"},
            {"bufferView": 5, "componentType": 5123, "count": 3, "type": "VEC2", "normalized": True},
            {"bufferView": 6, "componentType": 5125, "count": len(strip_idx), "type": "SCALAR"},
        ],
        "materials": [
            {"pbrMetallicRoughness": {"baseColorFactor": [0.8, 0.7, 0.6, 1.0], "roughnessFactor": 0.4, "metallicFactor": 0.1,
                                      "baseColorTexture": {"index": 0}, "metallicRoughnessTexture": {"index": 1}},
             "emissiveFactor": [0.5, 0.25, 0.125], "emissiveTexture": {"index": 2}, "normalTexture": {"index": 3},
             "occlusionTexture": {"index": 0}},
            {"pbrMetallicRoughness": {"baseColorTexture": {"index": 4}}},
        ],
        "textures": [{"source": 0, "sampler": 0}, {"source": 1, "sampler": 1}, {"source": 2}, {"source": 3, "sampler": 2}, {"source": 4, "sampler": 0}],
        "samplers": [{"wrapS": 33071, "wrapT": 33648, "magFilter": 9728}, {"wrapS": 10497, "wrapT": 33071}, {"magFilter": 9729}],
        "images": [
            {"bufferView": 7, "mimeType": "image/png"},
            {"uri": data_uri(png_bytes(im_rgba), "image/png")},
            {"uri": data_uri(png_bytes(im_pal), "image/png")},
            {"uri": data_uri(jb.getvalue(), "image/jpeg")},
            {"uri": "side car.png"},
        ],
    }
    with open(tmp_path / "side car.png", "wb") as f:
        f.write(png_bytes(im_l16))
    doc["images"][4]["uri"] = "side%20car.png"
    doc["buffers"][0] = {"byteLength": len(blob), "uri": data_uri(bytes(blob))}
    path = tmp_path / ("strip.gltf" if strip else "synthetic.gltf")
    with open(path, "w") as f:
        json.dump(doc, f)
    return str(path), doc


def world_from_converter(path):
    """the offline converter's reading of the same file, spawned the way scenes.py spawns an .npz"""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import make_assets
    z = make_assets.convert_gltf(path)
    w = plugin.World()
    for t in range(int(z["tex_count"])):
        info = z[f"t{t}_info"]
        w.add_texture(z[f"t{t}_rgba"], int(info[0]), int(info[1]), int(info[2]), int(info[3]))
    for i in range(int(z["mesh_count"])):
        w.add_mesh(z[f"m{i}_pos"], z[f"m{i}_nrm"], z[f"m{i}_uv"], z[f"m{i}_idx"])
    mats = np.zeros(len(z["mat_base_color"]), L.MATERIAL)
    mats["base_color"], mats["emissive"] = z["mat_base_color"], z["mat_emissive"]
    mats["perceptual_roughness"], mats["metallic"], mats["reflectance"] = z["mat_perceptual_roughness"], z["mat_metallic"], z["mat_reflectance"]
    for k, name in enumerate(("base_color_texture", "emissive_texture", "metallic_roughness_texture", "normal_map_texture", "occlusion_texture")):
        mats[name] = z["mat_textures"][:, k]
    for m in mats:
        w.add_material(m)
    for me, ma, xf in zip(z["inst_mesh"], z["inst_material"], z["inst_transform"]):
        w.add_instance(int(me), int(ma), xf)
    w.prepare()
    return w


def test_synthetic_document_equals_the_offline_converter(tmp_path):
    path, doc = synthetic_gltf(tmp_path)
    # the converter reads a primitive without material as material 0 and un-normalised u16 UVs as their integer values; give it the
    # same document with those two things spelled out (material named, UVs as floats) so that only shared rules are compared
    ref_doc = json.loads(json.dumps(doc))
    runtime = plugin.World()
    counts = runtime.load_gltf(path)
    assert (counts.mesh_count, counts.instance_count, counts.texture_count) == (3, 4, 6)
    assert counts.material_count == 3                    # two glTF materials + StandardMaterial::default() for mesh 1's primitive
    runtime.prepare()
    # reference document for the converter: explicit third material with bevy's defaults, float UVs
    ref_doc["materials"].append({"pbrMetallicRoughness": {"roughnessFactor": 0.089, "metallicFactor": 0.01}})
    ref_doc["meshes"][1]["primitives"][0]["material"] = 2
    blob = bytearray(base64.b64decode(ref_doc["buffers"][0]["uri"].split(",", 1)[1]))
    tri_uv = np.array([[0, 0], [1, 0], [0, 1]], np.float32)
    while len(blob) % 4:
        blob.append(0)
    off = len(blob); blob.extend(tri_uv.tobytes())
    ref_doc["bufferViews"].append({"buffer": 0, "byteOffset": off, "byteLength": tri_uv.nbytes})
    ref_doc["accessors"][6] = {"bufferView": len(ref_doc["bufferViews"]) - 1, "componentType": 5126, "count": 3, "type": "VEC2"}
    # ... and explicit indices 0 1 2 for the non-indexed triangle (the converter reads indexed primitives only)
    while len(blob) % 4:
        blob.append(0)
    off = len(blob); blob.extend(np.array([0, 1, 2], np.uint32).tobytes())
    ref_doc["bufferViews"].append({"buffer": 0, "byteOffset": off, "byteLength": 12})
    ref_doc["accessors"].append({"bufferView": len(ref_doc["bufferViews"]) - 1, "componentType": 5125, "count": 3, "type": "SCALAR"})
    ref_doc["meshes"][0]["primitives"][1]["indices"] = len(ref_doc["accessors"]) - 1
    ref_doc["meshes"][1]["primitives"][0]["indices"] = len(ref_doc["accessors"]) - 1
    ref_doc["buffers"][0] = {"byteLength": len(blob), "uri": data_uri(bytes(blob))}
    # ... and images as plain side-car files (the converter does not read data: URIs or percent-encoded names)
    for k, im in enumerate(ref_doc["images"]):
        uri = im.get("uri")
        if uri and uri.startswith("data:"):
            name = f"image{k}." + ("jpg" if "jpeg" in uri[:24] else "png")
            with open(tmp_path / name, "wb") as f:
                f.write(base64.b64decode(uri.split(",", 1)[1]))
            im["uri"] = name
        elif uri:
            im["uri"] = uri.replace("%20", " ")
    ref_path = tmp_path / "reference.gltf"
    with open(ref_path, "w") as f:
        json.dump(ref_doc, f)
    offline = world_from_converter(str(ref_path))
    same_worlds(runtime, offline)
    t_run, t_off = textures_of(runtime), textures_of(offline)
    assert len(t_run) == len(t_off) == 6                 # image 0 is used in two colour spaces
    for a, b in zip(t_run, t_off):
        assert a[1:] == b[1:], (a[1:], b[1:])
        assert np.array_equal(a[0], b[0])
    assert [t[4] for t in t_run] == [1, 1, 0, 0, 0, 1]   # first-use order: base colour, emissive (sRGB), metallic-roughness, normal, occlusion (linear); base colour of material 1
    assert t_run[0][1:4] == (1, 2, 0) and t_run[1][1:4] == (0, 0, 1) and t_run[2][1:4] == (0, 1, 1)   # clamp / mirror / nearest; no sampler; repeat / clamp


def test_triangle_strip_primitive_equals_its_list(tmp_path):
    path, _ = synthetic_gltf(tmp_path, strip=True)
    w = plugin.World()
    w.load_gltf(path)
    w.prepare()
    inst = w.buffers()["instances"]
    strip_mesh = inst[-1]["mesh"]                               # the last instance (node 3) uses the strip primitive
    # 8 strip indices -> 6 triangles (mod.rs:441-448); as many BLAS leaves
    nodes = w.buffers()["asset_nodes"][strip_mesh["node_offset"]:strip_mesh["node_offset"] + strip_mesh["node_count"]]
    assert int((nodes["entry_index"] >= 0x80000000).sum()) == 6 and strip_mesh["node_count"] == 3 * 6 - 2
    assert w.mesh_error(2) == 0


def test_missing_attribute_drops_the_instance_like_the_reference(tmp_path):
    path, doc = synthetic_gltf(tmp_path)
    del doc["meshes"][1]["primitives"][0]["attributes"]["NORMAL"]
    with open(path, "w") as f:
        json.dump(doc, f)
    w = plugin.World()
    c = w.load_gltf(path)
    w.prepare()
    assert c.instance_count == 4 and len(w.buffers()["instances"]) == 2        # the two instances of mesh 1 are dropped (mod.rs:301-308)
    assert w.mesh_error(c.first_mesh + 2) == 2                                 # MissingAttributeNormal


def test_jpeg_without_a_decoder_and_malformed_files_are_refused(tmp_path):
    path, _ = synthetic_gltf(tmp_path)
    with pytest.raises(RuntimeError, match="image/jpeg"):
        plugin.World().load_gltf(path, decoder=None)
    bad = tmp_path / "bad.gltf"
    bad.write_text('{"asset": {"version": "2.0"}, "scenes": [{"nodes": [0]}], "nodes": [{"children": [0]}]}')
    with pytest.raises(RuntimeError, match="cycle"):
        plugin.World().load_gltf(str(bad))
    bad.write_text('{"asset": ')
    with pytest.raises(RuntimeError, match="malformed"):
        plugin.World().load_gltf(str(bad))
    with pytest.raises(RuntimeError, match="cannot read"):
        plugin.World().load_gltf(str(tmp_path / "absent.glb"))


# ------------------------------------------------------------------------------------------------ PNG
def decode(raw):
    w, h = C.c_uint32(), C.c_uint32()
    buf = (C.c_uint8 * len(raw)).from_buffer_copy(raw)
    if not host_lib().hikari_decode_png(buf, len(raw), None, C.byref(w), C.byref(h)):
        return None
    out = np.zeros((h.value, w.value, 4), np.uint8)
    assert host_lib().hikari_decode_png(buf, len(raw), out.ctypes.data, C.byref(w), C.byref(h))
    return out


def raw_png(width, height, depth, ctype, rows, filters, extra=b""):
    """a PNG written by hand so that every scanline filter type is exercised (Pillow picks filters itself)"""
    def chunk(t, body):
        return struct.pack(">I", len(body)) + t + body + struct.pack(">I", zlib.crc32(t + body))
    channels = {0: 1, 2: 3, 3: 1, 4: 2, 6: 4}[ctype]
    bpp = max(1, channels * depth // 8)
    data, prev = b"", bytes(len(rows[0]))
    for y, line in enumerate(rows):
        f = filters[y % len(filters)]
        enc = bytearray(len(line))
        for x in range(len(line)):
            a = line[x - bpp] if x >= bpp else 0
            b = prev[x]
            c = prev[x - bpp] if x >= bpp else 0
            if f == 0: p = 0
            elif f == 1: p = a
            elif f == 2: p = b
            elif f == 3: p = (a + b) // 2
            else:
                pp = a + b - c
                pa, pb, pc = abs(pp - a), abs(pp - b), abs(pp - c)
                p = a if (pa <= pb and pa <= pc) else (b if pb <= pc else c)
            enc[x] = (line[x] - p) & 255
        data += bytes([f]) + bytes(enc)
        prev = line
    return (b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", width, height, depth, ctype, 0, 0, 0)) + extra +
            chunk(b"IDAT", zlib.compress(data)) + chunk(b"IEND", b""))


@pytest.mark.parametrize("mode", ["L", "LA", "RGB", "RGBA", "P", "1", "I;16"])
def test_png_decoder_equals_pillow(mode):
    rng = np.random.default_rng(11)
    for (w, h) in ((1, 1), (7, 5), (33, 17), (64, 64)):
        if mode == "P":
            im = PIL.fromarray(rng.integers(0, 256, (h, w, 3), dtype=np.uint8), "RGB").quantize(13)
        elif mode == "1":
            im = PIL.fromarray((rng.random((h, w)) > 0.5).astype(np.uint8) * 255, "L").convert("1")
        elif mode == "I;16":
            im = PIL.fromarray(rng.integers(0, 65536, (h, w)).astype(np.uint16))
        else:
            n = {"L": 1, "LA": 2, "RGB": 3, "RGBA": 4}[mode]
            a = rng.integers(0, 256, (h, w, n), dtype=np.uint8)
            im = PIL.fromarray(a[..., 0] if n == 1 else a, mode)
        raw = png_bytes(im)
        got = decode(raw)
        assert got is not None, (mode, w, h)
        if mode == "I;16":
            want = np.asarray(im, np.uint16) >> 8
            want = np.stack([want, want, want, np.full_like(want, 255)], -1).astype(np.uint8)
        else:
            want = np.asarray(im.convert("RGBA"), np.uint8)
        assert np.array_equal(got, want), (mode, w, h)


@pytest.mark.parametrize("ctype,depth", [(0, 8), (2, 8), (6, 8), (4, 8), (2, 16), (0, 4), (0, 2)])
def test_png_every_scanline_filter(ctype, depth):
    rng = np.random.default_rng(3)
    w, h = 19, 11
    channels = {0: 1, 2: 3, 4: 2, 6: 4}[ctype]
    row_bytes = (w * channels * depth + 7) // 8
    rows = [bytes(rng.integers(0, 256, row_bytes, dtype=np.uint8)) for _ in range(h)]
    raw = raw_png(w, h, depth, ctype, rows, [0, 1, 2, 3, 4])
    got = decode(raw)
    want = np.asarray(PIL.open(io.BytesIO(raw)).convert("RGBA"), np.uint8) if depth == 8 else None
    assert got is not None and got.shape == (h, w, 4)
    if want is not None:
        assert np.array_equal(got, want)
    elif depth == 16:
        px = np.frombuffer(b"".join(rows), np.uint8).reshape(h, w, channels, 2)[..., 0]     # high bytes
        assert np.array_equal(got[..., :3], px) and (got[..., 3] == 255).all()
    else:
        bits = np.unpackbits(np.frombuffer(b"".join(rows), np.uint8).reshape(h, row_bytes), axis=1)[:, :w * depth].reshape(h, w, depth)
        val = (bits * (1 << np.arange(depth - 1, -1, -1))).sum(-1)
        assert np.array_equal(got[..., 0], (val * 255 // ((1 << depth) - 1)).astype(np.uint8))


def test_png_decoder_refuses_what_it_does_not_decode():
    good = png_bytes(PIL.fromarray(np.zeros((4, 4, 3), np.uint8), "RGB"))
    assert decode(good) is not None
    assert decode(good[:40]) is None                         # truncated
    assert decode(b"\x89PNG\r\n\x1a\n" + b"\0" * 32) is None
    assert decode(b"not a png at all") is None
    b = io.BytesIO()
    PIL.fromarray(np.zeros((8, 8, 3), np.uint8), "RGB").save(b, "PNG", interlace=True) if False else None
    rows = [bytes(8 * 3)] * 8
    interlaced = bytearray(raw_png(8, 8, 8, 2, rows, [0]))
    interlaced[28] = 1                                        # IHDR interlace method = Adam7 (CRC now wrong too; refused either way)
    assert decode(bytes(interlaced)) is None


COMPONENT = {5123: np.uint16, 5125: np.uint32, 5126: np.float32}


def house_glb(glb, npz, tmp_path):
    """The reference's house model `glb` rebuilt from its JSON chunk (tests/golden/gltf_houses.json, tools/make_assets.py --house-fixture)
    and the shipped scene file: the geometry bytes are the original file's (SHA-256 checked), each image is the scene file's texture —
    the original PNG box-filtered to at most 512 px — PNG-encoded in the original's colour mode.  Returns the path of the GLB."""
    with open(os.path.join(ROOT, "tests", "golden", "gltf_houses.json")) as f:
        fx = json.load(f)[os.path.basename(glb)]
    assert fx["npz"] == npz
    doc, z = fx["json"], np.load(os.path.join(ROOT, "scenes", f"{npz}.npz"))
    views = doc["bufferViews"]
    image_views = {im["bufferView"] for im in doc["images"]}
    binary = bytearray(doc["buffers"][0]["byteLength"])
    prim = 0
    for mesh in doc["meshes"]:
        for p in mesh["primitives"]:
            for acc, key in ((p["attributes"]["POSITION"], "pos"), (p["attributes"]["NORMAL"], "nrm"), (p["attributes"]["TEXCOORD_0"], "uv"),
                             (p["indices"], "idx")):
                a = doc["accessors"][acc]
                raw = z[f"m{prim}_{key}"].astype(COMPONENT[a["componentType"]]).tobytes()
                start = views[a["bufferView"]].get("byteOffset", 0) + a.get("byteOffset", 0)
                binary[start:start + len(raw)] = raw
            prim += 1
    geometry = b"".join(binary[v.get("byteOffset", 0):v.get("byteOffset", 0) + v["byteLength"]] for i, v in enumerate(views) if i not in image_views)
    assert hashlib.sha256(geometry).hexdigest() == fx["geometry_sha256"], "geometry differs from the reference's file"
    for im, t, mode in zip(doc["images"], fx["image_texture"], fx["image_mode"]):
        png = png_bytes(PIL.fromarray(z[f"t{t}_rgba"]).convert(mode))
        binary += bytes(-len(binary) % 4)
        views[im["bufferView"]].update(byteOffset=len(binary), byteLength=len(png))
        binary += png
    binary += bytes(-len(binary) % 4)
    doc["buffers"][0]["byteLength"] = len(binary)
    js = json.dumps(doc).encode()
    js += b" " * (-len(js) % 4)
    path = tmp_path / f"{npz}.glb"
    path.write_bytes(struct.pack("<III", 0x46546C67, 2, 28 + len(js) + len(binary)) + struct.pack("<II", len(js), 0x4E4F534A) + js +
                     struct.pack("<II", len(binary), 0x004E4942) + bytes(binary))
    return str(path)


@pytest.mark.parametrize("glb,npz", [("Low Poly/Big House.glb", "house"), ("Low Poly/Big House 2.glb", "house2"), ("Low Poly/Big House 3.glb", "house3")])
def test_reference_house_models_at_run_time_equal_the_shipped_scene_files(glb, npz, tmp_path):
    """examples/city.rs:56-202 loads these three files; the benchmark's city scene is built from their offline conversions.  The
    run-time loader must give the same meshes, materials, BLAS records and textures (13 textures in all).  The files themselves are
    5 to 7 MB of PNG; what is loaded is the same document rebuilt around the textures at the size the scene files ship (house_glb)."""
    meshes, mats, textures, inst_mesh, inst_material, inst_transform = scenes._load_npz(npz)
    offline = plugin.World()
    for t in textures:
        offline.add_texture(t["rgba"], t["address_mode_u"], t["address_mode_v"], t["filter_linear"], t["srgb"])
    for m in meshes:
        offline.add_mesh(*m)
    for m in mats:
        offline.add_material(m)
    for me, ma, xf in zip(inst_mesh, inst_material, inst_transform):
        offline.add_instance(int(me), int(ma), xf)
    offline.prepare()
    runtime = plugin.World()
    runtime.load_gltf(house_glb(glb, npz, tmp_path))
    runtime.prepare()
    same_worlds(runtime, offline)
    t_run, t_off = textures_of(runtime), textures_of(offline)
    assert len(t_run) == len(t_off) and len(t_run) > 0
    for a, b in zip(t_run, t_off):
        assert a[1:] == b[1:]
        assert np.array_equal(a[0], b[0])


def test_shape_generators_of_the_host_mirror_equal_the_python_ones():
    """Mesh::from(shape::Plane / UVSphere / Box) in C++ (host/gltf_ingest.cpp) against scenes.py's generators: same vertices, same BLAS"""
    for kind, params, py in (("plane", (10.0,), scenes._plane_mesh(10.0)), ("uv_sphere", (0.5, 36, 18), scenes._uv_sphere_mesh(0.5, 36, 18)),
                             ("uv_sphere", (1.25, 7, 5), scenes._uv_sphere_mesh(1.25, 7, 5)), ("box", (1.0, 2.0, 0.5), scenes._box_mesh(1.0, 2.0, 0.5))):
        a, b = plugin.World(), plugin.World()
        assert a.add_shape(kind, *params) == 0
        b.add_mesh(*py)
        for w in (a, b):
            w.add_material(scenes._std_material())
            w.add_instance(0, 0, np.eye(4, dtype=np.float32).reshape(16))
            w.prepare()
        same_worlds(a, b)
