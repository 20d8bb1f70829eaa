#!/usr/bin/env python
"""Convert the reference's *data* assets into the small scene files this repo ships.

Runs only in the build container (it reads /root/reference, which does not exist on the GPU box); its outputs
are committed:

  data/noise_rgba8_64x64x16.bin   <- src/noise/LDR_RGBA_{0..15}.png   (lib.rs:189-219: 16 blue-noise textures,
                                     decoded as linear Rgba8Unorm, `is_srgb = false`)
  scenes/cornell.npz              <- assets/models/cornell.glb         (examples/cornell.rs:40)
  scenes/city.npz                 <- assets/models/Low Poly/Big House{, 2, 3}.glb (examples/city.rs:56-202), meshes
                                     + materials + textures only; the instance list is built in scenes.py
  scenes/town.npz                 <- assets/models/scene.gltf          (examples/scene.rs:80-84; BASELINE configs[2]),
                                     84 meshes / 120 440 triangles / 66 materials; the 52 embedded PNGs are shipped
                                     box-filtered to at most 256 x 256 (--scene)
  tests/golden/gltf_houses.json   <- the three house GLBs: what rebuilds them from scenes/house*.npz (--house-fixture)

A scene file holds what a Bevy app would hand to the plugin: meshes (position/normal/uv/indices per glTF
primitive), per-instance (mesh, material, world transform), StandardMaterial parameters, RGBA8 textures.
Entity / HandleId order is random in the reference (SURVEY.md App. C.16); here instance order = depth-first glTF
node order and material order = glTF material order.
"""
import io
import json
import os
import struct
import sys

import numpy as np

REF = "/root/reference"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

F32 = np.float32


def load_glb(path):
    d = open(path, "rb").read()
    magic, ver, length = struct.unpack("<III", d[:12])
    assert magic == 0x46546C67
    off = 12
    js, binchunk = None, None
    while off < length:
        clen, ctype = struct.unpack("<II", d[off:off + 8])
        body = d[off + 8:off + 8 + clen]
        if ctype == 0x4E4F534A:
            js = json.loads(body)
        elif ctype == 0x004E4942:
            binchunk = body
        off += 8 + clen
    return js, [binchunk]


def load_gltf(path):
    """.gltf with embedded (data: URI) or side-car buffers."""
    import base64
    js = json.load(open(path))
    bufs = []
    for b in js["buffers"]:
        uri = b["uri"]
        if uri.startswith("data:"):
            bufs.append(base64.b64decode(uri.split(",", 1)[1]))
        else:
            bufs.append(open(os.path.join(os.path.dirname(path), uri), "rb").read())
    return js, bufs


COMP = {5120: np.int8, 5121: np.uint8, 5122: np.int16, 5123: np.uint16, 5125: np.uint32, 5126: np.float32}
NCOMP = {"SCALAR": 1, "VEC2": 2, "VEC3": 3, "VEC4": 4, "MAT4": 16}


def accessor(js, bufs, idx):
    a = js["accessors"][idx]
    bv = js["bufferViews"][a["bufferView"]]
    dt = np.dtype(COMP[a["componentType"]])
    n = NCOMP[a["type"]]
    start = bv.get("byteOffset", 0) + a.get("byteOffset", 0)
    stride = bv.get("byteStride", 0)
    buf = bufs[bv["buffer"]]
    if stride and stride != dt.itemsize * n:
        out = np.zeros((a["count"], n), dt)
        for i in range(a["count"]):
            out[i] = np.frombuffer(buf, dt, n, start + i * stride)
        return out
    return np.frombuffer(buf, dt, a["count"] * n, start).reshape(a["count"], n).copy()


def quat_to_mat3(q):
    # glam Mat3::from_quat (f32)
    x, y, z, w = [F32(v) for v in q]
    x2, y2, z2 = x + x, y + y, z + z
    xx, xy, xz = x * x2, x * y2, x * z2
    yy, yz, zz = y * y2, y * z2, z * z2
    wx, wy, wz = w * x2, w * y2, w * z2
    one = F32(1)
    return np.array([[one - (yy + zz), xy + wz, xz - wy],
                     [xy - wz, one - (xx + zz), yz + wx],
                     [xz + wy, yz - wx, one - (xx + yy)]], F32)  # rows here are COLUMNS of the matrix


def node_local_matrix(node):
    """Column-major 4x4 as a (4,4) array m[col][row]."""
    if "matrix" in node:
        return np.array(node["matrix"], F32).reshape(4, 4)
    t = np.array(node.get("translation", [0, 0, 0]), F32)
    r = node.get("rotation", [0, 0, 0, 1])
    s = np.array(node.get("scale", [1, 1, 1]), F32)
    cols = quat_to_mat3(r)
    m = np.zeros((4, 4), F32)
    for c in range(3):
        m[c, :3] = cols[c] * s[c]
    m[3, :3] = t
    m[3, 3] = 1
    return m


def mat_mul(a, b):
    """a*b for column-major [col][row] arrays, float32 accumulation left to right."""
    out = np.zeros((4, 4), F32)
    for c in range(4):
        for r in range(4):
            acc = F32(0)
            for k in range(4):
                acc = F32(acc + a[k, r] * b[c, k])
            out[c, r] = acc
    return out


def decode_image(js, bufs, image_index, base_dir):
    from PIL import Image
    img = js["images"][image_index]
    if "bufferView" in img:
        bv = js["bufferViews"][img["bufferView"]]
        raw = bufs[bv["buffer"]][bv.get("byteOffset", 0):bv.get("byteOffset", 0) + bv["byteLength"]]
        im = Image.open(io.BytesIO(raw))
    else:
        im = Image.open(os.path.join(base_dir, img["uri"]))
    return np.asarray(im.convert("RGBA"), np.uint8).copy()


def box_filtered(img, max_tex):
    """`img` box-filtered so that its larger side is at most `max_tex` (None: unchanged)"""
    if max_tex and max(img.shape[:2]) > max_tex:
        from PIL import Image
        s = max_tex / max(img.shape[:2])
        img = np.asarray(Image.fromarray(img).resize((max(1, int(img.shape[1] * s)), max(1, int(img.shape[0] * s))),
                                                     Image.BOX), np.uint8).copy()
    return img


def convert_gltf(path, max_tex=None):
    """Return dict of arrays: meshes, instances (depth-first node order), materials, textures."""
    js, bufs = load_gltf(path) if path.endswith(".gltf") else load_glb(path)
    out = {}
    meshes = []       # one entry per glTF primitive
    prim_of_mesh = {}  # (mesh, prim) -> flat mesh index
    for mi, m in enumerate(js["meshes"]):
        for pi, p in enumerate(m["primitives"]):
            assert p.get("mode", 4) == 4, "triangle lists only"
            at = p["attributes"]
            pos = accessor(js, bufs, at["POSITION"]).astype(F32)
            nrm = accessor(js, bufs, at["NORMAL"]).astype(F32)
            uv = accessor(js, bufs, at["TEXCOORD_0"]).astype(F32)
            idx = accessor(js, bufs, p["indices"]).astype(np.uint32).reshape(-1)
            prim_of_mesh[(mi, pi)] = len(meshes)
            meshes.append((pos, nrm, uv, idx, p.get("material", 0)))
    inst_mesh, inst_mat, inst_xf = [], [], []

    def walk(ni, parent):
        node = js["nodes"][ni]
        world = mat_mul(parent, node_local_matrix(node))
        if "mesh" in node:
            for pi in range(len(js["meshes"][node["mesh"]]["primitives"])):
                fm = prim_of_mesh[(node["mesh"], pi)]
                inst_mesh.append(fm)
                inst_mat.append(meshes[fm][4])
                inst_xf.append(world.reshape(16).copy())
        for c in node.get("children", []):
            walk(c, world)

    ident = np.eye(4, dtype=F32)
    for ni in js["scenes"][js.get("scene", 0)]["nodes"]:
        walk(ni, ident)

    mats = js.get("materials", [])
    M = len(mats)
    base = np.ones((M, 4), F32)
    emis = np.zeros((M, 4), F32)
    emis[:, 3] = 1
    rough = np.ones(M, F32)
    metal = np.ones(M, F32)
    refl = np.full(M, 0.5, F32)
    tex = np.full((M, 5), 0xFFFFFFFF, np.uint32)  # base, emissive, metallic_roughness, normal, occlusion
    tex_srgb = {}
    tex_images = []

    def tex_id(info, srgb):
        if info is None:
            return 0xFFFFFFFF
        t = js["textures"][info["index"]]
        key = (t["source"], srgb)
        if key not in tex_srgb:
            tex_srgb[key] = len(tex_images)
            tex_images.append((t["source"], srgb, t.get("sampler")))
        return tex_srgb[key]

    for i, m in enumerate(mats):
        pbr = m.get("pbrMetallicRoughness", {})
        base[i] = np.array(pbr.get("baseColorFactor", [1, 1, 1, 1]), F32)
        e = m.get("emissiveFactor", [0, 0, 0])
        emis[i] = np.array([e[0], e[1], e[2], 1.0], F32)
        rough[i] = F32(pbr.get("roughnessFactor", 1.0))
        metal[i] = F32(pbr.get("metallicFactor", 1.0))
        tex[i, 0] = tex_id(pbr.get("baseColorTexture"), True)
        tex[i, 1] = tex_id(m.get("emissiveTexture"), True)
        tex[i, 2] = tex_id(pbr.get("metallicRoughnessTexture"), False)
        tex[i, 3] = tex_id(m.get("normalTexture"), False)
        tex[i, 4] = tex_id(m.get("occlusionTexture"), False)

    out["mesh_count"] = np.array(len(meshes), np.uint32)
    for i, (pos, nrm, uv, idx, _) in enumerate(meshes):
        out[f"m{i}_pos"], out[f"m{i}_nrm"], out[f"m{i}_uv"], out[f"m{i}_idx"] = pos, nrm, uv, idx
    out["inst_mesh"] = np.array(inst_mesh, np.uint32)
    out["inst_material"] = np.array(inst_mat, np.uint32)
    out["inst_transform"] = np.array(inst_xf, F32).reshape(-1, 16)
    out["mat_base_color"], out["mat_emissive"] = base, emis
    out["mat_perceptual_roughness"], out["mat_metallic"], out["mat_reflectance"] = rough, metal, refl
    out["mat_textures"] = tex
    out["tex_count"] = np.array(len(tex_images), np.uint32)
    base_dir = os.path.dirname(path)
    for ti, (src, srgb, sampler) in enumerate(tex_images):
        out[f"t{ti}_rgba"] = box_filtered(decode_image(js, bufs, src, base_dir), max_tex)
        smp = js["samplers"][sampler] if sampler is not None and "samplers" in js else {}
        wrap = {10497: 0, 33071: 1, 33648: 2}
        out[f"t{ti}_info"] = np.array([wrap[smp.get("wrapS", 10497)], wrap[smp.get("wrapT", 10497)],
                                       0 if smp.get("magFilter", 9729) == 9728 else 1, 1 if srgb else 0], np.uint32)
    return out


def make_noise():
    from PIL import Image
    planes = []
    for i in range(16):
        im = Image.open(f"{REF}/src/noise/LDR_RGBA_{i}.png")
        a = np.asarray(im.convert("RGBA"), np.uint8)
        assert a.shape == (64, 64, 4), a.shape
        planes.append(a)
    arr = np.stack(planes)
    os.makedirs(f"{ROOT}/data", exist_ok=True)
    arr.tofile(f"{ROOT}/data/noise_rgba8_64x64x16.bin")
    print("noise", arr.shape, arr.mean())


HOUSES = (("house", "Big House.glb"), ("house2", "Big House 2.glb"), ("house3", "Big House 3.glb"))


def house_fixture():
    """tests/golden/gltf_houses.json: what tests/test_gltf_ingest.py needs to rebuild the three house GLBs (5 to 7 MB each, nearly all
    of it PNG) from the shipped scene files: each file's JSON chunk, the SHA-256 of its geometry bytes (every buffer view that is not an
    image), and for each image the scene-file texture that holds it box-filtered, with the PNG's colour mode"""
    import hashlib
    from PIL import Image
    out = {}
    for name, fn in HOUSES:
        js, bufs = load_glb(f"{REF}/assets/models/Low Poly/{fn}")
        z = np.load(f"{ROOT}/scenes/{name}.npz")
        views = js["bufferViews"]
        image_views = {im["bufferView"] for im in js["images"]}
        geometry = b"".join(bufs[0][v.get("byteOffset", 0):v.get("byteOffset", 0) + v["byteLength"]]
                            for i, v in enumerate(views) if i not in image_views)
        texture, mode = [], []
        for i, im in enumerate(js["images"]):
            v = views[im["bufferView"]]
            m = Image.open(io.BytesIO(bufs[0][v.get("byteOffset", 0):v.get("byteOffset", 0) + v["byteLength"]])).mode
            assert m in ("RGB", "RGBA"), (fn, i, m)
            img = box_filtered(decode_image(js, bufs, i, None), 512)
            texture.append(next(t for t in range(int(z["tex_count"])) if np.array_equal(z[f"t{t}_rgba"], img)))
            mode.append(m)
        out[fn] = {"npz": name, "json": js, "geometry_sha256": hashlib.sha256(geometry).hexdigest(), "image_texture": texture,
                   "image_mode": mode}
    with open(f"{ROOT}/tests/golden/gltf_houses.json", "w") as f:
        json.dump(out, f, indent=None, separators=(",", ":"))
        f.write("\n")


def main():
    if "--house-fixture" in sys.argv:
        house_fixture()
        return
    make_noise()
    os.makedirs(f"{ROOT}/scenes", exist_ok=True)
    c = convert_gltf(f"{REF}/assets/models/cornell.glb")
    np.savez_compressed(f"{ROOT}/scenes/cornell.npz", **c)
    print("cornell: meshes", int(c["mesh_count"]), "instances", len(c["inst_mesh"]),
          "tris", sum(len(c[f"m{i}_idx"]) // 3 for i in range(int(c["mesh_count"]))))
    if "--city" in sys.argv:
        from PIL import Image
        earth = Image.open(f"{REF}/assets/models/Earth/earth_daymap.jpg").convert("RGBA").resize((512, 256), Image.BOX)
        np.savez_compressed(f"{ROOT}/scenes/earth.npz", rgba=np.asarray(earth, np.uint8))
        for name, fn in HOUSES:
            h = convert_gltf(f"{REF}/assets/models/Low Poly/{fn}", max_tex=512)
            np.savez_compressed(f"{ROOT}/scenes/{name}.npz", **h)
            print(name, "meshes", int(h["mesh_count"]), "instances", len(h["inst_mesh"]), "textures", int(h["tex_count"]),
                  "tris", sum(len(h[f"m{i}_idx"]) // 3 for i in range(int(h["mesh_count"]))))
    if "--scene" in sys.argv:
        t = convert_gltf(f"{REF}/assets/models/scene.gltf", max_tex=256)
        np.savez_compressed(f"{ROOT}/scenes/town.npz", **t)
        print("town: meshes", int(t["mesh_count"]), "instances", len(t["inst_mesh"]), "materials", len(t["mat_base_color"]),
              "textures", int(t["tex_count"]), "tris", sum(len(t[f"m{i}_idx"]) // 3 for i in range(int(t["mesh_count"]))))


if __name__ == "__main__":
    main()
