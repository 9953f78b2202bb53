#!/usr/bin/env python3
"""Extract BASELINE.json configs[3] -- the reference's own asset resources/data/scenes/matpreview (matpreview.xml,
matpreview.serialized, envmap.exr) -- into tests/golden/matpreview_scene.npz, and render small reference images of it.

    python oracle/run_ref.py tests/golden/gen_matpreview.py

The scene is loaded by the UNMODIFIED reference (mi.load_file) with the one change SURVEY.md 8(d) prescribes:
`bsdf-matpreview` (stock: plastic) becomes `principled` (base_color .94/.271/.361, roughness .3, metallic 0,
specular .5), max_depth 8. What is stored: the three meshes as the reference holds them after loading (world-space
positions, normals, texcoords, faces), the envmap as linear float32 RGB (mi.Bitmap), its to_world / scale, the sensor.
mitsuba3_b200.matpreview_scene() rebuilds the scene dictionary from it. Reference renders (llvm_ad_rgb, equal seeds ->
per pixel) go to tests/golden/matpreview_renders.npz.
"""
import os
import re
import sys
import tempfile

import numpy as np

import mitsuba as mi

mi.set_variant("llvm_ad_rgb")
import drjit as dr

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = "/root/reference/resources/data/scenes/matpreview"
PRINCIPLED = '''<bsdf type="principled" id="bsdf-matpreview">
        <rgb name="base_color" value="0.940, 0.271, 0.361" />
        <float name="roughness" value="0.3" />
        <float name="metallic" value="0.0" />
        <float name="specular" value="0.5" />
    </bsdf>'''


def load(width, height, spp, max_depth=8):
    xml = open(os.path.join(SRC, "matpreview.xml")).read()
    xml, n = re.subn(r'<bsdf type="plastic" id="bsdf-matpreview">.*?</bsdf>', PRINCIPLED, xml, flags=re.S)
    assert n == 1
    fr = mi.file_resolver()
    fr.append(SRC)
    with tempfile.NamedTemporaryFile("w", suffix=".xml", delete=False) as f:
        f.write(xml)
    try:
        return mi.load_file(f.name, width=width, height=height, spp=spp, max_depth=max_depth, optimize=False)
    finally:
        os.unlink(f.name)


def main():
    scene = load(64, 64, 16)
    params = mi.traverse(scene)
    out = {}
    for s in scene.shapes():
        sid = s.id()
        pv = np.array(s.packed_vertices(), np.float32).reshape(-1, 8)       # Mesh::packed_vertices: pos3, normal3, uv2
        out[f"{sid}|positions"], out[f"{sid}|normals"], out[f"{sid}|texcoords"] = pv[:, 0:3].copy(), pv[:, 3:6].copy(), pv[:, 6:8].copy()
        out[f"{sid}|faces"] = np.array(s.faces(), np.uint32).reshape(-1, 3)
        out[f"{sid}|has_normals"] = np.array(not s.has_face_normals() and bool(np.any(pv[:, 3:6] != 0)))
        print(sid, out[f"{sid}|positions"].shape, out[f"{sid}|faces"].shape, "normals", out[f"{sid}|normals"].shape, "uv", out[f"{sid}|texcoords"].shape)
    bmp = mi.Bitmap(os.path.join(SRC, "envmap.exr")).convert(mi.Bitmap.PixelFormat.RGB, mi.Struct.Type.Float32, False)
    out["envmap"] = np.array(bmp, np.float32)
    out["envmap_to_world"] = np.array(params["emitter-envmap.to_world"].matrix, np.float32).reshape(4, 4)
    out["envmap_scale"] = np.array(params["emitter-envmap.scale"], np.float32)
    out["sensor_to_world"] = np.array(params["camera.to_world"].matrix, np.float32).reshape(4, 4)
    out["sensor_fov"] = np.array([28.8415], np.float32)
    out["sensor_clip"] = np.array([params["camera.near_clip"], params["camera.far_clip"]], np.float32)
    print("envmap", out["envmap"].shape, out["envmap"].dtype, "x_fov", params["camera.x_fov"])
    # the envmap goes to a file of its own: together with the meshes it would exceed 1 MB
    np.savez_compressed(os.path.join(HERE, "matpreview_envmap.npz"), envmap=out.pop("envmap"))
    np.savez_compressed(os.path.join(HERE, "matpreview_scene.npz"), **out)
    for f in ("matpreview_scene.npz", "matpreview_envmap.npz"):
        print("wrote", f, os.path.getsize(os.path.join(HERE, f)) / 1e6, "MB")
    ren = {}
    for (res, spp, seed) in [(64, 16, 0), (96, 8, 3)]:
        sc = load(res, res, spp)
        ren[f"matpreview_{res}_spp{spp}_seed{seed}"] = np.array(sc.integrator().render(sc, seed=seed, spp=spp), np.float32)
    sc = load(64, 64, 1024)
    ren["matpreview_64_ref1024"] = np.array(sc.integrator().render(sc, seed=9, spp=1024), np.float32)
    np.savez_compressed(os.path.join(HERE, "matpreview_renders.npz"), **ren)


if __name__ == "__main__":
    main()
