"""BASELINE.json configs[3] for the reference arm of bench.py (oracle/ref_bench.py): the matpreview scene rebuilt INSIDE
the unmodified reference from tests/golden/matpreview_scene.npz (the arrays tests/golden/gen_matpreview.py extracted
from resources/data/scenes/matpreview), so that the arm also runs on the GPU box where /root/reference does not exist.
Meshes go through mi.Mesh + write_ply + the `ply` plugin; the envmap through mi.Bitmap. Measurement infrastructure."""
import os
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load_matpreview(mi, width, height, spp, max_depth=8, integrator="path"):
    import drjit as dr
    z = np.load(os.path.join(ROOT, "tests", "golden", "matpreview_scene.npz"), allow_pickle=False)
    envmap = np.load(os.path.join(ROOT, "tests", "golden", "matpreview_envmap.npz"), allow_pickle=False)["envmap"]
    tmp = tempfile.mkdtemp(prefix="matpreview_")

    def ply(sid):
        pos, nrm, uv, faces = z[f"{sid}|positions"], z[f"{sid}|normals"], z[f"{sid}|texcoords"], z[f"{sid}|faces"]
        has_n = bool(z[f"{sid}|has_normals"])
        m = mi.Mesh(sid, mi.TensorXu(faces.astype(np.uint32)), mi.TensorXf(pos), mi.TensorXf(nrm if has_n else np.zeros((0, 3), np.float32)), mi.TensorXf(uv))
        fn = os.path.join(tmp, sid + ".ply")
        m.write_ply(fn)
        return fn

    T4 = mi.ScalarTransform4f
    d = {
        "type": "scene",
        "integrator": {"type": integrator, "max_depth": max_depth},
        "sensor": {"type": "perspective", "fov_axis": "smaller", "fov": float(z["sensor_fov"][0]), "near_clip": float(z["sensor_clip"][0]),
                   "far_clip": float(z["sensor_clip"][1]), "to_world": T4(z["sensor_to_world"].tolist()),
                   "sampler": {"type": "independent", "sample_count": spp},
                   "film": {"type": "hdrfilm", "width": width, "height": height, "pixel_format": "rgb", "rfilter": {"type": "gaussian"}}},
        "emitter-envmap": {"type": "envmap", "bitmap": mi.Bitmap(envmap), "scale": float(z["envmap_scale"]), "to_world": T4(z["envmap_to_world"].tolist())},
        "bsdf-diffuse": {"type": "diffuse", "reflectance": {"type": "rgb", "value": [0.18, 0.18, 0.18]}},
        "bsdf-plane": {"type": "diffuse", "reflectance": {"type": "checkerboard", "color0": {"type": "rgb", "value": [0.4, 0.4, 0.4]},
                                                          "color1": {"type": "rgb", "value": [0.2, 0.2, 0.2]}, "to_uv": mi.ScalarTransform3f().scale([8, 8])}},
        "bsdf-matpreview": {"type": "principled", "base_color": {"type": "rgb", "value": [0.940, 0.271, 0.361]}, "roughness": 0.3, "metallic": 0.0, "specular": 0.5},
    }
    for sid, b in (("shape-plane", "bsdf-plane"), ("shape-matpreview-interior", "bsdf-diffuse"), ("shape-matpreview-exterior", "bsdf-matpreview")):
        d[sid] = {"type": "ply", "filename": ply(sid), "bsdf": {"type": "ref", "id": b}}
    return mi.load_dict(d)
