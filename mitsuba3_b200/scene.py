"""Host-side scene description: the subset of ``mi.load_dict`` that the hot
path needs (SURVEY.md 8(b): what the plugin extracts from live Mitsuba
objects), and its conversion to the POD ``b200pt_scene_desc``.

Supported plugin types (same property names as the reference):
  scene; integrators ``path`` / ``prb`` (max_depth, rr_depth, hide_emitters);
  sensor ``perspective`` (to_world, fov, fov_axis, near_clip, far_clip) with
  ``hdrfilm`` (width, height, crop_*, rfilter ``gaussian``/``box``) and
  ``independent`` sampler (sample_count, seed); shapes ``rectangle`` / ``cube``
  (src/shapes/rectangle.cpp, cube.cpp) and ``mesh`` (packed arrays, as produced
  by the host's loaders); BSDFs ``diffuse`` / ``conductor`` / ``dielectric`` /
  ``principled`` / ``roughconductor`` / ``roughdielectric`` / ``plastic`` / ``twosided``; emitters ``area`` / ``constant`` / ``envmap``; textures ``rgb`` / float /
  ``bitmap`` (raw float32 data); ``ref``.

Everything else (XML, OBJ/PLY loaders, spectra, other plugins) stays in the
host Mitsuba -- see INTEGRATION.md for the extraction from live objects.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Any

import numpy as np

from . import abi
from .transform import Transform4f, f32, fma, parse_fov, perspective_sample_to_camera, _cross, _normalize, _sqnorm

# include/mitsuba/render/ior.h:24-48
IOR_TABLE = {
    "vacuum": 1.0, "helium": 1.000036, "hydrogen": 1.000132, "air": 1.000277,
    "carbon dioxide": 1.00045, "water": 1.3330, "acetone": 1.36, "ethanol": 1.361,
    "carbon tetrachloride": 1.461, "glycerol": 1.4729, "benzene": 1.501,
    "silicone oil": 1.52045, "bromine": 1.661, "water ice": 1.31, "fused quartz": 1.458,
    "pyrex": 1.470, "acrylic glass": 1.49, "polypropylene": 1.49, "bk7": 1.5046,
    "sodium chloride": 1.544, "amber": 1.55, "pet": 1.5750, "diamond": 2.419,
}


def lookup_ior(v, default):
    v = default if v is None else v
    if isinstance(v, str):
        return float(f32(IOR_TABLE[v.lower()]))
    return float(v)


@dataclass
class TextureData:
    name: str
    kind: int = abi.TEX_CONST
    channels: int = 3
    value: np.ndarray = field(default_factory=lambda: np.zeros(3, f32))
    value1: np.ndarray = field(default_factory=lambda: np.zeros(3, f32))   # checkerboard color1
    data: np.ndarray | None = None           # (H, W, C) float32
    wrap: int = abi.WRAP_REPEAT
    filter: int = abi.FILTER_BILINEAR
    to_uv: np.ndarray = field(default_factory=lambda: np.eye(3, dtype=f32))
    # True / False, or None = "wherever the PRB adjoint has the derivative" (resolved by Scene.build_desc: a texture
    # that sits in a BSDF slot without an implemented derivative is not a gradient target -- asking
    # render_backward for it by name raises instead of returning zeros)
    differentiable: bool | None = None

    @property
    def size(self) -> int:
        if self.kind == abi.TEX_BITMAP:
            return int(self.data.size)
        return self.channels * (2 if self.kind == abi.TEX_CHECKERBOARD else 1)

    def array(self) -> np.ndarray:
        if self.kind == abi.TEX_BITMAP:
            return self.data
        if self.kind == abi.TEX_CHECKERBOARD:      # (2, channels): color0, color1
            return np.stack([self.value[: self.channels], self.value1[: self.channels]])
        return self.value[: self.channels]


@dataclass
class BsdfData:
    id: str
    type: int
    twosided: bool = False
    tex: list = field(default_factory=lambda: [-1] * abi.MAX_SLOTS)
    eta: float = 1.0
    spec_srate: float = 1.0
    clearcoat_srate: float = 1.0
    diff_refl_srate: float = 1.0
    flags: int = 0
    plastic_fdr_int: float = 0.0
    plastic_spec_weight: float = 0.0


@dataclass
class ShapeData:
    id: str
    vertices: np.ndarray      # (V, 8) float32: pos3, normal3, uv2
    faces: np.ndarray         # (F, 4) uint32: v0 v1 v2 flags
    layout: int
    bsdf: int
    emitter: int = -1
    sampling: int = abi.SAMPLING_NONE
    to_world: np.ndarray = field(default_factory=lambda: np.eye(4, dtype=f32))
    frame_n: np.ndarray = field(default_factory=lambda: np.zeros(3, f32))
    inv_area: float = 0.0


@dataclass
class EmitterData:
    shape: int                # area: index of the shape; -1 for the environment emitter
    radiance_tex: int         # area / constant: rgb texture; envmap: bitmap texture with the (H, W, 3) map, real columns
    sampling_weight: float = 1.0
    type: int = abi.EMITTER_AREA
    env_scale: float = 1.0
    env_mis_compensation: bool = False
    to_world: np.ndarray = field(default_factory=lambda: np.eye(4, dtype=f32))
    to_world_inv: np.ndarray = field(default_factory=lambda: np.eye(4, dtype=f32))


@dataclass
class SensorData:
    sample_to_camera: np.ndarray
    to_world: np.ndarray
    near_clip: float
    far_clip: float
    film_size: tuple
    crop_size: tuple
    crop_offset: tuple
    rfilter: int
    rfilter_stddev: float
    base_seed: int
    sample_count: int
    x_fov: float


class Scene:
    """Parsed scene + the parameter map that plays the role of ``mi.traverse``."""

    def __init__(self):
        self.shapes: list[ShapeData] = []
        self.bsdfs: list[BsdfData] = []
        self.textures: list[TextureData] = []
        self.emitters: list[EmitterData] = []
        self.sensor: SensorData | None = None
        self.integrator: dict[str, Any] = {"type": "path", "max_depth": -1, "rr_depth": 5, "hide_emitters": False}
        self._handle = None      # lazily created device scene (mitsuba3_b200.integrators)

    # ---- parameters (mi.traverse analogue) ----------------------------------
    def parameters(self) -> dict[str, int]:
        return {t.name: i for i, t in enumerate(self.textures)}

    @property
    def film_shape(self):
        return (self.sensor.crop_size[1], self.sensor.crop_size[0], 3)

    @property
    def n_triangles(self) -> int:
        return int(sum(s.faces.shape[0] for s in self.shapes))

    # ---- POD descriptor -----------------------------------------------------
    def build_desc(self):
        """Returns (SceneDesc, keepalive) -- keepalive owns every buffer the
        descriptor points to and must outlive the C call."""
        keep = []
        texs = (abi.Texture * max(1, len(self.textures)))()
        uncovered = set()
        for b in self.bsdfs:
            for k, ti in enumerate(b.tex):
                if ti >= 0 and not abi.adjoint_covers_slot(b.type, b.flags, k):
                    uncovered.add(ti)
        for i, t in enumerate(self.textures):
            if t.differentiable is None:
                t.differentiable = i not in uncovered
        for i, t in enumerate(self.textures):
            ct = texs[i]
            ct.kind, ct.channels = t.kind, t.channels
            v = np.zeros(3, f32); v[: t.channels] = np.asarray(t.value, f32)[: t.channels]
            ct.value = (C.c_float * 3)(*v.tolist())
            v1 = np.zeros(3, f32); v1[: t.channels] = np.asarray(t.value1, f32)[: t.channels]
            ct.value1 = (C.c_float * 3)(*v1.tolist())
            if t.kind == abi.TEX_BITMAP:
                d = np.ascontiguousarray(t.data, dtype=f32)
                keep.append(d)
                ct.height, ct.width = d.shape[0], d.shape[1]
                ct.data = d.ctypes.data_as(C.POINTER(C.c_float))
            ct.wrap, ct.filter = t.wrap, t.filter
            ct.to_uv = (C.c_float * 9)(*np.asarray(t.to_uv, f32).reshape(9).tolist())
            ct.differentiable = int(t.differentiable)
        bsdfs = (abi.Bsdf * max(1, len(self.bsdfs)))()
        for i, b in enumerate(self.bsdfs):
            cb = bsdfs[i]
            cb.type, cb.twosided = b.type, int(b.twosided)
            cb.tex = (C.c_int32 * abi.MAX_SLOTS)(*b.tex)
            cb.eta, cb.spec_srate, cb.clearcoat_srate, cb.diff_refl_srate = b.eta, b.spec_srate, b.clearcoat_srate, b.diff_refl_srate
            cb.flags = b.flags
            cb.plastic_fdr_int, cb.plastic_spec_weight = b.plastic_fdr_int, b.plastic_spec_weight
        shapes = (abi.Shape * max(1, len(self.shapes)))()
        for i, s in enumerate(self.shapes):
            cs = shapes[i]
            v = np.ascontiguousarray(s.vertices, dtype=f32); f = np.ascontiguousarray(s.faces, dtype=np.uint32)
            keep += [v, f]
            cs.n_vertices, cs.n_faces = v.shape[0], f.shape[0]
            cs.vertices = v.ctypes.data_as(C.POINTER(C.c_float))
            cs.faces = f.ctypes.data_as(C.POINTER(C.c_uint32))
            cs.layout, cs.bsdf, cs.emitter, cs.sampling = s.layout, s.bsdf, s.emitter, s.sampling
            cs.to_world = (C.c_float * 16)(*np.asarray(s.to_world, f32).reshape(16).tolist())
            cs.frame_n = (C.c_float * 3)(*np.asarray(s.frame_n, f32).tolist())
            cs.inv_area = float(s.inv_area)
        ems = (abi.Emitter * max(1, len(self.emitters)))()
        for i, e in enumerate(self.emitters):
            ems[i].shape, ems[i].radiance_tex, ems[i].sampling_weight = e.shape, e.radiance_tex, e.sampling_weight
            ems[i].type = e.type
            ems[i].to_world = (C.c_float * 16)(*np.asarray(e.to_world, f32).reshape(16).tolist())
            ems[i].to_world_inv = (C.c_float * 16)(*np.asarray(e.to_world_inv, f32).reshape(16).tolist())
            if e.type == abi.EMITTER_ENVMAP:
                ems[i].env_scale, ems[i].env_mis_compensation = float(e.env_scale), int(e.env_mis_compensation)
        d = abi.SceneDesc()
        d.abi_version = abi.ABI_VERSION
        d.n_shapes, d.shapes = len(self.shapes), shapes
        d.n_bsdfs, d.bsdfs = len(self.bsdfs), bsdfs
        d.n_emitters, d.emitters = len(self.emitters), ems
        d.n_textures, d.textures = len(self.textures), texs
        se = self.sensor
        d.sensor.sample_to_camera = (C.c_float * 16)(*np.asarray(se.sample_to_camera, f32).reshape(16).tolist())
        d.sensor.to_world = (C.c_float * 16)(*np.asarray(se.to_world, f32).reshape(16).tolist())
        d.sensor.near_clip, d.sensor.far_clip = se.near_clip, se.far_clip
        d.sensor.film_size = (C.c_uint32 * 2)(*se.film_size)
        d.sensor.crop_size = (C.c_uint32 * 2)(*se.crop_size)
        d.sensor.crop_offset = (C.c_uint32 * 2)(*se.crop_offset)
        d.sensor.rfilter, d.sensor.rfilter_stddev, d.sensor.base_seed = se.rfilter, se.rfilter_stddev, se.base_seed
        keep += [texs, bsdfs, shapes, ems]
        return d, keep


# ---------------------------------------------------------------------------
# dict parser
# ---------------------------------------------------------------------------
_WRAP = {"repeat": abi.WRAP_REPEAT, "mirror": abi.WRAP_MIRROR, "clamp": abi.WRAP_CLAMP}
_FILT = {"bilinear": abi.FILTER_BILINEAR, "nearest": abi.FILTER_NEAREST}


def _as_transform(t) -> Transform4f:
    if t is None:
        return Transform4f()
    if isinstance(t, Transform4f):
        return t
    return Transform4f(np.asarray(t, f32).reshape(4, 4))


_BSDF_TYPES = ("diffuse", "conductor", "roughconductor", "dielectric", "roughdielectric", "plastic", "principled", "twosided")


def fresnel_diffuse_reflectance(eta):
    """fresnel.h:326-360 in fp32 (fmadd chains / Horner as written there)."""
    eta = f32(eta); inv_eta = f32(1) / eta
    approx_1 = fma(f32(0.0636), inv_eta, fma(eta, fma(eta, f32(-1.4399), f32(0.7099)), f32(0.6681)))
    acc = f32(-1.36881)
    for c in (4.98554, -7.80989, 6.75335, -3.4793, 0.919317):
        acc = fma(inv_eta, acc, f32(c))
    return approx_1 if eta < f32(1) else acc


class _Parser:
    def __init__(self):
        self.scene = Scene()
        self.named_bsdfs: dict[str, int] = {}

    # -- textures ------------------------------------------------------------
    def texture(self, name: str, spec, channels: int, default=None) -> int:
        if spec is None:
            if default is None:
                return -1
            spec = default
        t = TextureData(name=name, channels=channels)
        if isinstance(spec, (int, float)):
            t.value = np.full(3, spec, f32); t.name = name + ".value"
        elif isinstance(spec, (list, tuple, np.ndarray)):
            v = np.asarray(spec, f32).reshape(-1)
            t.value = np.full(3, v[0], f32) if v.size == 1 else v[:3].astype(f32)
            t.name = name + ".value"
        elif isinstance(spec, dict):
            ty = spec.get("type")
            if ty == "rgb":
                v = np.asarray(spec["value"], f32).reshape(-1)
                t.value = np.full(3, v[0], f32) if v.size == 1 else v[:3].astype(f32)
                t.name = name + ".value"
            elif ty == "bitmap":
                data = np.asarray(spec["data"], f32)
                if data.ndim == 2:
                    data = data[:, :, None]
                if not spec.get("raw", True):
                    raise NotImplementedError("bitmap textures must be raw float data (sRGB decoding stays in the host)")
                if channels == 3 and data.shape[2] == 1:
                    pass  # luminance broadcast happens at lookup
                t.kind, t.data, t.channels = abi.TEX_BITMAP, np.ascontiguousarray(data), data.shape[2]
                t.wrap = _WRAP[spec.get("wrap_mode", "repeat")]
                t.filter = _FILT[spec.get("filter_type", "bilinear")]
                if "to_uv" in spec:
                    t.to_uv = np.asarray(spec["to_uv"], f32).reshape(3, 3)
                t.name = name + ".data"
            elif ty == "checkerboard":
                def const(c, dflt):
                    c = dflt if c is None else c
                    if isinstance(c, dict):
                        if c.get("type") != "rgb":
                            raise NotImplementedError("checkerboard colours must be constants")
                        c = c["value"]
                    c = np.asarray(c, f32).reshape(-1)
                    return np.full(3, c[0], f32) if c.size == 1 else c[:3].astype(f32)
                t.kind = abi.TEX_CHECKERBOARD
                t.value, t.value1 = const(spec.get("color0"), 0.4), const(spec.get("color1"), 0.2)
                if "to_uv" in spec:
                    t.to_uv = np.asarray(getattr(spec["to_uv"], "matrix", spec["to_uv"]), f32).reshape(3, 3)
                t.name = name + ".colors"       # (2, channels): color0, color1
            else:
                raise NotImplementedError(f"texture type {ty!r} is outside the hot-path scope")
        else:
            raise TypeError(f"cannot interpret texture {spec!r}")
        self.scene.textures.append(t)
        return len(self.scene.textures) - 1

    # -- bsdfs ---------------------------------------------------------------
    def bsdf(self, bid: str, d: dict, twosided=False) -> int:
        ty = d["type"]
        if ty == "ref":
            return self.named_bsdfs[d["id"]]
        if ty == "twosided":
            inner = d.get("bsdf") or next(v for k, v in d.items() if isinstance(v, dict) and k != "type")
            return self.bsdf(bid, inner, twosided=True)
        b = BsdfData(id=bid, type=-1, twosided=twosided)
        if ty == "diffuse":
            b.type = abi.BSDF_DIFFUSE
            b.tex[abi.SLOT_REFLECTANCE] = self.texture(f"{bid}.reflectance", d.get("reflectance"), 3, 0.5)
        elif ty in ("conductor", "roughconductor"):
            b.type = abi.BSDF_CONDUCTOR
            mat = d.get("material")
            if mat not in (None, "none") and ("eta" not in d):
                raise NotImplementedError("conductor `material` presets need the host's spectral data; pass rgb eta/k")
            eta, k = (d.get("eta", 0.0), d.get("k", 1.0))
            b.tex[abi.SLOT_ETA] = self.texture(f"{bid}.eta", eta, 3)
            b.tex[abi.SLOT_K] = self.texture(f"{bid}.k", k, 3)
            if ty == "roughconductor":
                # roughconductor.cpp:172-205: specular_reflectance only if given
                b.tex[abi.SLOT_SPEC_REFL] = self.texture(f"{bid}.specular_reflectance", d.get("specular_reflectance"), 3)
                self._microfacet(b, bid, d, abi.SLOT_ALPHA_U, abi.SLOT_ALPHA_V)
            else:
                b.tex[abi.SLOT_SPEC_REFL] = self.texture(f"{bid}.specular_reflectance", d.get("specular_reflectance"), 3, 1.0)
        elif ty in ("dielectric", "roughdielectric"):
            b.type = abi.BSDF_DIELECTRIC
            if ty == "roughdielectric":
                self._microfacet(b, bid, d, abi.SLOT_D_ALPHA_U, abi.SLOT_D_ALPHA_V)
            b.eta = float(f32(f32(lookup_ior(d.get("int_ior"), "bk7")) / f32(lookup_ior(d.get("ext_ior"), "air"))))
            b.tex[abi.SLOT_D_SPEC_REFL] = self.texture(f"{bid}.specular_reflectance", d.get("specular_reflectance"), 3)
            b.tex[abi.SLOT_D_SPEC_TRANS] = self.texture(f"{bid}.specular_transmittance", d.get("specular_transmittance"), 3)
        elif ty == "plastic":
            # plastic.cpp:156-208
            b.type = abi.BSDF_PLASTIC
            b.eta = float(f32(f32(lookup_ior(d.get("int_ior"), "polypropylene")) / f32(lookup_ior(d.get("ext_ior"), "air"))))
            b.tex[abi.SLOT_PL_DIFFUSE] = self.texture(f"{bid}.diffuse_reflectance", d.get("diffuse_reflectance"), 3, 0.5)
            b.tex[abi.SLOT_PL_SPEC_REFL] = self.texture(f"{bid}.specular_reflectance", d.get("specular_reflectance"), 3)
            if bool(d.get("nonlinear", False)):
                b.flags |= abi.M_NONLINEAR
            b.plastic_fdr_int = float(fresnel_diffuse_reflectance(f32(1) / f32(b.eta)))
            def mean(ti):      # Texture::mean (srgb.cpp:117-122; bitmap: average of all texels)
                t = self.scene.textures[ti]
                return f32(np.mean(t.data, dtype=np.float64)) if t.kind == abi.TEX_BITMAP else f32((f32(t.value[0]) + f32(t.value[1]) + f32(t.value[2])) / f32(3))
            if self.scene.textures[b.tex[abi.SLOT_PL_DIFFUSE]].kind == abi.TEX_CHECKERBOARD:
                raise NotImplementedError("plastic with a checkerboard reflectance: Texture::mean() of checkerboard is not restated")
            d_mean = mean(b.tex[abi.SLOT_PL_DIFFUSE])
            s_mean = mean(b.tex[abi.SLOT_PL_SPEC_REFL]) if b.tex[abi.SLOT_PL_SPEC_REFL] >= 0 else f32(1)
            b.plastic_spec_weight = float(f32(s_mean / f32(d_mean + s_mean)))
        elif ty == "principled":
            self._principled(b, bid, d)
        else:
            raise NotImplementedError(f"BSDF {ty!r} is outside the hot-path scope (SURVEY.md 8(a))")
        self.scene.bsdfs.append(b)
        return len(self.scene.bsdfs) - 1

    def _microfacet(self, b: BsdfData, bid: str, d: dict, slot_u: int, slot_v: int):
        """Microfacet parameters shared by roughconductor / roughdielectric (roughconductor.cpp:172-200,
        roughdielectric.cpp:190-225): `distribution` beckmann (default) | ggx, `alpha` or `alpha_u`+`alpha_v`."""
        distr = d.get("distribution", "beckmann")
        if distr not in ("beckmann", "ggx"):
            raise ValueError(f'Specified an invalid distribution "{distr}", must be "beckmann" or "ggx"!')
        if not bool(d.get("sample_visible", True)):
            raise NotImplementedError("sample_visible=false is outside the hot-path scope")
        b.flags |= abi.M_ROUGH | (abi.M_GGX if distr == "ggx" else 0)
        if "alpha_u" in d or "alpha_v" in d:
            if "alpha_u" not in d or "alpha_v" not in d:
                raise ValueError("Microfacet model: both 'alpha_u' and 'alpha_v' must be specified.")
            if "alpha" in d:
                raise ValueError("Microfacet model: please specify either 'alpha' or 'alpha_u'/'alpha_v'.")
            b.tex[slot_u] = self.texture(f"{bid}.alpha_u", d["alpha_u"], 1)
            b.tex[slot_v] = self.texture(f"{bid}.alpha_v", d["alpha_v"], 1)
        else:
            b.tex[slot_u] = b.tex[slot_v] = self.texture(f"{bid}.alpha", d.get("alpha"), 1, 0.1)

    def _principled(self, b: BsdfData, bid: str, d: dict):
        # principled.cpp:190-330 constructor
        b.type = abi.BSDF_PRINCIPLED
        def has(k): return k in d
        def active(k, dflt):
            # principledhelpers.h:122-132 get_flag: absent -> False; constant 0 -> False
            if k not in d:
                return False
            v = d[k]
            if isinstance(v, (int, float)):
                return float(v) != 0.0
            return True
        b.tex[abi.SLOT_P_BASE_COLOR] = self.texture(f"{bid}.base_color", d.get("base_color"), 3, 0.5)
        b.tex[abi.SLOT_P_ROUGHNESS] = self.texture(f"{bid}.roughness", d.get("roughness"), 1, 0.5)
        flags = 0
        if active("anisotropic", 0.0): flags |= abi.P_HAS_ANISOTROPIC
        if active("spec_trans", 0.0): flags |= abi.P_HAS_SPEC_TRANS
        if active("sheen", 0.0): flags |= abi.P_HAS_SHEEN
        if active("sheen_tint", 0.0): flags |= abi.P_HAS_SHEEN_TINT
        if active("flatness", 0.0): flags |= abi.P_HAS_FLATNESS
        if active("spec_tint", 0.0): flags |= abi.P_HAS_SPEC_TINT
        if active("metallic", 0.0): flags |= abi.P_HAS_METALLIC
        if active("clearcoat", 0.0): flags |= abi.P_HAS_CLEARCOAT
        b.tex[abi.SLOT_P_ANISOTROPIC] = self.texture(f"{bid}.anisotropic", d.get("anisotropic"), 1, 0.0)
        b.tex[abi.SLOT_P_SPEC_TRANS] = self.texture(f"{bid}.spec_trans", d.get("spec_trans"), 1, 0.0)
        b.tex[abi.SLOT_P_SHEEN] = self.texture(f"{bid}.sheen", d.get("sheen"), 1, 0.0)
        b.tex[abi.SLOT_P_SHEEN_TINT] = self.texture(f"{bid}.sheen_tint", d.get("sheen_tint"), 1, 0.0)
        b.tex[abi.SLOT_P_FLATNESS] = self.texture(f"{bid}.flatness", d.get("flatness"), 1, 0.0)
        b.tex[abi.SLOT_P_SPEC_TINT] = self.texture(f"{bid}.spec_tint", d.get("spec_tint"), 1, 0.0)
        b.tex[abi.SLOT_P_METALLIC] = self.texture(f"{bid}.metallic", d.get("metallic"), 1, 0.0)
        b.tex[abi.SLOT_P_CLEARCOAT] = self.texture(f"{bid}.clearcoat", d.get("clearcoat"), 1, 0.0)
        b.tex[abi.SLOT_P_CLEARCOAT_GLOSS] = self.texture(f"{bid}.clearcoat_gloss", d.get("clearcoat_gloss"), 1, 0.0)
        if has("eta") and has("specular"):
            raise ValueError("Specified an invalid index of refraction property \"eta\", either use \"eta\" or \"specular\" !")
        has_st = bool(flags & abi.P_HAS_SPEC_TRANS)
        if has("eta"):
            flags |= abi.P_ETA_SPECULAR
            eta = f32(d["eta"])
            if has_st and eta == f32(1):            # principled.cpp:221: eta = 1 is not plausible for transmission
                eta = f32(1.001)
            b.eta = float(eta)
        else:
            spec = f32(d.get("specular", 0.5))
            if has_st and spec == f32(0):           # principled.cpp:226
                spec = f32(1e-3)
            # principled.cpp:227: eta = 2 * rcp(1 - sqrt(0.08 * specular)) - 1 (fp32)
            b.eta = float(f32(2) * (f32(1) / (f32(1) - np.sqrt(f32(0.08) * spec, dtype=f32))) - f32(1))
        b.tex[abi.SLOT_P_SPECULAR] = -1
        b.spec_srate = float(d.get("main_specular_sampling_rate", 1.0))
        b.clearcoat_srate = float(d.get("clearcoat_sampling_rate", 1.0))
        b.diff_refl_srate = float(d.get("diffuse_reflectance_sampling_rate", 1.0))
        b.flags = flags

    # -- shapes --------------------------------------------------------------
    def shape(self, sid: str, d: dict):
        ty = d["type"]
        bs = d.get("bsdf")
        if bs is None:
            for k, v in d.items():
                if isinstance(v, dict) and v.get("type") in _BSDF_TYPES + ("ref",) and k != "emitter":
                    bs = v
                    break
        if bs is None:
            bs = {"type": "diffuse"}     # Shape default BSDF (shape.cpp: diffuse 0.5)
        bidx = self.bsdf(f"{sid}.bsdf", bs)
        bd = self.scene.bsdfs[bidx]
        aniso = (bd.type == abi.BSDF_PRINCIPLED and bd.flags & abi.P_HAS_ANISOTROPIC) or \
                (bd.type == abi.BSDF_CONDUCTOR and bd.flags & abi.M_ROUGH and bd.tex[abi.SLOT_ALPHA_U] != bd.tex[abi.SLOT_ALPHA_V]) or \
                (bd.type == abi.BSDF_DIELECTRIC and bd.flags & abi.M_ROUGH and bd.tex[abi.SLOT_D_ALPHA_U] != bd.tex[abi.SLOT_D_ALPHA_V])
        to_world = _as_transform(d.get("to_world"))
        flip = bool(d.get("flip_normals", False))
        if ty == "rectangle":
            sh = make_rectangle(sid, to_world, flip, bidx)
        elif ty == "cube":
            sh = make_cube(sid, to_world, flip, bidx)
        elif ty == "mesh":
            sh = make_mesh(sid, d, to_world, bidx)
        else:
            raise NotImplementedError(f"shape {ty!r}: only triangle meshes are on the hot path; "
                                      "load it with the host Mitsuba and pass the packed records as type 'mesh'")
        if aniso and not (sh.layout & abi.LAYOUT_TANGENTS):
            # BSDFFlags::Anisotropic makes the reference's meshes pack per-vertex tangent frames (mesh.cpp:355,2417-2429,
            # interaction.h:570-598). Generating them is the host loaders' job (mesh.cpp:600-700); this mirror takes them
            # ready-made: `packed_vertices` whose frame slot holds frame_encode(n, s), `faces` (F, 4) with the FaceUVFlipped
            # bit and `layout` including LAYOUT_TANGENTS -- what mitsuba_plugin.extract_scene reads off a live mesh.
            raise NotImplementedError("anisotropic BSDFs need a mesh with packed tangent frames (packed_vertices + layout with LAYOUT_TANGENTS)")
        em = d.get("emitter")
        if em is not None:
            if em["type"] != "area":
                raise NotImplementedError("only `area` emitters are on the hot path")
            rad = self.texture(f"{sid}.emitter.radiance", em.get("radiance"), 3, 1.0)
            if self.scene.textures[rad].kind != abi.TEX_CONST:
                raise NotImplementedError("spatially varying area-light radiance is outside the hot path")
            self.scene.emitters.append(EmitterData(shape=len(self.scene.shapes), radiance_tex=rad,
                                                   sampling_weight=float(em.get("sampling_weight", 1.0))))
            sh.emitter = len(self.scene.emitters) - 1
            if sh.sampling == abi.SAMPLING_NONE:
                sh.sampling = abi.SAMPLING_MESH
        elif sh.sampling == abi.SAMPLING_RECTANGLE:
            pass
        self.scene.shapes.append(sh)

    # -- environment emitters ------------------------------------------------
    def environment(self, eid: str, d: dict):
        """``constant`` (constant.cpp:60-74) and ``envmap`` (envmap.cpp:107-200). The map is passed
        as a float32 array under ``bitmap`` / ``data`` (H x W x 3, linear RGB, real columns) or as a
        ``.npy`` ``filename``; image decoding stays in the host."""
        if any(e.type != abi.EMITTER_AREA for e in self.scene.emitters):
            raise ValueError("Only one environment emitter can be specified per scene.")      # scene.cpp:64
        tw = _as_transform(d.get("to_world"))
        inv = np.ascontiguousarray(tw.inverse_transpose.T, dtype=f32)
        if d["type"] == "constant":
            rad = self.texture(f"{eid}.radiance", d.get("radiance"), 3, 1.0)
            if self.scene.textures[rad].kind != abi.TEX_CONST:
                raise ValueError("Expected a non-spatially varying radiance spectra!")        # constant.cpp:64
            self.scene.emitters.append(EmitterData(shape=-1, radiance_tex=rad, type=abi.EMITTER_CONSTANT,
                                                   sampling_weight=float(d.get("sampling_weight", 1.0))))
            return
        data = d.get("bitmap", d.get("data"))
        if data is None and str(d.get("filename", "")).endswith(".npy"):
            data = np.load(d["filename"])
        if data is None:
            raise NotImplementedError("envmap: pass the decoded image as a float32 array under `bitmap` (or a .npy `filename`)")
        data = np.asarray(data, dtype=f32)
        if data.ndim == 2:
            data = np.repeat(data[..., None], 3, axis=2)
        if data.ndim != 3 or data.shape[2] < 3:
            raise ValueError("envmap: expected an (H, W, 3) array")
        data = np.ascontiguousarray(data[..., :3])
        # Bitmap::pad_to(2, 3) (envmap.cpp:141): replicate the last column / row
        if data.shape[1] < 2:
            data = np.concatenate([data, np.repeat(data[:, -1:, :], 2 - data.shape[1], axis=1)], axis=1)
        if data.shape[0] < 3:
            data = np.concatenate([data, np.repeat(data[-1:, :, :], 3 - data.shape[0], axis=0)], axis=0)
        t = TextureData(name=f"{eid}.data", channels=3)
        t.kind, t.data = abi.TEX_BITMAP, data
        t.wrap, t.filter = abi.WRAP_CLAMP, abi.FILTER_BILINEAR      # ignored for the environment map
        self.scene.textures.append(t)
        self.scene.emitters.append(EmitterData(
            shape=-1, radiance_tex=len(self.scene.textures) - 1, type=abi.EMITTER_ENVMAP, env_scale=float(d.get("scale", 1.0)),
            env_mis_compensation=bool(d.get("mis_compensation", False)), to_world=tw.matrix.copy(), to_world_inv=inv,
            sampling_weight=float(d.get("sampling_weight", 1.0))))

    # -- sensor --------------------------------------------------------------
    def sensor(self, d: dict):
        if d["type"] != "perspective":
            raise NotImplementedError("only the `perspective` sensor is on the hot path")
        film = d.get("film", {"type": "hdrfilm"})
        w, h = int(film.get("width", 768)), int(film.get("height", 576))
        cw, ch = int(film.get("crop_width", w)), int(film.get("crop_height", h))
        cx, cy = int(film.get("crop_offset_x", 0)), int(film.get("crop_offset_y", 0))
        if film.get("sample_border", False):
            raise NotImplementedError("sample_border is outside the hot-path scope")
        rf = film.get("rfilter", {"type": "gaussian"})
        if rf["type"] == "box":
            rfilter, stddev = abi.RFILTER_BOX, 0.0
        elif rf["type"] == "gaussian":
            rfilter, stddev = abi.RFILTER_GAUSSIAN, float(rf.get("stddev", 0.5))
        else:
            raise NotImplementedError(f"rfilter {rf['type']!r} is outside the hot-path scope")
        sampler = d.get("sampler", {"type": "independent"})
        if sampler.get("type", "independent") != "independent":
            raise NotImplementedError("only the `independent` sampler is on the hot path")
        to_world = _as_transform(d.get("to_world"))
        near, far = float(d.get("near_clip", 1e-2)), float(d.get("far_clip", 1e4))
        fov = float(d.get("fov", 0.0)) if "fov" in d else None
        if fov is None:
            raise NotImplementedError("specify `fov` (focal_length parsing stays in the host)")
        x_fov = float(f32(parse_fov(fov, d.get("fov_axis", "x"), w / h)))
        s2c = perspective_sample_to_camera((w, h), (cw, ch), (cx, cy), x_fov, f32(near), f32(far))
        self.scene.sensor = SensorData(
            sample_to_camera=s2c, to_world=to_world.matrix.copy(), near_clip=float(f32(near)), far_clip=float(f32(far)),
            film_size=(w, h), crop_size=(cw, ch), crop_offset=(cx, cy), rfilter=rfilter, rfilter_stddev=stddev,
            base_seed=int(sampler.get("seed", 0)), sample_count=int(sampler.get("sample_count", 4)), x_fov=x_fov)

    def parse(self, d: dict) -> Scene:
        if d.get("type") != "scene":
            raise ValueError("top-level dictionary must have type 'scene'")
        # first pass: named BSDFs (so that refs resolve irrespective of order)
        for k, v in d.items():
            if isinstance(v, dict) and v.get("type") in _BSDF_TYPES:
                self.named_bsdfs[k] = self.bsdf(k, v)
        for k, v in d.items():
            if not isinstance(v, dict):
                continue
            ty = v.get("type")
            if ty in ("path", "prb", "b200_path", "b200_prb"):
                self.scene.integrator = {"type": "prb" if "prb" in ty else "path",
                                         "max_depth": int(v.get("max_depth", 6 if "prb" in ty else -1)),
                                         "rr_depth": int(v.get("rr_depth", 5)),
                                         "hide_emitters": bool(v.get("hide_emitters", False))}
            elif ty == "perspective":
                self.sensor(v)
            elif ty in ("rectangle", "cube", "mesh"):
                self.shape(k, v)
            elif ty in ("constant", "envmap"):
                self.environment(k, v)
            elif ty in _BSDF_TYPES:
                pass
            else:
                raise NotImplementedError(f"plugin type {ty!r} is outside the hot-path scope (SURVEY.md 8)")
        if self.scene.sensor is None:
            raise ValueError("scene has no sensor")
        return self.scene


def load_dict(d: dict) -> Scene:
    """Counterpart of ``mi.load_dict`` for the hot-path subset."""
    return _Parser().parse(d)


# ---------------------------------------------------------------------------
# shape construction (mirrors rectangle.cpp:110-153, cube.cpp:61-113,
# mesh_utils.cpp:103-133, mesh.cpp:1160-1200)
# ---------------------------------------------------------------------------
def _pack(positions, normals, uvs, to_world: Transform4f):
    n = len(positions)
    v = np.zeros((n, 8), f32)
    for i in range(n):
        v[i, 0:3] = to_world.point(positions[i])
        nn = to_world.normal(normals[i])
        il = f32(1) / np.sqrt(_sqnorm(nn), dtype=f32)
        v[i, 3:6] = nn * (il if np.isfinite(il) else f32(1))
        v[i, 6:8] = uvs[i]
    return v


def make_rectangle(sid, to_world: Transform4f, flip: bool, bsdf: int) -> ShapeData:
    tw = to_world
    if flip:
        tw = tw @ Transform4f().scale([1, 1, -1])
    pos = [[-1, -1, 0], [1, -1, 0], [-1, 1, 0], [1, 1, 0]]
    nrm = [[0, 0, 1]] * 4
    uv = [[0, 0], [1, 0], [0, 1], [1, 1]]
    faces = np.array([[1, 2, 0, 0], [1, 3, 2, 0]], np.uint32)
    verts = _pack(pos, nrm, uv, tw)
    if tw.det3() < 0:
        faces = faces[:, [2, 1, 0, 3]].copy()
    n = _normalize(tw.normal([0, 0, 1]))
    dp_du, dp_dv = tw.vector([2, 0, 0]), tw.vector([0, 2, 0])
    area = np.sqrt(_sqnorm(_cross(dp_du, dp_dv)), dtype=f32)
    # NOTE rectangle.cpp:159-166 samples with m_to_world (the un-flipped transform)
    return ShapeData(id=sid, vertices=verts, faces=faces, layout=abi.LAYOUT_NORMALS | abi.LAYOUT_TEXCOORDS,
                     bsdf=bsdf, sampling=abi.SAMPLING_RECTANGLE, to_world=to_world.matrix.copy(),
                     frame_n=n.astype(f32), inv_area=float(f32(1) / area))


def make_cube(sid, to_world: Transform4f, flip: bool, bsdf: int) -> ShapeData:
    side_normals = [[0, -1, 0], [0, 1, 0], [1, 0, 0], [0, 0, 1], [-1, 0, 0], [0, 0, -1]]
    side_uv = [[0, 1], [1, 1], [1, 0], [0, 0]]
    position_index = [1, 5, 4, 0, 3, 2, 6, 7, 1, 3, 7, 5, 5, 7, 6, 4, 4, 6, 2, 0, 3, 1, 0, 2]
    corners = [[1.0 if c & 1 else -1.0, 1.0 if c & 2 else -1.0, 1.0 if c & 4 else -1.0] for c in range(8)]
    pos, nrm, uv, faces = [], [], [], []
    for s in range(6):
        v = 4 * s
        for k in range(4):
            pos.append(corners[position_index[v + k]]); nrm.append(side_normals[s]); uv.append(side_uv[k])
        faces += [[v, v + 1, v + 2, 0], [v + 3, v, v + 2, 0]]
    verts = _pack(pos, nrm, uv, to_world)
    faces = np.array(faces, np.uint32)
    mirrored = to_world.det3() < 0
    if flip:
        verts[:, 3:6] = -verts[:, 3:6]
    if mirrored != flip:
        faces = faces[:, [2, 1, 0, 3]].copy()
    return ShapeData(id=sid, vertices=verts, faces=faces, layout=abi.LAYOUT_NORMALS | abi.LAYOUT_TEXCOORDS, bsdf=bsdf)


def make_mesh(sid, d: dict, to_world: Transform4f, bsdf: int) -> ShapeData:
    """Triangle mesh from arrays. Either ``packed_vertices`` (V,8) + ``faces``
    (F,3|4) in world space (what the host's loaders hold, mesh_utils.h:19-46),
    or ``positions`` (+ optional ``normals``, ``texcoords``) + ``faces``."""
    faces = np.asarray(d["faces"], np.uint32)
    if faces.shape[1] == 3:
        faces = np.concatenate([faces, np.zeros((faces.shape[0], 1), np.uint32)], axis=1)
    if "packed_vertices" in d:
        verts = np.asarray(d["packed_vertices"], f32).reshape(-1, 8)
        layout = int(d.get("layout", abi.LAYOUT_NORMALS | abi.LAYOUT_TEXCOORDS))
    else:
        pos = np.asarray(d["positions"], f32).reshape(-1, 3)
        verts = np.zeros((pos.shape[0], 8), f32)
        layout = 0
        m = to_world.matrix.astype(np.float64)
        verts[:, 0:3] = (pos.astype(np.float64) @ m[:3, :3].T + m[:3, 3]).astype(f32)
        if d.get("normals") is not None:
            nr = np.asarray(d["normals"], f32).reshape(-1, 3).astype(np.float64) @ to_world.inverse_transpose[:3, :3].astype(np.float64).T
            nr /= np.maximum(np.linalg.norm(nr, axis=1, keepdims=True), 1e-30)
            verts[:, 3:6] = nr.astype(f32); layout |= abi.LAYOUT_NORMALS
        if d.get("texcoords") is not None:
            verts[:, 6:8] = np.asarray(d["texcoords"], f32).reshape(-1, 2); layout |= abi.LAYOUT_TEXCOORDS
        if to_world.det3() < 0:
            faces = faces[:, [2, 1, 0, 3]].copy()
    return ShapeData(id=sid, vertices=verts, faces=faces, layout=layout, bsdf=bsdf)


# ---------------------------------------------------------------------------
# mi.cornell_box() (src/python/python/util.py:569-703)
# ---------------------------------------------------------------------------
def cornell_box() -> dict:
    T = Transform4f
    white = {"type": "ref", "id": "white"}
    return {
        "type": "scene",
        "integrator": {"type": "path", "max_depth": 8},
        "sensor": {
            "type": "perspective", "fov_axis": "smaller", "near_clip": 0.001, "far_clip": 100.0,
            "focus_distance": 1000, "fov": 39.3077,
            "to_world": T().look_at(origin=[0, 0, 3.90], target=[0, 0, 0], up=[0, 1, 0]),
            "sampler": {"type": "independent", "sample_count": 64},
            "film": {"type": "hdrfilm", "width": 256, "height": 256, "rfilter": {"type": "gaussian"},
                     "pixel_format": "rgb", "component_format": "float32"},
        },
        "white": {"type": "diffuse", "reflectance": {"type": "rgb", "value": [0.885809, 0.698859, 0.666422]}},
        "green": {"type": "diffuse", "reflectance": {"type": "rgb", "value": [0.105421, 0.37798, 0.076425]}},
        "red": {"type": "diffuse", "reflectance": {"type": "rgb", "value": [0.570068, 0.0430135, 0.0443706]}},
        "light": {"type": "rectangle",
                  "to_world": T().translate([0.0, 0.99, 0.01]).rotate([1, 0, 0], 90).scale([0.23, 0.19, 0.19]),
                  "bsdf": white,
                  "emitter": {"type": "area", "radiance": {"type": "rgb", "value": [18.387, 13.9873, 6.75357]}}},
        "floor": {"type": "rectangle", "to_world": T().translate([0.0, -1.0, 0.0]).rotate([1, 0, 0], -90), "bsdf": white},
        "ceiling": {"type": "rectangle", "to_world": T().translate([0.0, 1.0, 0.0]).rotate([1, 0, 0], 90), "bsdf": white},
        "back": {"type": "rectangle", "to_world": T().translate([0.0, 0.0, -1.0]), "bsdf": white},
        "green-wall": {"type": "rectangle", "to_world": T().translate([1.0, 0.0, 0.0]).rotate([0, 1, 0], -90),
                       "bsdf": {"type": "ref", "id": "green"}},
        "red-wall": {"type": "rectangle", "to_world": T().translate([-1.0, 0.0, 0.0]).rotate([0, 1, 0], 90),
                     "bsdf": {"type": "ref", "id": "red"}},
        "small-box": {"type": "cube", "to_world": T().translate([0.335, -0.7, 0.38]).rotate([0, 1, 0], -17).scale(0.3), "bsdf": white},
        "large-box": {"type": "cube", "to_world": T().translate([-0.33, -0.4, -0.28]).rotate([0, 1, 0], 18.25).scale([0.3, 0.61, 0.3]), "bsdf": white},
    }


# ---------------------------------------------------------------------------
# synthetic stand-ins for the larger BASELINE.json configs (no external assets)
# ---------------------------------------------------------------------------
def heightfield_mesh(n: int, amplitude: float = 0.08, y0: float = -1.0, extent: float = 1.0, freq: float = 5.0):
    """(n x n quads = 2 n^2 triangles) bumpy floor over [-extent, extent]^2 at height y0,
    with analytic smooth normals and uv -- a triangle-count knob for BVH tests/benchmarks."""
    g = np.linspace(-extent, extent, n + 1, dtype=np.float64)
    x, z = np.meshgrid(g, g, indexing="xy")
    h = amplitude * (np.sin(freq * x) * np.cos(freq * z) + 0.5 * np.sin(2.3 * freq * x + 1.0) * np.sin(1.7 * freq * z))
    y = y0 + h
    dhdx = amplitude * (freq * np.cos(freq * x) * np.cos(freq * z) + 0.5 * 2.3 * freq * np.cos(2.3 * freq * x + 1.0) * np.sin(1.7 * freq * z))
    dhdz = amplitude * (-freq * np.sin(freq * x) * np.sin(freq * z) + 0.5 * 1.7 * freq * np.sin(2.3 * freq * x + 1.0) * np.cos(1.7 * freq * z))
    nrm = np.stack([-dhdx, np.ones_like(h), -dhdz], axis=-1)
    nrm /= np.linalg.norm(nrm, axis=-1, keepdims=True)
    pos = np.stack([x, y, z], axis=-1).reshape(-1, 3).astype(f32)
    uv = np.stack([(x + extent) / (2 * extent), (z + extent) / (2 * extent)], axis=-1).reshape(-1, 2).astype(f32)
    idx = np.arange((n + 1) * (n + 1)).reshape(n + 1, n + 1)
    a, b, c, d = idx[:-1, :-1].ravel(), idx[:-1, 1:].ravel(), idx[1:, :-1].ravel(), idx[1:, 1:].ravel()
    # winding such that the geometric normal points up (+y)
    faces = np.concatenate([np.stack([a, c, b], axis=1), np.stack([b, c, d], axis=1)], axis=0).astype(np.uint32)
    return {"type": "mesh", "positions": pos, "normals": nrm.reshape(-1, 3).astype(f32), "texcoords": uv, "faces": faces}


def cornell_box_heightfield(n: int = 64, **kw) -> dict:
    """Cornell box whose floor is an (2 n^2)-triangle heightfield (n = 320 -> 204 800 triangles:
    the documented synthetic stand-in for BASELINE.json's 200k-triangle config)."""
    d = cornell_box()
    hf = heightfield_mesh(n, **kw)
    hf["bsdf"] = {"type": "ref", "id": "white"}
    del d["floor"]
    d["floor"] = hf
    return d


# ---------------------------------------------------------------------------
# Synthetic scene of the flavour of BASELINE.json configs[3] (principled BSDF + envmap), used by unit tests; the
# reference's real matpreview asset is loaded by matpreview_scene() further down.
# ---------------------------------------------------------------------------
def uv_sphere_mesh(n_theta: int = 128, n_phi: int = 256, radius: float = 1.0, center=(0.0, 0.0, 0.0)) -> dict:
    """Latitude-longitude sphere with smooth normals and texture coordinates:
    2 * n_phi * (n_theta - 1) triangles."""
    th = (np.arange(n_theta + 1, dtype=np.float64) / n_theta) * np.pi
    ph = (np.arange(n_phi + 1, dtype=np.float64) / n_phi) * 2 * np.pi
    T, P = np.meshgrid(th, ph, indexing="ij")
    nrm = np.stack([np.sin(T) * np.cos(P), np.cos(T), np.sin(T) * np.sin(P)], -1).reshape(-1, 3)
    pos = nrm * radius + np.asarray(center, np.float64)
    uv = np.stack([P / (2 * np.pi), T / np.pi], -1).reshape(-1, 2)
    idx = lambda i, j: i * (n_phi + 1) + j
    faces = []
    for i in range(n_theta):
        j = np.arange(n_phi)
        a, b, c, d = idx(i, j), idx(i + 1, j), idx(i + 1, j + 1), idx(i, j + 1)
        if i > 0:
            faces.append(np.stack([a, d, c], -1))      # counter-clockwise seen from outside
        if i < n_theta - 1:
            faces.append(np.stack([a, c, b], -1))
    return {"type": "mesh", "positions": pos.astype(f32), "normals": nrm.astype(f32), "texcoords": uv.astype(f32),
            "faces": np.concatenate(faces, 0).astype(np.uint32)}


def synthetic_sky(width: int = 1024, height: int = 512) -> np.ndarray:
    """Procedural lat-long HDR sky (float32 RGB): horizon gradient, a bright sun, soft 'clouds', dark ground."""
    y, x = np.meshgrid((np.arange(height) + 0.5) / height, (np.arange(width) + 0.5) / width, indexing="ij")
    up = np.clip(1 - 2 * y, 0, 1)
    sky = np.stack([0.25 + 0.35 * (1 - up), 0.35 + 0.4 * (1 - up), 0.6 + 0.35 * up], -1)
    clouds = 0.5 + 0.5 * np.sin(18 * x + 3 * np.sin(9 * y)) * np.sin(14 * y + 2 * np.cos(11 * x))
    sky = sky * (0.8 + 0.5 * (clouds * up)[..., None])
    ground = np.array([0.12, 0.1, 0.08]) * (0.6 + 0.4 * clouds)[..., None]
    img = np.where((y < 0.5)[..., None], sky, ground)
    dx = np.minimum(np.abs(x - 0.62), 1 - np.abs(x - 0.62))
    sun = 6000.0 * np.exp(-((dx / 0.006) ** 2 + ((y - 0.27) / 0.012) ** 2)) + 6.0 * np.exp(-((dx / 0.05) ** 2 + ((y - 0.27) / 0.08) ** 2))
    img = img + sun[..., None] * np.array([1.0, 0.93, 0.8])
    return np.ascontiguousarray(img, f32)


def matpreview_like(n_theta: int = 256, n_phi: int = 512, env_res=(1024, 512)) -> dict:
    """Material-preview style scene: a principled sphere (2 * n_phi * (n_theta - 1) triangles, smooth
    normals) and a rough metallic sphere on a checkerboard ground plane, lit ONLY by an HDR
    environment map -- the feature mix of BASELINE.json configs[3] (principled BSDF + envmap)."""
    T = Transform4f
    d = {"type": "scene",
         "integrator": {"type": "path", "max_depth": 8},
         "sensor": {"type": "perspective", "fov": 38, "near_clip": 0.01, "far_clip": 100,
                    "to_world": T().look_at(origin=[3.2, 2.1, 3.9], target=[0.1, 0.75, 0], up=[0, 1, 0]),
                    "film": {"type": "hdrfilm", "width": 1024, "height": 1024, "rfilter": {"type": "gaussian"}, "pixel_format": "rgb"},
                    "sampler": {"type": "independent", "sample_count": 128}},
         "ground-mat": {"type": "diffuse", "reflectance": {"type": "checkerboard", "color0": {"type": "rgb", "value": [0.35, 0.35, 0.35]},
                                                            "color1": {"type": "rgb", "value": [0.7, 0.7, 0.7]},
                                                            "to_uv": np.diag([10.0, 10.0, 1.0]).astype(f32)}},
         "paint": {"type": "principled", "base_color": {"type": "rgb", "value": [0.8, 0.15, 0.1]}, "roughness": 0.25, "metallic": 0.1,
                   "specular": 0.6, "clearcoat": 0.8, "clearcoat_gloss": 0.9, "sheen": 0.2},
         "brushed": {"type": "principled", "base_color": {"type": "rgb", "value": [0.9, 0.75, 0.4]}, "roughness": 0.4, "metallic": 1.0},
         "ground": {"type": "rectangle", "to_world": T().rotate([1, 0, 0], -90).scale(6.0), "bsdf": {"type": "ref", "id": "ground-mat"}}}
    s1 = uv_sphere_mesh(n_theta, n_phi, 1.0, (0.0, 1.0, 0.0)); s1["bsdf"] = {"type": "ref", "id": "paint"}
    s2 = uv_sphere_mesh(max(8, n_theta // 4), max(16, n_phi // 4), 0.45, (1.7, 0.45, 0.9)); s2["bsdf"] = {"type": "ref", "id": "brushed"}
    d["preview-object"] = s1
    d["small-sphere"] = s2
    d["sky"] = {"type": "envmap", "bitmap": synthetic_sky(*env_res), "scale": 1.0, "to_world": T().rotate([0, 1, 0], 25)}
    return d


def matpreview_scene(path: str | None = None) -> dict:
    """BASELINE.json configs[3]: the reference's own asset resources/data/scenes/matpreview, from the arrays that
    tests/golden/gen_matpreview.py extracted with the unmodified reference (three meshes as loaded, envmap / sensor
    transforms; envmap.exr as linear float32 RGB in matpreview_envmap.npz beside `path`, a file of its own so that
    neither exceeds 1 MB). `bsdf-matpreview` is the principled model of SURVEY.md 8(d)
    (base_color .94/.271/.361, roughness .3, metallic 0, specular .5); everything else follows matpreview.xml."""
    import os
    if path is None:
        path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "matpreview_scene.npz")
    z = np.load(path, allow_pickle=False)
    envmap = np.load(os.path.join(os.path.dirname(path), "matpreview_envmap.npz"), allow_pickle=False)["envmap"]

    def mesh(sid, bsdf):
        m = {"type": "mesh", "positions": z[f"{sid}|positions"], "texcoords": z[f"{sid}|texcoords"], "faces": z[f"{sid}|faces"], "bsdf": {"type": "ref", "id": bsdf}}
        if bool(z[f"{sid}|has_normals"]):
            m["normals"] = z[f"{sid}|normals"]
        return m
    return {
        "type": "scene",
        "integrator": {"type": "path", "max_depth": 8},
        "sensor": {"type": "perspective", "fov_axis": "smaller", "fov": float(z["sensor_fov"][0]), "near_clip": float(z["sensor_clip"][0]),
                   "far_clip": float(z["sensor_clip"][1]), "to_world": Transform4f(z["sensor_to_world"]),
                   "sampler": {"type": "independent", "sample_count": 64},
                   "film": {"type": "hdrfilm", "width": 683, "height": 512, "pixel_format": "rgb", "rfilter": {"type": "gaussian"}}},
        "emitter-envmap": {"type": "envmap", "data": envmap, "scale": float(np.asarray(z["envmap_scale"]).reshape(-1)[0]), "to_world": Transform4f(z["envmap_to_world"])},
        "bsdf-diffuse": {"type": "diffuse", "reflectance": {"type": "rgb", "value": [0.18, 0.18, 0.18]}},
        "bsdf-plane": {"type": "diffuse", "reflectance": {"type": "checkerboard", "color0": {"type": "rgb", "value": [0.4, 0.4, 0.4]},
                                                          "color1": {"type": "rgb", "value": [0.2, 0.2, 0.2]}, "to_uv": [[8, 0, 0], [0, 8, 0], [0, 0, 1]]}},
        "bsdf-matpreview": {"type": "principled", "base_color": {"type": "rgb", "value": [0.940, 0.271, 0.361]}, "roughness": 0.3, "metallic": 0.0, "specular": 0.5},
        "shape-plane": mesh("shape-plane", "bsdf-plane"),
        "shape-matpreview-interior": mesh("shape-matpreview-interior", "bsdf-diffuse"),
        "shape-matpreview-exterior": mesh("shape-matpreview-exterior", "bsdf-matpreview"),
    }
