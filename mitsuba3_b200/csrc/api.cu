// api.cu -- C ABI of libb200pt.so (include/b200pt.h) and the host-side wavefront
// scheduler: scene upload + BVH build, per-chunk kernel sequence on a CUDA stream
// (no host synchronisation inside a chunk: queue sizes stay on the device and the
// kernels are persistent grid-stride loops), film / gradient management.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/b200pt.h"
#include "bvh.h"
#include "env_host.h"
#include "kernels.cuh"

using namespace pt;

// ---------------------------------------------------------------------------
// error handling
// ---------------------------------------------------------------------------
static thread_local std::string g_error;
static b200pt_status fail(b200pt_status st, const std::string &msg) { g_error = msg; return st; }

#define CU_TRY(expr)                                                                                   \
    do {                                                                                               \
        cudaError_t _e = (expr);                                                                       \
        if (_e != cudaSuccess)                                                                         \
            return fail(B200PT_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));          \
    } while (0)

// ---------------------------------------------------------------------------
// scene object
// ---------------------------------------------------------------------------
struct TexMeta { int32_t kind, channels; size_t n; uint32_t grad_offset; bool differentiable; float *dev_data; };

struct Wavefront {
    size_t cap = 0;
    PathBuf buf[2];
    float4 *hit = nullptr, *lane_result = nullptr, *lane_dL = nullptr;
    uint32_t *vis = nullptr;        // NEE visibility bits of a gradient call (PathBuf::vis)
    Queues q;
    uint32_t *counts = nullptr; size_t n_counts = 0;
    std::vector<void *> allocs;
};

struct b200pt_scene {
    int device = 0;
    DevScene dev;
    std::vector<void *> allocs;
    std::vector<TexMeta> tex;
    bool type_present[N_BSDF_TYPES] = { false, false, false, false };
    size_t grad_floats = 0;
    uint32_t n_sm = 148;
    Launch launch;
    Wavefront wf;
    int shade_blocks_per_sm = 8;
    // shard pixel list cache
    uint32_t *pix_ids = nullptr; uint32_t n_shard_pix = 0; uint32_t pix_key[3] = { ~0u, ~0u, ~0u };
    uint32_t *all_pix_ids = nullptr;   // identity list (whole frame; weights pre-pass of the gaussian adjoint)
    uint32_t *cur_pix_ids = nullptr; uint32_t n_pix_ids = 0;   // the list selected by the last ensure_pix_ids
    // device refit (b200pt_scene_update_vertices): per shape (first vertex, count, sampling), BVH levels, un-inflated boxes
    std::vector<uint32_t> shape_first_vertex, shape_n_vertices; std::vector<int32_t> shape_sampling;
    std::vector<uint32_t> bvh_level_start; float *bvh_tight = nullptr;
    unsigned long long *stats_dev = nullptr;
    float *film_own = nullptr, *out_dev = nullptr, *grad_in_dev = nullptr, *film_w = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_stats = nullptr;
    std::vector<cudaEvent_t> trace_events; size_t trace_ev_used = 0;
    bool profile = false;
    b200pt_stats stats;
    // statistics are read back lazily (b200pt_get_stats): a render call never waits for the device on their account
    unsigned long long *stats_host = nullptr; bool stats_pending = false;
    // envmap emitter: its `data` texture and the device buffers rebuilt when that texture is updated
    // first differentiable texture that sits in a BSDF slot whose derivative the adjoint does not implement (-1: none):
    // the gradient entry points refuse such a scene instead of returning zeros for that parameter
    int32_t unsupported_grad_tex = -1; std::string unsupported_grad_why;
    int32_t env_tex = -1; bool env_mis_compensation = false; float *env_dev_tex = nullptr, *env_dev_warp = nullptr;
    uint32_t env_w = 0, env_h = 0;
};

// Host-to-device copy that has LANDED when it returns. cudaMemcpy from pageable host memory returns once the data sits in the
// driver's staging buffer; the DMA to the device is ordered on the legacy default stream only, and every stream this library
// launches on is non-blocking -- a kernel launched right after the call may read the old contents (measured: a device BVH refit
// of a 205k-triangle mesh that saw part of the previous vertices, tests/test_gpu_parity.py). Waiting for the legacy stream closes it.
static cudaError_t h2d(void *dst, const void *src, size_t bytes) {
    cudaError_t e = cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return e;
    return cudaStreamSynchronize(cudaStreamLegacy);
}

template <typename T>
static cudaError_t dev_upload(b200pt_scene *s, const T *host, size_t n, T **out) {
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T));
    if (e != cudaSuccess) return e;
    s->allocs.push_back(p);
    if (n) e = h2d(p, host, n * sizeof(T));
    *out = (T *) p;
    return e;
}

// BSDF slots whose parameter derivative the PRB adjoint implements: diffuse reflectance in closed form
// (kernels.cu: bsdf_backward), every texture slot of the principled, rough conductor, rough dielectric and plastic
// models through the dual-number evaluation of pt_bsdf_grad.cuh. Delta lobes (smooth conductor / dielectric, the
// specular component of plastic) have a zero gradient in detached PRB by construction (prb.py:296: bsdf.eval of a delta
// lobe is 0), so their slots are covered -- by an exact zero. Not covered: principled `specular` (it enters through
// the index of refraction, which the reference keeps as a non-differentiable float as well).
static bool adjoint_covers_slot(int32_t type, uint32_t flags, int slot) {
    (void) flags;
    if (type == B200PT_BSDF_PRINCIPLED) return slot != B200PT_SLOT_P_SPECULAR;
    return type >= B200PT_BSDF_DIFFUSE && type <= B200PT_BSDF_PLASTIC;
}

extern "C" {

uint32_t b200pt_abi_version(void) { return B200PT_ABI_VERSION; }
const char *b200pt_last_error(void) { return g_error.c_str(); }

int b200pt_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

static std::vector<int> g_devices;     // b200pt_set_devices

b200pt_status b200pt_set_devices(int n, const int *ids) {
    if (n < 0 || (n > 0 && !ids)) return fail(B200PT_ERR_INVALID, "null device list");
    int count = b200pt_device_count();
    for (int i = 0; i < n; ++i) if (ids[i] < 0 || ids[i] >= count) return fail(B200PT_ERR_CUDA, "no such CUDA device (mitsuba3_b200 has no CPU fallback)");
    g_devices.assign(ids, ids + n);
    return B200PT_OK;
}

void b200pt_scene_destroy(b200pt_scene *s) {
    if (!s) return;
    cudaSetDevice(s->device);
    if (s->stream) cudaStreamSynchronize(s->stream);
    for (void *p : s->allocs) cudaFree(p);
    for (void *p : s->wf.allocs) cudaFree(p);
    if (s->pix_ids) cudaFree(s->pix_ids);
    if (s->all_pix_ids) cudaFree(s->all_pix_ids);
    for (cudaEvent_t e : s->trace_events) cudaEventDestroy(e);
    if (s->ev0) cudaEventDestroy(s->ev0);
    if (s->ev1) cudaEventDestroy(s->ev1);
    if (s->ev_stats) cudaEventDestroy(s->ev_stats);
    if (s->stats_host) cudaFreeHost(s->stats_host);
    if (s->stream) cudaStreamDestroy(s->stream);
    delete s;
}

static void init_gaussian(DevScene &d, float stddev) {
    // gaussian.cpp:48-91: Remez fit to exp(-x/2), rescaled by stddev, zero at the radius
    d.gauss_radius = 4.f * stddev;
    static const double coeff[10] = { 9.992604880e-1, -4.977025247e-1, 1.222248550e-1, -1.932406282e-2, 2.136713061e-3,
                                      -1.679873860e-4, 9.202145248e-6, -3.329417433e-7, 7.128382794e-9, -6.821193280e-11 };
    float cs[10]; double scale = 1;
    for (int i = 0; i < 10; ++i) { cs[i] = (float) (coeff[i] * scale); scale /= (double) stddev * (double) stddev; }
    auto estrin = [&](float x) {
        float x2 = x * x, x4 = x2 * x2, x8 = x4 * x4;
        float p01 = fmaf(cs[1], x, cs[0]), p23 = fmaf(cs[3], x, cs[2]), p45 = fmaf(cs[5], x, cs[4]), p67 = fmaf(cs[7], x, cs[6]), p89 = fmaf(cs[9], x, cs[8]);
        return fmaf(p89, x8, fmaf(fmaf(p67, x2, p45), x4, fmaf(p23, x2, p01)));
    };
    cs[0] -= estrin(d.gauss_radius * d.gauss_radius);
    memcpy(d.gauss_coeff, cs, sizeof(cs));
    d.gauss_alpha = -1.f / (2.f * stddev * stddev);
    d.gauss_bias = expf(d.gauss_alpha * d.gauss_radius * d.gauss_radius);
}

b200pt_status b200pt_scene_create(const b200pt_scene_desc *desc, int device, b200pt_scene **out) {
    if (!desc || !out) return fail(B200PT_ERR_INVALID, "null argument");
    if (desc->abi_version != B200PT_ABI_VERSION) return fail(B200PT_ERR_INVALID, "ABI version mismatch");
    if (device == B200PT_DEVICE_AUTO) {      // b200pt_set_devices: the rank's device of the job's list
        const char *lr = getenv("LOCAL_RANK");
        int r = lr ? atoi(lr) : 0;
        device = g_devices.empty() ? 0 : g_devices[(size_t) (r < 0 ? 0 : r) % g_devices.size()];
    }
    if (b200pt_device_count() <= device || device < 0) return fail(B200PT_ERR_CUDA, "no such CUDA device (mitsuba3_b200 has no CPU fallback)");
    if (desc->sensor.rfilter == B200PT_RFILTER_GAUSSIAN_TABLE)
        return fail(B200PT_ERR_UNSUPPORTED, "the tabulated filter belongs to the scalar variants; JIT variants evaluate the filter analytically");
    CU_TRY(cudaSetDevice(device));
    b200pt_scene *s = new b200pt_scene();
    s->device = device;
    memset(&s->dev, 0, sizeof(s->dev));
    memset(&s->stats, 0, sizeof(s->stats));
    DevScene &d = s->dev;
#define S_TRY(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { std::string m = std::string(#expr) + ": " + cudaGetErrorString(_e); b200pt_scene_destroy(s); return fail(B200PT_ERR_CUDA, m); } } while (0)
#define S_FAIL(st, msg) do { b200pt_scene_destroy(s); return fail(st, msg); } while (0)
    cudaDeviceProp prop; S_TRY(cudaGetDeviceProperties(&prop, device));
    s->n_sm = (uint32_t) prop.multiProcessorCount;
    S_TRY(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
    S_TRY(cudaEventCreate(&s->ev0)); S_TRY(cudaEventCreate(&s->ev1)); S_TRY(cudaEventCreate(&s->ev_stats));
    { const char *e = getenv("B200PT_SHADE_BLOCKS_PER_SM"); s->shade_blocks_per_sm = e ? std::max(1, atoi(e)) : 8; }
    S_TRY(cudaMallocHost(&s->stats_host, ST_COUNT * sizeof(unsigned long long)));
    s->profile = getenv("B200PT_PROFILE") != nullptr;

    // ---- textures ----------------------------------------------------------
    std::vector<DevTexture> htex(desc->n_textures);
    size_t grad_off = 0;
    for (uint32_t i = 0; i < desc->n_textures; ++i) {
        const b200pt_texture &t = desc->textures[i];
        DevTexture &o = htex[i]; memset(&o, 0, sizeof(o));
        if (t.channels != 1 && t.channels != 3) S_FAIL(B200PT_ERR_INVALID, "texture channels must be 1 or 3");
        o.kind = t.kind; o.channels = t.channels; o.width = t.width; o.height = t.height; o.wrap = t.wrap; o.filter = t.filter;
        o.differentiable = t.differentiable;
        memcpy(o.value, t.value, sizeof(o.value)); memcpy(o.value1, t.value1, sizeof(o.value1)); memcpy(o.to_uv, t.to_uv, sizeof(o.to_uv));
        TexMeta m; m.kind = t.kind; m.channels = t.channels; m.differentiable = t.differentiable != 0; m.dev_data = nullptr;
        if (t.kind == B200PT_TEX_BITMAP) {
            if (!t.data || t.width <= 0 || t.height <= 0) S_FAIL(B200PT_ERR_INVALID, "bitmap texture without data");
            m.n = (size_t) t.width * t.height * t.channels;
            float *dd = nullptr; S_TRY(dev_upload(s, t.data, m.n, &dd));
            o.data = dd; m.dev_data = dd;
        } else m.n = (size_t) t.channels * (t.kind == B200PT_TEX_CHECKERBOARD ? 2 : 1);
        m.grad_offset = (uint32_t) grad_off; o.grad_offset = (uint32_t) grad_off;
        if (m.differentiable) grad_off += m.n;
        s->tex.push_back(m);
    }
    s->grad_floats = grad_off;
    d.n_textures = desc->n_textures;
    { float *g = nullptr; S_TRY(cudaMalloc(&g, std::max<size_t>(grad_off, 1) * sizeof(float))); s->allocs.push_back(g); S_TRY(cudaMemset(g, 0, std::max<size_t>(grad_off, 1) * sizeof(float))); d.grad = g; }
    { float *g = nullptr; S_TRY(cudaMalloc(&g, std::max<size_t>(grad_off, 1) * sizeof(float))); s->allocs.push_back(g); S_TRY(cudaMemset(g, 0, std::max<size_t>(grad_off, 1) * sizeof(float))); d.tangent = g; }

    // ---- bsdfs / emitters ----------------------------------------------------
    std::vector<DevBsdf> hb(desc->n_bsdfs);
    for (uint32_t i = 0; i < desc->n_bsdfs; ++i) {
        const b200pt_bsdf &b = desc->bsdfs[i];
        if (b.type < 0 || b.type > B200PT_BSDF_PLASTIC) S_FAIL(B200PT_ERR_UNSUPPORTED, "BSDF model outside the hot-path scope");
        hb[i].type = b.type; hb[i].twosided = b.twosided; memcpy(hb[i].tex, b.tex, sizeof(b.tex));
        for (int k = 0; k < B200PT_MAX_SLOTS; ++k) if (b.tex[k] >= (int32_t) desc->n_textures) S_FAIL(B200PT_ERR_INVALID, "BSDF references a missing texture");
        hb[i].eta = b.eta; hb[i].spec_srate = b.spec_srate; hb[i].clearcoat_srate = b.clearcoat_srate; hb[i].diff_refl_srate = b.diff_refl_srate; hb[i].flags = b.flags & ~PT_M_PLASTIC;
        hb[i].plastic_fdr_int = b.plastic_fdr_int; hb[i].plastic_spec_weight = b.plastic_spec_weight;
        if (b.type == B200PT_BSDF_PLASTIC) { hb[i].type = B200PT_BSDF_CONDUCTOR; hb[i].flags |= PT_M_PLASTIC; }   // shares the conductor queue / kernel
    }
    d.n_bsdfs = desc->n_bsdfs;
    for (uint32_t i = 0; i < desc->n_bsdfs && s->unsupported_grad_tex < 0; ++i) {
        const b200pt_bsdf &b = desc->bsdfs[i];
        for (int k = 0; k < B200PT_MAX_SLOTS; ++k) {
            int32_t t = b.tex[k];
            if (t < 0 || !desc->textures[t].differentiable || adjoint_covers_slot(b.type, b.flags, k)) continue;
            s->unsupported_grad_tex = t;
            s->unsupported_grad_why = "texture " + std::to_string(t) + " (slot " + std::to_string(k) + " of BSDF " + std::to_string(i) + ", model " + std::to_string(b.type) +
                                      ") is differentiable, but the PRB adjoint has no derivative for that slot; mark it non-differentiable";
            break;
        }
    }
    std::vector<DevEmitter> he(desc->n_emitters);
    DevEnv henv; memset(&henv, 0, sizeof(henv)); henv.type = -1; henv.emitter_index = -1; henv.radiance_tex = -1;
    d.env = nullptr; d.env_type = -1; d.env_emitter = -1; d.env_radiance_tex = -1;
    int env_index = -1;
    for (uint32_t i = 0; i < desc->n_emitters; ++i) {
        const b200pt_emitter &e = desc->emitters[i];
        if (!(e.sampling_weight >= 0.f)) S_FAIL(B200PT_ERR_INVALID, "emitter sampling_weight must be non-negative");
        he[i].shape = e.shape; he[i].radiance_tex = e.radiance_tex; he[i].sampling_weight = e.sampling_weight; he[i].type = e.type;
        if (e.type == B200PT_EMITTER_AREA) {
            if (e.shape < 0 || e.shape >= (int32_t) desc->n_shapes || e.radiance_tex < 0 || e.radiance_tex >= (int32_t) desc->n_textures)
                S_FAIL(B200PT_ERR_INVALID, "emitter references a missing shape/texture");
            if (desc->textures[e.radiance_tex].kind != B200PT_TEX_CONST) S_FAIL(B200PT_ERR_UNSUPPORTED, "textured area lights are outside the hot-path scope");
            continue;
        }
        if (e.type != B200PT_EMITTER_CONSTANT && e.type != B200PT_EMITTER_ENVMAP) S_FAIL(B200PT_ERR_UNSUPPORTED, "emitter type outside the hot-path scope");
        if (env_index >= 0) S_FAIL(B200PT_ERR_INVALID, "Only one environment emitter can be specified per scene.");   // scene.cpp:63-65
        env_index = (int) i;
        he[i].shape = -1;
        henv.type = e.type; d.env_type = e.type; d.env_emitter = (int32_t) i; d.env_radiance_tex = e.radiance_tex; d.env_scale = e.env_scale; henv.emitter_index = (int32_t) i; henv.radiance_tex = e.radiance_tex; henv.scale = e.env_scale;
        for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) { henv.m[r * 3 + c] = e.to_world[r * 4 + c]; henv.mi[r * 3 + c] = e.to_world_inv[r * 4 + c]; }
        if (e.type == B200PT_EMITTER_CONSTANT) {
            if (e.radiance_tex < 0 || e.radiance_tex >= (int32_t) desc->n_textures || desc->textures[e.radiance_tex].kind != B200PT_TEX_CONST)
                S_FAIL(B200PT_ERR_INVALID, "constant emitter: expected a non-spatially varying radiance");                // constant.cpp:64
        } else {
            if (e.radiance_tex < 0 || e.radiance_tex >= (int32_t) desc->n_textures) S_FAIL(B200PT_ERR_INVALID, "envmap: radiance_tex must name the bitmap texture holding the map");
            const b200pt_texture &et = desc->textures[e.radiance_tex];
            if (et.kind != B200PT_TEX_BITMAP || et.channels != 3 || !et.data) S_FAIL(B200PT_ERR_INVALID, "envmap: the map must be a 3-channel bitmap texture");
            EnvHost eh;
            if (!build_envmap(et.data, (uint32_t) et.width, (uint32_t) et.height, e.env_mis_compensation != 0, eh)) S_FAIL(B200PT_ERR_INVALID, "envmap: need float32 RGB data of at least 2 x 3 texels");
            if (eh.lvl_width.size() > (size_t) ENV_MAX_LEVELS) S_FAIL(B200PT_ERR_UNSUPPORTED, "envmap resolution too large");
            float *dt = nullptr, *dw = nullptr;
            S_TRY(dev_upload(s, eh.tex.data(), eh.tex.size(), &dt)); S_TRY(dev_upload(s, eh.warp.data(), eh.warp.size(), &dw));
            henv.tex = (const float4 *) dt; henv.warp = dw; henv.W = (uint32_t) et.width; henv.H = (uint32_t) et.height;
            s->env_tex = e.radiance_tex; s->env_mis_compensation = e.env_mis_compensation != 0; s->env_dev_tex = dt; s->env_dev_warp = dw; s->env_w = (uint32_t) et.width; s->env_h = (uint32_t) et.height;
            htex[e.radiance_tex].wrap = PT_WRAP_ENVMAP;      // gradient / tangent taps follow eval_spectrum (pt_device.cuh: tex_lookup)
            henv.n_levels = (uint32_t) eh.lvl_width.size();
            for (size_t l = 0; l < eh.lvl_width.size(); ++l) { henv.lvl_width[l] = eh.lvl_width[l]; henv.lvl_offset[l] = eh.lvl_offset[l]; }
            for (int k = 0; k < 2; ++k) { henv.patch_size[k] = eh.patch_size[k]; henv.inv_patch_size[k] = eh.inv_patch_size[k]; henv.max_patch_index[k] = eh.max_patch_index[k]; }
        }
    }
    d.n_emitters = desc->n_emitters;
    {
        // Scene::update_emitter_sampling_distribution (scene.cpp:120-140): DiscreteDistribution over the
        // sampling weights only if one of them differs from 1 (cdf accumulated in double, core/distr_1d.h:236-267)
        bool non_uniform = false;
        for (uint32_t i = 0; i < desc->n_emitters; ++i) if (desc->emitters[i].sampling_weight != 1.f) non_uniform = true;
        d.em_cdf = d.em_pmf = nullptr; d.em_sum = d.em_norm = 0.f;
        if (non_uniform) {
            std::vector<float> cdf(desc->n_emitters), pmf(desc->n_emitters);
            double acc = 0;
            for (uint32_t i = 0; i < desc->n_emitters; ++i) { pmf[i] = desc->emitters[i].sampling_weight; acc += (double) pmf[i]; cdf[i] = (float) acc; }
            if (!(cdf.back() > 0.f)) S_FAIL(B200PT_ERR_INVALID, "all emitter sampling weights are zero");
            float *dc = nullptr, *dp = nullptr; S_TRY(dev_upload(s, cdf.data(), cdf.size(), &dc)); S_TRY(dev_upload(s, pmf.data(), pmf.size(), &dp));
            d.em_cdf = dc; d.em_pmf = dp; d.em_sum = cdf.back(); d.em_norm = 1.0f / d.em_sum;
        }
    }

    // ---- shapes: flatten to one vertex / primitive array ---------------------
    size_t n_verts = 0, n_prims = 0;
    for (uint32_t i = 0; i < desc->n_shapes; ++i) { n_verts += desc->shapes[i].n_vertices; n_prims += desc->shapes[i].n_faces; }
    if (n_prims >= (1u << 28)) S_FAIL(B200PT_ERR_UNSUPPORTED, "too many triangles");
    std::vector<float> verts(n_verts * 8); std::vector<uint32_t> pv(n_prims * 4); std::vector<float> tri9(n_prims * 9);
    std::vector<DevShape> hs(desc->n_shapes);
    std::vector<uint32_t> uv_flipped((n_prims + 31) / 32 + 1, 0u); bool any_tangents = false;     // FaceUVFlipped bits (mesh_utils.h:32)
    size_t vo = 0, po = 0;
    for (uint32_t i = 0; i < desc->n_shapes; ++i) {
        const b200pt_shape &sh = desc->shapes[i];
        if ((sh.layout & B200PT_LAYOUT_TANGENTS) && (sh.layout & (B200PT_LAYOUT_NORMALS | B200PT_LAYOUT_TEXCOORDS)) != (B200PT_LAYOUT_NORMALS | B200PT_LAYOUT_TEXCOORDS))
            S_FAIL(B200PT_ERR_INVALID, "packed tangent frames need normals and texture coordinates (mesh.cpp:523)");
        any_tangents |= (sh.layout & B200PT_LAYOUT_TANGENTS) != 0;
        if (sh.bsdf < 0 || sh.bsdf >= (int32_t) desc->n_bsdfs) S_FAIL(B200PT_ERR_INVALID, "shape references a missing BSDF");
        if (sh.emitter >= (int32_t) desc->n_emitters) S_FAIL(B200PT_ERR_INVALID, "shape references a missing emitter");
        DevShape &o = hs[i]; memset(&o, 0, sizeof(o));
        o.layout = sh.layout; o.bsdf = sh.bsdf; o.emitter = sh.emitter; o.sampling = sh.sampling;
        o.first_prim = (uint32_t) po; o.n_prims = sh.n_faces; o.first_vertex = (uint32_t) vo;
        s->shape_first_vertex.push_back((uint32_t) vo); s->shape_n_vertices.push_back(sh.n_vertices); s->shape_sampling.push_back(sh.sampling);
        memcpy(o.to_world, sh.to_world, sizeof(o.to_world)); memcpy(o.frame_n, sh.frame_n, sizeof(o.frame_n)); o.inv_area = sh.inv_area;
        s->type_present[hb[sh.bsdf].type] = true;       // the queue / kernel class (plastic -> conductor)
        memcpy(&verts[vo * 8], sh.vertices, (size_t) sh.n_vertices * 8 * sizeof(float));
        std::vector<float> cdf, pmf;
        double acc = 0;
        for (uint32_t f = 0; f < sh.n_faces; ++f) {
            const uint32_t *fr = sh.faces + 4 * (size_t) f;
            for (int k = 0; k < 3; ++k) {
                if (fr[k] >= sh.n_vertices) S_FAIL(B200PT_ERR_INVALID, "face index out of range");
                pv[(po + f) * 4 + k] = (uint32_t) (vo + fr[k]);
                memcpy(&tri9[(po + f) * 9 + 3 * k], sh.vertices + 8 * (size_t) fr[k], 3 * sizeof(float));
            }
            pv[(po + f) * 4 + 3] = i;
            if ((sh.layout & B200PT_LAYOUT_TANGENTS) && (fr[3] & 0x80000000u)) uv_flipped[(po + f) >> 5] |= 1u << ((po + f) & 31u);
            if (sh.sampling == B200PT_SAMPLING_MESH) {
                // Mesh::build_pmf: face areas, cdf accumulated in double (core/distr_1d.h)
                const float *p0 = &tri9[(po + f) * 9], *p1 = p0 + 3, *p2 = p0 + 6;
                float e0[3] = { p1[0] - p0[0], p1[1] - p0[1], p1[2] - p0[2] }, e1[3] = { p2[0] - p0[0], p2[1] - p0[1], p2[2] - p0[2] };
                float c[3] = { fmaf(e0[1], e1[2], -(e0[2] * e1[1])), fmaf(e0[2], e1[0], -(e0[0] * e1[2])), fmaf(e0[0], e1[1], -(e0[1] * e1[0])) };
                float area = .5f * sqrtf(fmaf(c[2], c[2], fmaf(c[1], c[1], c[0] * c[0])));
                acc += (double) area; cdf.push_back((float) acc); pmf.push_back(area);
            }
        }
        if (sh.sampling == B200PT_SAMPLING_MESH) {
            // DiscreteDistribution::compute_cdf_scalar (core/distr_1d.h:236-267)
            float *dc = nullptr, *dp = nullptr; S_TRY(dev_upload(s, cdf.data(), cdf.size(), &dc)); S_TRY(dev_upload(s, pmf.data(), pmf.size(), &dp));
            o.area_cdf = dc; o.area_pmf = dp; o.area_sum = cdf.empty() ? 0.f : cdf.back(); o.area_norm = 1.0f / o.area_sum;
        }
        vo += sh.n_vertices; po += sh.n_faces;
    }
    if (env_index >= 0) {
        scene_bounding_sphere(verts.data(), n_verts, henv.center, henv.radius);
        DevEnv *de = nullptr; S_TRY(dev_upload(s, &henv, 1, &de)); d.env = de;
    }
    { float *p; S_TRY(dev_upload(s, verts.data(), verts.size(), &p)); d.vertices = (const float4 *) p; }
    { uint32_t *p; S_TRY(dev_upload(s, pv.data(), pv.size(), &p)); d.prim_verts = (const uint4 *) p; }
    d.uv_flipped = nullptr;
    if (any_tangents) { uint32_t *p; S_TRY(dev_upload(s, uv_flipped.data(), uv_flipped.size(), &p)); d.uv_flipped = p; }
    d.n_shapes = desc->n_shapes;
    {
        // one contiguous blob: shapes | bsdfs | emitters | textures, every section 16-byte aligned
        auto al = [](size_t x) { return (x + 15) & ~(size_t) 15; };
        size_t o_b = al(hs.size() * sizeof(DevShape)), o_e = al(o_b + hb.size() * sizeof(DevBsdf)), o_t = al(o_e + he.size() * sizeof(DevEmitter));
        size_t total = al(o_t + htex.size() * sizeof(DevTexture));
        std::vector<unsigned char> blob(std::max<size_t>(total, 16), 0);
        memcpy(blob.data(), hs.data(), hs.size() * sizeof(DevShape)); memcpy(blob.data() + o_b, hb.data(), hb.size() * sizeof(DevBsdf));
        memcpy(blob.data() + o_e, he.data(), he.size() * sizeof(DevEmitter)); memcpy(blob.data() + o_t, htex.data(), htex.size() * sizeof(DevTexture));
        unsigned char *p; S_TRY(dev_upload(s, blob.data(), blob.size(), &p));
        d.tables = p; d.tables_bytes = (uint32_t) blob.size(); d.off_bsdfs = (uint32_t) o_b; d.off_emitters = (uint32_t) o_e; d.off_textures = (uint32_t) o_t;
        d.shapes = (const DevShape *) p; d.bsdfs = (const DevBsdf *) (p + o_b); d.emitters = (const DevEmitter *) (p + o_e); d.textures = (const DevTexture *) (p + o_t);
        d.geom_bytes = (uint32_t) std::min<size_t>(n_prims * 16 + n_verts * 32, 0x7fffffff); d.n_vertices = (uint32_t) n_verts;
    }

    // ---- BVH ----------------------------------------------------------------
    Bvh bvh = build_bvh(tri9.data(), (uint32_t) n_prims);
    std::vector<float> tris(n_prims * 12);
    for (size_t i = 0; i < n_prims; ++i) {
        uint32_t src = bvh.order[i];
        const float *p0 = &tri9[(size_t) src * 9], *p1 = p0 + 3, *p2 = p0 + 6;
        float *o = &tris[i * 12];
        o[0] = p0[0]; o[1] = p0[1]; o[2] = p0[2]; memcpy(&o[3], &src, 4);
        o[4] = p1[0] - p0[0]; o[5] = p1[1] - p0[1]; o[6] = p1[2] - p0[2]; o[7] = 0.f;
        o[8] = p2[0] - p0[0]; o[9] = p2[1] - p0[1]; o[10] = p2[2] - p0[2]; o[11] = 0.f;
    }
    { BvhNode *p; S_TRY(dev_upload(s, bvh.nodes.data(), bvh.nodes.size(), &p)); d.nodes = (const float4 *) p; d.n_nodes = (uint32_t) bvh.nodes.size(); }
    { float *p; S_TRY(dev_upload(s, tris.data(), tris.size(), &p)); d.tris = (const float4 *) p; d.n_tris = (uint32_t) n_prims; }
    if (bvh.depth > 60) S_FAIL(B200PT_ERR_UNSUPPORTED, "BVH deeper than the traversal stack");
    s->bvh_level_start = bvh.level_start;
    { float *p = nullptr; S_TRY(cudaMalloc(&p, std::max<size_t>(bvh.nodes.size(), 1) * 12 * sizeof(float))); s->allocs.push_back(p); s->bvh_tight = p; }

    // ---- sensor / film -------------------------------------------------------
    const b200pt_sensor &se = desc->sensor;
    memcpy(d.s2c, se.sample_to_camera, sizeof(d.s2c)); memcpy(d.cam_to_world, se.to_world, sizeof(d.cam_to_world));
    d.near_clip = se.near_clip; d.far_clip = se.far_clip;
    d.film_w = se.film_size[0]; d.film_h = se.film_size[1]; d.crop_w = se.crop_size[0]; d.crop_h = se.crop_size[1];
    d.crop_x = se.crop_offset[0]; d.crop_y = se.crop_offset[1];
    if (d.crop_w == 0 || d.crop_h == 0) S_FAIL(B200PT_ERR_INVALID, "empty film");
    d.rfilter = se.rfilter; d.base_seed = se.base_seed;
    if (se.rfilter != B200PT_RFILTER_BOX) {
        if (!(se.rfilter_stddev > 0.f) || 4.f * se.rfilter_stddev > 7.5f) S_FAIL(B200PT_ERR_INVALID, "gaussian stddev out of range");
        init_gaussian(d, se.rfilter_stddev);
    }

    // ---- launch geometry: persistent grids, top of the BVH staged in shared memory
    s->launch.n_smem_nodes = std::min<uint32_t>(d.n_nodes, 512);         // 32 KiB of nodes
    s->launch.n_smem_tris = d.n_tris <= 512 ? d.n_tris : 0;              // <= 24 KiB of triangles
    s->launch.smem_trace = ((size_t) s->launch.n_smem_nodes * 64 + (size_t) s->launch.n_smem_tris * 48 + 127) & ~(size_t) 127;
    s->launch.smem_tables = (d.tables_bytes <= 12288 ? d.tables_bytes : 0) + (d.geom_bytes <= 20480 ? d.geom_bytes : 0);
    { const char *e = getenv("B200PT_TRACE_BLOCKS_PER_SM"); s->launch.grid = (int) s->n_sm * (e ? std::max(1, atoi(e)) : 5); }
    { const char *e = getenv("B200PT_REFILL_IDLE"); s->launch.refill_idle = e ? std::min(32, std::max(1, atoi(e))) : 8; }
    {   // scenes of at most 32 leaves whose tree and triangles are staged whole: flat traversal (kernels.cu: k_trace_flat)
        uint32_t n_leaves = 0;
        for (const auto &nd : bvh.nodes) { if (nd.left < 0) n_leaves++; if (nd.right < 0) n_leaves++; }
        const char *e = getenv("B200PT_FLAT_TRAVERSAL");
        s->launch.flat = (e ? atoi(e) != 0 : true) && n_leaves >= 1 && n_leaves <= 32 && d.n_tris <= 256 && s->launch.n_smem_nodes == d.n_nodes && s->launch.n_smem_tris == d.n_tris;
        const char *g = getenv("B200PT_FLAT_BLOCKS_PER_SM");
        s->launch.grid_flat = (int) s->n_sm * (g ? std::max(1, atoi(g)) : 4);
    }
    set_trace_smem_attr(s->launch.smem_trace + s->launch.smem_tables);
    S_TRY(cudaMalloc(&s->stats_dev, ST_COUNT * sizeof(unsigned long long))); s->allocs.push_back(s->stats_dev);
    size_t npix = (size_t) d.crop_w * d.crop_h;
    S_TRY(cudaMalloc(&s->film_own, npix * 4 * sizeof(float))); s->allocs.push_back(s->film_own);
    S_TRY(cudaMalloc(&s->film_w, npix * 4 * sizeof(float))); s->allocs.push_back(s->film_w);
    S_TRY(cudaMalloc(&s->out_dev, npix * 3 * sizeof(float))); s->allocs.push_back(s->out_dev);
    S_TRY(cudaMalloc(&s->grad_in_dev, npix * 3 * sizeof(float))); s->allocs.push_back(s->grad_in_dev);
    S_TRY(cudaDeviceSynchronize());
    *out = s;
    return B200PT_OK;
#undef S_TRY
#undef S_FAIL
}

b200pt_status b200pt_scene_update_vertices(b200pt_scene *s, uint32_t shape, const float *vertices, uint32_t n_vertices) {
    if (!s || !vertices) return fail(B200PT_ERR_INVALID, "null argument");
    if (shape >= s->shape_first_vertex.size() || n_vertices != s->shape_n_vertices[shape]) return fail(B200PT_ERR_INVALID, "shape index / vertex count mismatch");
    if (s->shape_sampling[shape] != B200PT_SAMPLING_NONE)
        return fail(B200PT_ERR_UNSUPPORTED, "the shape is sampled as an emitter (host-built sampling tables): create the scene again");
    if (s->dev.geom_bytes <= 20480) { /* small scenes: the shading kernels stage the geometry per launch from these arrays, nothing else to do */ }
    CU_TRY(cudaSetDevice(s->device));
    CU_TRY(cudaStreamSynchronize(s->stream));
    CU_TRY(h2d((float *) s->dev.vertices + 8 * (size_t) s->shape_first_vertex[shape], vertices, (size_t) n_vertices * 8 * sizeof(float)));
    launch_refit(s->dev, s->bvh_tight, s->bvh_level_start.data(), (uint32_t) s->bvh_level_start.size() - 1, (int) s->n_sm * 4, s->stream);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaStreamSynchronize(s->stream));
    return B200PT_OK;
}

b200pt_status b200pt_scene_update_texture(b200pt_scene *s, uint32_t tex, const float *host_data, size_t n) {
    if (!s || !host_data) return fail(B200PT_ERR_INVALID, "null argument");
    if (tex >= s->tex.size() || n != s->tex[tex].n) return fail(B200PT_ERR_INVALID, "texture index/size mismatch");
    CU_TRY(cudaSetDevice(s->device));
    CU_TRY(cudaStreamSynchronize(s->stream));
    if (s->tex[tex].kind == B200PT_TEX_BITMAP) {
        CU_TRY(h2d(s->tex[tex].dev_data, host_data, n * sizeof(float)));
        if ((int32_t) tex == s->env_tex) {
            // EnvironmentMapEmitter::parameters_changed (envmap.cpp:207-258): refresh the halo texture and
            // rebuild the sampling distribution (same sizes: the device buffers are reused)
            EnvHost eh;
            if (!build_envmap(host_data, s->env_w, s->env_h, s->env_mis_compensation, eh)) return fail(B200PT_ERR_INVALID, "envmap rebuild failed");
            CU_TRY(h2d(s->env_dev_tex, eh.tex.data(), eh.tex.size() * sizeof(float)));
            CU_TRY(h2d(s->env_dev_warp, eh.warp.data(), eh.warp.size() * sizeof(float)));
        }
    }
    else {
        const DevTexture *dt = s->dev.textures + tex;
        int ch = s->tex[tex].channels;
        CU_TRY(h2d((char *) dt + offsetof(DevTexture, value), host_data, ch * sizeof(float)));
        if (s->tex[tex].kind == B200PT_TEX_CHECKERBOARD)   // color0 then color1
            CU_TRY(h2d((char *) dt + offsetof(DevTexture, value1), host_data + ch, ch * sizeof(float)));
    }
    return B200PT_OK;
}

} // extern "C"

// ---------------------------------------------------------------------------
// wavefront buffers
// ---------------------------------------------------------------------------
constexpr uint32_t MAX_BOUNCE_SLOTS = 1024;   // counters for this many bounces per chunk

static b200pt_status ensure_wavefront(b200pt_scene *s, size_t cap, bool adjoint) {
    Wavefront &w = s->wf;
    bool need_adj = adjoint && (w.cap == 0 || w.buf[0].adj_L == nullptr);
    if (w.cap >= cap && !need_adj) return B200PT_OK;
    for (void *p : w.allocs) cudaFree(p);
    w.allocs.clear(); w.cap = 0;
    auto A = [&](size_t bytes, void **out) -> cudaError_t { cudaError_t e = cudaMalloc(out, bytes); if (e == cudaSuccess) w.allocs.push_back(*out); return e; };
    size_t slack = cap + 64;
    for (int b = 0; b < 2; ++b) {
        PathBuf &pb = w.buf[b]; memset(&pb, 0, sizeof(pb));
        CU_TRY(A(slack * 16, (void **) &pb.ray_o)); CU_TRY(A(slack * 16, (void **) &pb.ray_d)); CU_TRY(A(slack * 16, (void **) &pb.thr));
        CU_TRY(A(slack * 16, (void **) &pb.prev)); CU_TRY(A(slack * 16, (void **) &pb.rng)); CU_TRY(A(slack * 16, (void **) &pb.result));
        CU_TRY(A(slack * 16, (void **) &pb.sh_o)); CU_TRY(A(slack * 16, (void **) &pb.sh_d)); CU_TRY(A(slack * 8, (void **) &pb.sh_c));
        if (adjoint) { CU_TRY(A(slack * 16, (void **) &pb.adj_L)); CU_TRY(A(slack * 16, (void **) &pb.adj_dL)); }
    }
    w.vis = nullptr;
    if (adjoint) CU_TRY(A(slack * 4, (void **) &w.vis));
    CU_TRY(A(slack * 16, (void **) &w.hit)); CU_TRY(A(slack * 16, (void **) &w.lane_result)); CU_TRY(A(slack * 16, (void **) &w.lane_dL));
    for (int t = 0; t < N_BSDF_TYPES; ++t) {
        if (s->type_present[t]) CU_TRY(A(slack * 4, (void **) &w.q.slots[t])); else w.q.slots[t] = nullptr;
    }
    if (s->dev.env_type >= 0) CU_TRY(A(slack * 4, (void **) &w.q.slots[Q_ENV])); else w.q.slots[Q_ENV] = nullptr;
    w.n_counts = (size_t) (MAX_BOUNCE_SLOTS + 2) * 8;
    CU_TRY(A(w.n_counts * 4, (void **) &w.counts));
    w.q.counts = w.counts;
    w.cap = cap;
    return B200PT_OK;
}

// Tile (tx, ty) belongs to rank (tx + ty * stride) % count with the smallest stride >= count/2 + 1 that is coprime
// with count (count = 2: stride 1, a checkerboard) -- a diagonal deal: every rank meets every tile column and row, so
// no rank owns whole columns of the image (a plain t % count does when count divides the tiles per row: 16 % load
// imbalance on the Cornell box at 8 GPUs against 1.9 %). Same rule as mitsuba3_b200/dist.py: tile_owner.
static uint32_t tile_stride(uint32_t count) {
    if (count <= 2) return 1;
    auto gcd = [](uint32_t a, uint32_t b) { while (b) { uint32_t t = a % b; a = b; b = t; } return a; };
    uint32_t st = count / 2 + 1;
    while (gcd(st, count) != 1) ++st;
    return st;
}

static b200pt_status ensure_pix_ids(b200pt_scene *s, const b200pt_render_params *p) {
    uint32_t count = std::max(1u, p->shard_count), rank = p->shard_rank, ts = p->tile_size ? p->tile_size : 32;
    if (rank >= count) return fail(B200PT_ERR_INVALID, "shard_rank >= shard_count");
    uint32_t W = s->dev.crop_w, H = s->dev.crop_h;
    if (count == 1) {
        // whole frame in scanline order: its own cache slot (the gaussian adjoint uses it next to the shard's list)
        if (!s->all_pix_ids) {
            std::vector<uint32_t> ids((size_t) W * H);
            for (uint32_t i = 0; i < W * H; ++i) ids[i] = i;
            CU_TRY(cudaMalloc(&s->all_pix_ids, std::max<size_t>(ids.size(), 1) * 4));
            CU_TRY(h2d(s->all_pix_ids, ids.data(), ids.size() * 4));
        }
        s->cur_pix_ids = s->all_pix_ids; s->n_pix_ids = W * H;
        return B200PT_OK;
    }
    if (!(s->pix_ids && s->pix_key[0] == rank && s->pix_key[1] == count && s->pix_key[2] == ts)) {
        std::vector<uint32_t> ids; ids.reserve((size_t) W * H / count + 1024);
        uint32_t tiles_x = (W + ts - 1) / ts, tiles_y = (H + ts - 1) / ts;
        // within a rank the pixels are enumerated tile by tile in scanline order of the tiles, row-major inside a tile
        const uint32_t stride = tile_stride(count);
        for (uint32_t t = 0; t < tiles_x * tiles_y; ++t) {
            uint32_t ty = t / tiles_x, tx = t - ty * tiles_x;
            if ((tx + ty * stride) % count != rank) continue;
            for (uint32_t y = ty * ts; y < std::min(H, (ty + 1) * ts); ++y)
                for (uint32_t x = tx * ts; x < std::min(W, (tx + 1) * ts); ++x) ids.push_back(y * W + x);
        }
        if (s->pix_ids) { cudaFree(s->pix_ids); s->pix_ids = nullptr; }
        CU_TRY(cudaMalloc(&s->pix_ids, std::max<size_t>(ids.size(), 1) * 4));
        CU_TRY(h2d(s->pix_ids, ids.data(), ids.size() * 4));
        s->n_shard_pix = (uint32_t) ids.size();
        s->pix_key[0] = rank; s->pix_key[1] = count; s->pix_key[2] = ts;
    }
    s->cur_pix_ids = s->pix_ids; s->n_pix_ids = s->n_shard_pix;
    return B200PT_OK;
}

static cudaEvent_t next_trace_event(b200pt_scene *s) {
    if (s->trace_ev_used == s->trace_events.size()) { cudaEvent_t e; cudaEventCreate(&e); s->trace_events.push_back(e); }
    return s->trace_events[s->trace_ev_used++];
}

static int grid_for(const b200pt_scene *s, size_t n) {
    size_t blocks = (n + BLOCK - 1) / BLOCK;
    return (int) std::max<size_t>(1, std::min<size_t>(blocks, (size_t) s->n_sm * 8));
}

// One chunk of the wavefront: lanes [pix0*spp, (pix0+npix)*spp) of this shard.
// mode 0: primal (path / prb) -> lane_result; mode 1: PRB adjoint replay; mode 2: PRB forward-mode
// replay (lane_result <- dL of every sample).
static b200pt_status run_chunk(b200pt_scene *s, RenderCfg cfg, int mode, cudaStream_t st, bool use_vis = false) {
    Wavefront &w = s->wf;
    // gradient calls: the primal pass records the NEE visibility bits, the replay reads them (max_depth <= 32)
    w.buf[0].vis = w.buf[1].vis = use_vis ? w.vis : nullptr;
    const DevScene &d = s->dev;
    uint32_t lanes = cfg.chunk_lanes;
    cfg.adjoint = mode >= 1; cfg.forward = mode == 2;
    CU_TRY(cudaMemsetAsync(w.counts, 0, w.n_counts * 4, st));
    int g_all = grid_for(s, lanes);
    launch_generate(d, cfg, s->cur_pix_ids, w.buf[0], w.lane_dL, w.lane_result, g_all, st);
    s->stats.kernel_launches++;
    Launch L = s->launch;
    L.grid = std::min<int>(s->launch.grid, (int) ((lanes + BLOCK - 1) / BLOCK)); if (L.grid < 1) L.grid = 1;
    Launch Ls = L; Ls.grid = (int) std::min<size_t>((size_t) g_all, (size_t) s->n_sm * (size_t) s->shade_blocks_per_sm);
    auto trace = [&](int bufi, const uint32_t *n_in, uint32_t *qcounts, bool first) {
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        if (s->profile) { e0 = next_trace_event(s); e1 = next_trace_event(s); cudaEventRecord(e0, st); }
        launch_trace(d, cfg, w.buf[bufi], w.hit, n_in, w.q, qcounts, w.lane_result, s->stats_dev, first, L, st);
        if (s->profile) cudaEventRecord(e1, st);
        s->stats.kernel_launches++; s->stats.trace_launches++;
    };
    int cur = 0;
    trace(cur, nullptr, w.counts + 0, true);
    uint32_t max_b = std::min<uint32_t>(cfg.max_depth, MAX_BOUNCE_SLOTS);
    for (uint32_t b = 0; b < max_b; ++b) {
        uint32_t *cnt = w.counts + (size_t) b * 8;
        if (d.env_type >= 0) {     // rays of this bounce that left the scene: environment emitter, then the path ends
            launch_shade_env(d, cfg, w.buf[cur], w.q.slots[Q_ENV], cnt + QCOUNT_ENV, w.lane_result, s->stats_dev, g_all, st);
            s->stats.kernel_launches++;
        }
        for (int t = 0; t < N_BSDF_TYPES; ++t) {
            if (!s->type_present[t]) continue;
            const uint32_t *queue = w.q.slots[t];
            launch_shade(t, d, cfg, w.buf[cur], w.hit, queue, cnt + t, w.buf[cur ^ 1], cnt + 4, w.lane_result, s->stats_dev, Ls, st);
            s->stats.kernel_launches++;
        }
        cur ^= 1;
        trace(cur, cnt + 4, w.counts + (size_t) (b + 1) * 8, false);
        if (b >= 15 && (b & 7) == 7) {
            // long / unbounded paths: stop as soon as the wavefront is empty
            uint32_t alive[8];
            CU_TRY(cudaMemcpyAsync(alive, w.counts + (size_t) (b + 1) * 8, sizeof(alive), cudaMemcpyDeviceToHost, st));
            CU_TRY(cudaStreamSynchronize(st));
            if (alive[0] + alive[1] + alive[2] + alive[3] + alive[QCOUNT_ENV] == 0) break;
        }
    }
    if (max_b < cfg.max_depth && !(cfg.adjoint && !cfg.forward)) {
        // the bounce counters ran out before max_depth (unbounded paths only): the lanes still queued hand in the radiance
        // they have gathered so far instead of leaving their lane_result entry unwritten
        launch_flush(w.buf[cur], w.q, w.counts + (size_t) max_b * 8, w.lane_result, g_all, st);
        s->stats.kernel_launches++;
    }
    CU_TRY(cudaGetLastError());
    return B200PT_OK;
}

static RenderCfg make_cfg(const b200pt_scene *s, const b200pt_render_params *p) {
    RenderCfg c; memset(&c, 0, sizeof(c));
    c.seed_value = s->dev.base_seed + p->seed;
    c.spp = p->spp;
    c.max_depth = p->max_depth < 0 ? 0xffffffffu : (uint32_t) p->max_depth;
    c.rr_depth = (uint32_t) std::max(1, p->rr_depth);
    c.hide_emitters = p->hide_emitters; c.prb = p->prb;
    return c;
}

// bytes of wavefront state per lane (ensure_wavefront)
static size_t wavefront_bytes_per_lane(const b200pt_scene *s, bool adjoint) {
    size_t per = 2 * (8 * 16 + 8 + (adjoint ? 32 : 0)) + 3 * 16 + (adjoint ? 4 : 0);      // two path buffers + hit, lane_result, lane_dL
    for (int t = 0; t < N_BSDF_TYPES; ++t) if (s->type_present[t]) per += 4;
    if (s->dev.env_type >= 0) per += 4;
    return per;
}

// Chunking of a call over `n_pix` pixels of this shard: equal chunks of at most 64 Mi lanes (fewest launches measured best,
// profiles/r01_tuning.md), clamped to what the device can hold.
static size_t chunk_pixels(const b200pt_scene *s, const b200pt_render_params *p, uint32_t n_pix, bool adjoint) {
    size_t lanes = p->chunk_lanes;
    if (!lanes) { const char *e = getenv("B200PT_CHUNK_LANES"); lanes = e ? (size_t) atoll(e) : ((size_t) 1 << 26); }
    // never ask for more state than the device can hold next to what other users of the GPU (torch, NCCL) have taken:
    // the wavefront already allocated counts as available, 10 % of the free memory stays untouched
    // (only when the wavefront has to grow: the state already allocated for an earlier call of this size needs no new
    //  question to the driver -- cudaMemGetInfo is a host-side cost of every frame otherwise)
    const bool have_adj = s->wf.cap && s->wf.buf[0].adj_L != nullptr;
    const size_t want = std::min<size_t>(lanes, (size_t) n_pix * std::max(1u, p->spp));
    size_t free_b = 0, total_b = 0;
    if ((s->wf.cap < want || (adjoint && !have_adj)) && cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) {
        size_t per = wavefront_bytes_per_lane(s, adjoint);
        size_t held = s->wf.cap * wavefront_bytes_per_lane(s, have_adj);
        size_t fit = (size_t) ((double) (free_b + held) * 0.9) / per;
        if (lanes > fit) lanes = std::max<size_t>(fit, 1024);
    }
    size_t px = std::max<size_t>(1, lanes / std::max(1u, p->spp));
    size_t n_chunks = (n_pix + px - 1) / px;                              // equal chunks: no short tail pass
    return std::max<size_t>(1, (n_pix + n_chunks - 1) / std::max<size_t>(n_chunks, 1));
}

// Runs body(cfg of the chunk, pixels of the chunk) for every chunk of the shard, in order, on the caller's stream.
template <typename Body>
static b200pt_status for_each_chunk(b200pt_scene *s, const b200pt_render_params *p, RenderCfg cfg, bool adjoint, Body body) {
    const size_t cpx = chunk_pixels(s, p, s->n_pix_ids, adjoint);
    b200pt_status e = ensure_wavefront(s, cpx * p->spp, adjoint); if (e) return e;
    for (size_t pix0 = 0; pix0 < s->n_pix_ids; pix0 += cpx) {
        size_t npx = std::min<size_t>(cpx, s->n_pix_ids - pix0);
        cfg.chunk_pix0 = (uint32_t) pix0; cfg.chunk_lanes = (uint32_t) (npx * p->spp);
        e = body(cfg, npx); if (e) return e;
    }
    CU_TRY(cudaGetLastError());
    return B200PT_OK;
}

static b200pt_status validate_params(const b200pt_scene *s, const b200pt_render_params *p) {
    if (!s || !p) return fail(B200PT_ERR_INVALID, "null argument");
    if (p->spp == 0) return fail(B200PT_ERR_INVALID, "spp must be > 0");
    if (p->max_depth < -1) return fail(B200PT_ERR_INVALID, "\"max_depth\" must be set to -1 (infinite) or a value >= 0");
    if (p->rr_depth <= 0) return fail(B200PT_ERR_INVALID, "\"rr_depth\" must be set to a value greater than zero!");
    if ((uint64_t) s->dev.crop_w * s->dev.crop_h * p->spp > 0xffffffffull)
        return fail(B200PT_ERR_UNSUPPORTED, "more than 2^32 samples: split the render into passes (integrator.cpp:276-294)");
    return B200PT_OK;
}

static void begin_stats(b200pt_scene *s, cudaStream_t st) {
    memset(&s->stats, 0, sizeof(s->stats));
    s->stats_pending = false;
    s->trace_ev_used = 0;
    cudaMemsetAsync(s->stats_dev, 0, ST_COUNT * sizeof(unsigned long long), st);
    cudaEventRecord(s->ev0, st);
}

static b200pt_status end_stats(b200pt_scene *s, cudaStream_t st, uint64_t samples) {
    // no host synchronisation here: the counters travel to pinned host memory behind the kernels of this call and
    // are resolved by b200pt_get_stats (a frame that is followed by an NCCL all-reduce must not stall the host first)
    CU_TRY(cudaEventRecord(s->ev1, st));
    CU_TRY(cudaMemcpyAsync(s->stats_host, s->stats_dev, ST_COUNT * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaEventRecord(s->ev_stats, st));
    s->stats.samples = samples;
    s->stats_pending = true;
    return B200PT_OK;
}

static b200pt_status resolve_stats(b200pt_scene *s) {
    if (!s->stats_pending) return B200PT_OK;
    CU_TRY(cudaEventSynchronize(s->ev_stats));
    const unsigned long long *h = s->stats_host;
    float ms = 0.f; CU_TRY(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
    s->stats.device_ms = ms; s->stats.bounces = h[ST_BOUNCES]; s->stats.shadow_rays = h[ST_SHADOW];
    s->stats.trace_rays = h[ST_CLOSEST] + h[ST_SHADOW];
    double tms = 0;
    for (size_t i = 0; i + 1 < s->trace_ev_used; i += 2) { float m = 0.f; if (cudaEventElapsedTime(&m, s->trace_events[i], s->trace_events[i + 1]) == cudaSuccess) tms += m; }
    s->stats.trace_ms = tms;
    s->stats_pending = false;
#ifdef B200PT_WATCHDOG
    { unsigned long long wd[4]; read_watchdog(wd); if (wd[0] | wd[1] | wd[2]) fprintf(stderr, "b200pt watchdog: mbarrier %llu, walk %llu, rounds %llu\n", wd[0], wd[1], wd[2]); }
#endif
    return B200PT_OK;
}

// Scratch device allocations of the query entry points below; released on every exit
// path (CU_TRY returns early on a failed copy or launch).
struct DevScratch {
    std::vector<void *> ptrs;
    template <typename T> cudaError_t alloc(T **p, size_t bytes) {
        cudaError_t e = cudaMalloc((void **) p, bytes);
        if (e == cudaSuccess) ptrs.push_back((void *) *p);
        return e;
    }
    ~DevScratch() { for (void *p : ptrs) cudaFree(p); }
};

extern "C" {

b200pt_status b200pt_render_accumulate(b200pt_scene *s, const b200pt_render_params *p, float *film_device, void *cuda_stream) {
    b200pt_status vs = validate_params(s, p); if (vs) return vs;
    if (!film_device) return fail(B200PT_ERR_INVALID, "null film");
    CU_TRY(cudaSetDevice(s->device));
    cudaStream_t st = (cudaStream_t) cuda_stream;   // NULL = the CUDA default stream, as everywhere in CUDA
    b200pt_status e = ensure_pix_ids(s, p); if (e) return e;
    begin_stats(s, st);
    if (p->max_depth == 0 || s->n_pix_ids == 0) {
        // path.cpp:102: nothing to trace; the film still receives the sample weights
        return end_stats(s, st, 0);
    }
    RenderCfg cfg = make_cfg(s, p);
    e = for_each_chunk(s, p, cfg, false, [&](const RenderCfg &c, size_t npx) -> b200pt_status {
        b200pt_status e2 = run_chunk(s, c, 0, st); if (e2) return e2;
        launch_splat(s->dev, c, s->cur_pix_ids, s->wf.lane_result, film_device, grid_for(s, s->dev.rfilter == B200PT_RFILTER_BOX ? npx * 32 : c.chunk_lanes), st);
        s->stats.kernel_launches++;
        return B200PT_OK;
    });
    if (e) return e;
    return end_stats(s, st, (uint64_t) s->n_pix_ids * p->spp);
}

b200pt_status b200pt_develop(b200pt_scene *s, const float *film_device, float *out_device, void *cuda_stream) {
    if (!s || !film_device || !out_device) return fail(B200PT_ERR_INVALID, "null argument");
    CU_TRY(cudaSetDevice(s->device));
    cudaStream_t st = (cudaStream_t) cuda_stream;   // NULL = the CUDA default stream, as everywhere in CUDA
    launch_develop(s->dev, film_device, out_device, st);
    CU_TRY(cudaGetLastError());
    return B200PT_OK;
}

b200pt_status b200pt_render(b200pt_scene *s, const b200pt_render_params *p, float *out_host) {
    if (!s || !out_host) return fail(B200PT_ERR_INVALID, "null argument");
    CU_TRY(cudaSetDevice(s->device));
    size_t npix = (size_t) s->dev.crop_w * s->dev.crop_h;
    CU_TRY(cudaMemsetAsync(s->film_own, 0, npix * 4 * sizeof(float), s->stream));
    b200pt_status e = b200pt_render_accumulate(s, p, s->film_own, s->stream); if (e) return e;
    e = b200pt_develop(s, s->film_own, s->out_dev, s->stream); if (e) return e;
    CU_TRY(cudaMemcpyAsync(out_host, s->out_dev, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, s->stream));
    CU_TRY(cudaStreamSynchronize(s->stream));
    return B200PT_OK;
}

b200pt_status b200pt_render_backward_device(b200pt_scene *s, const b200pt_render_params *p_, const float *grad_in_device, void *cuda_stream) {
    b200pt_status vs = validate_params(s, p_); if (vs) return vs;
    if (!grad_in_device) return fail(B200PT_ERR_INVALID, "null grad_in");
    if (s->unsupported_grad_tex >= 0) return fail(B200PT_ERR_UNSUPPORTED, s->unsupported_grad_why);
    b200pt_render_params p = *p_; p.prb = 1;
    CU_TRY(cudaSetDevice(s->device));
    cudaStream_t st = (cudaStream_t) cuda_stream;   // NULL = the CUDA default stream, as everywhere in CUDA
    begin_stats(s, st);
    if (p.max_depth == 0) return end_stats(s, st, 0);
    RenderCfg cfg = make_cfg(s, &p);
    const DevScene &d = s->dev;
    size_t npix = (size_t) d.crop_w * d.crop_h;
    if (d.rfilter != B200PT_RFILTER_BOX) {
        // accumulated filter weights of THIS sample set over the whole frame (common.py:696-746):
        // cheap (RNG + splat of the weight channel), so every shard computes the full image itself
        b200pt_render_params all = p; all.shard_rank = 0; all.shard_count = 1;
        b200pt_status e = ensure_pix_ids(s, &all); if (e) return e;
        CU_TRY(cudaMemsetAsync(s->film_w, 0, npix * 4 * sizeof(float), st));
        RenderCfg wc = cfg; wc.chunk_pix0 = 0;
        size_t cpx = std::max<size_t>(1, ((size_t) 1 << 24) / p.spp);
        for (size_t pix0 = 0; pix0 < npix; pix0 += cpx) {
            size_t npx = std::min(cpx, npix - pix0);
            wc.chunk_pix0 = (uint32_t) pix0; wc.chunk_lanes = (uint32_t) (npx * p.spp);
            launch_weights(d, wc, s->cur_pix_ids, s->film_w, grid_for(s, wc.chunk_lanes), st);
            s->stats.kernel_launches++;
        }
    }
    b200pt_status e = ensure_pix_ids(s, &p); if (e) return e;
    if (s->n_pix_ids == 0) return end_stats(s, st, 0);
    const bool use_vis = cfg.max_depth <= 32 && !getenv("B200PT_INLINE_VISIBILITY");
    e = for_each_chunk(s, &p, cfg, true, [&](const RenderCfg &c, size_t) -> b200pt_status {
        // pass 1: primal with the same stream (sampler.clone(), common.py:752) -> L per lane
        b200pt_status e2 = run_chunk(s, c, 0, st, use_vis); if (e2) return e2;
        // dL per lane: adjoint of splat + develop
        launch_splat_adjoint(d, c, s->cur_pix_ids, grad_in_device, s->film_w, s->wf.lane_dL, grid_for(s, c.chunk_lanes), st);
        s->stats.kernel_launches++;
        // pass 2: adjoint replay (common.py:765)
        return run_chunk(s, c, 1, st, use_vis);
    });
    if (e) return e;
    return end_stats(s, st, (uint64_t) s->n_pix_ids * p.spp);
}

b200pt_status b200pt_render_backward(b200pt_scene *s, const b200pt_render_params *p, const float *grad_in_host) {
    if (!s || !grad_in_host) return fail(B200PT_ERR_INVALID, "null argument");
    CU_TRY(cudaSetDevice(s->device));
    size_t npix = (size_t) s->dev.crop_w * s->dev.crop_h;
    CU_TRY(cudaMemcpyAsync(s->grad_in_dev, grad_in_host, npix * 3 * sizeof(float), cudaMemcpyHostToDevice, s->stream));
    b200pt_status e = b200pt_render_backward_device(s, p, s->grad_in_dev, s->stream); if (e) return e;
    CU_TRY(cudaStreamSynchronize(s->stream));
    return B200PT_OK;
}

// RBIntegrator.render_forward (common.py:560-623): primal pass (L per lane), forward-mode replay
// (dL per lane, the parameter tangents come from b200pt_tangent_write), splat + develop of the dL.
b200pt_status b200pt_render_forward(b200pt_scene *s, const b200pt_render_params *p_, float *out_host) {
    b200pt_status vs = validate_params(s, p_); if (vs) return vs;
    if (!out_host) return fail(B200PT_ERR_INVALID, "null argument");
    if (s->unsupported_grad_tex >= 0) return fail(B200PT_ERR_UNSUPPORTED, s->unsupported_grad_why);
    b200pt_render_params p = *p_; p.prb = 1;
    CU_TRY(cudaSetDevice(s->device));
    cudaStream_t st = s->stream;
    size_t npix = (size_t) s->dev.crop_w * s->dev.crop_h;
    CU_TRY(cudaMemsetAsync(s->film_own, 0, npix * 4 * sizeof(float), st));
    b200pt_status e = ensure_pix_ids(s, &p); if (e) return e;
    begin_stats(s, st);
    if (p.max_depth != 0 && s->n_pix_ids != 0) {
        RenderCfg cfg = make_cfg(s, &p);
        const bool use_vis = cfg.max_depth <= 32 && !getenv("B200PT_INLINE_VISIBILITY");
        e = for_each_chunk(s, &p, cfg, true, [&](const RenderCfg &c, size_t npx) -> b200pt_status {
            b200pt_status e2 = run_chunk(s, c, 0, st, use_vis); if (e2) return e2;      // primal: L per lane (+ NEE visibility bits)
            e2 = run_chunk(s, c, 2, st, use_vis); if (e2) return e2;                     // forward replay: dL per lane
            launch_splat(s->dev, c, s->cur_pix_ids, s->wf.lane_result, s->film_own, grid_for(s, s->dev.rfilter == B200PT_RFILTER_BOX ? npx * 32 : c.chunk_lanes), st);
            s->stats.kernel_launches++;
            return B200PT_OK;
        });
        if (e) return e;
    }
    e = end_stats(s, st, (uint64_t) s->n_pix_ids * p.spp); if (e) return e;
    e = b200pt_develop(s, s->film_own, s->out_dev, st); if (e) return e;
    CU_TRY(cudaMemcpyAsync(out_host, s->out_dev, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    return B200PT_OK;
}

b200pt_status b200pt_tangent_zero(b200pt_scene *s) {
    if (!s) return fail(B200PT_ERR_INVALID, "null argument");
    CU_TRY(cudaSetDevice(s->device));
    CU_TRY(cudaMemsetAsync((void *) s->dev.tangent, 0, std::max<size_t>(s->grad_floats, 1) * sizeof(float), s->stream));
    CU_TRY(cudaStreamSynchronize(s->stream));
    return B200PT_OK;
}

b200pt_status b200pt_tangent_write(b200pt_scene *s, uint32_t tex, const float *host_in, size_t n) {
    size_t off = 0, cnt = 0;
    b200pt_status e = b200pt_grad_offset(s, tex, &off, &cnt); if (e) return e;
    if (n != cnt || !host_in) return fail(B200PT_ERR_INVALID, "tangent size mismatch");
    CU_TRY(cudaSetDevice(s->device));
    CU_TRY(h2d((void *) (s->dev.tangent + off), host_in, n * sizeof(float)));
    return B200PT_OK;
}

b200pt_status b200pt_grad_zero(b200pt_scene *s) {
    if (!s) return fail(B200PT_ERR_INVALID, "null argument");
    CU_TRY(cudaSetDevice(s->device));
    CU_TRY(cudaMemsetAsync(s->dev.grad, 0, std::max<size_t>(s->grad_floats, 1) * sizeof(float), s->stream));
    CU_TRY(cudaStreamSynchronize(s->stream));
    return B200PT_OK;
}

b200pt_status b200pt_grad_offset(b200pt_scene *s, uint32_t tex, size_t *offset, size_t *n) {
    if (!s || tex >= s->tex.size()) return fail(B200PT_ERR_INVALID, "texture index out of range");
    if (!s->tex[tex].differentiable) return fail(B200PT_ERR_INVALID, "texture is not differentiable");
    if (offset) *offset = s->tex[tex].grad_offset;
    if (n) *n = s->tex[tex].n;
    return B200PT_OK;
}

b200pt_status b200pt_grad_read(b200pt_scene *s, uint32_t tex, float *host_out, size_t n) {
    size_t off = 0, cnt = 0;
    b200pt_status e = b200pt_grad_offset(s, tex, &off, &cnt); if (e) return e;
    if (n != cnt || !host_out) return fail(B200PT_ERR_INVALID, "gradient size mismatch");
    CU_TRY(cudaSetDevice(s->device));
    CU_TRY(cudaStreamSynchronize(s->stream));
    CU_TRY(cudaMemcpy(host_out, s->dev.grad + off, n * sizeof(float), cudaMemcpyDeviceToHost));
    return B200PT_OK;
}

b200pt_status b200pt_grad_device_view(b200pt_scene *s, float **ptr, size_t *n) {
    if (!s || !ptr || !n) return fail(B200PT_ERR_INVALID, "null argument");
    *ptr = s->dev.grad; *n = s->grad_floats;
    return B200PT_OK;
}

// ---- operators ----------------------------------------------------------------
b200pt_status b200pt_ray_intersect(b200pt_scene *s, uint32_t n, const float *rays_host, float *t_out, float *uv_out, uint32_t *prim_out, int32_t *shape_out) {
    if (!s || (n && (!rays_host || !t_out || !uv_out || !prim_out || !shape_out))) return fail(B200PT_ERR_INVALID, "null argument");
    if (n == 0) return B200PT_OK;   // empty batch
    CU_TRY(cudaSetDevice(s->device));
    float *dr, *dt, *duv; uint32_t *dp; int32_t *ds; DevScratch tmp;
    CU_TRY(tmp.alloc(&dr, (size_t) n * 28)); CU_TRY(tmp.alloc(&dt, (size_t) n * 4)); CU_TRY(tmp.alloc(&duv, (size_t) n * 8));
    CU_TRY(tmp.alloc(&dp, (size_t) n * 4)); CU_TRY(tmp.alloc(&ds, (size_t) n * 4));
    CU_TRY(cudaMemcpyAsync(dr, rays_host, (size_t) n * 28, cudaMemcpyHostToDevice, s->stream));
    Launch L = s->launch; L.grid = grid_for(s, n);
    launch_ray_intersect(s->dev, n, dr, dt, duv, dp, ds, L, s->stream);
    CU_TRY(cudaMemcpyAsync(t_out, dt, (size_t) n * 4, cudaMemcpyDeviceToHost, s->stream));
    CU_TRY(cudaMemcpyAsync(uv_out, duv, (size_t) n * 8, cudaMemcpyDeviceToHost, s->stream));
    CU_TRY(cudaMemcpyAsync(prim_out, dp, (size_t) n * 4, cudaMemcpyDeviceToHost, s->stream));
    CU_TRY(cudaMemcpyAsync(shape_out, ds, (size_t) n * 4, cudaMemcpyDeviceToHost, s->stream));
    CU_TRY(cudaStreamSynchronize(s->stream));
    return B200PT_OK;
}

b200pt_status b200pt_ray_test(b200pt_scene *s, uint32_t n, const float *rays_host, uint8_t *hit_out) {
    if (!s || (n && (!rays_host || !hit_out))) return fail(B200PT_ERR_INVALID, "null argument");
    if (n == 0) return B200PT_OK;
    CU_TRY(cudaSetDevice(s->device));
    float *dr; uint8_t *dh; DevScratch tmp;
    CU_TRY(tmp.alloc(&dr, (size_t) n * 28)); CU_TRY(tmp.alloc(&dh, n));
    CU_TRY(cudaMemcpyAsync(dr, rays_host, (size_t) n * 28, cudaMemcpyHostToDevice, s->stream));
    Launch L = s->launch; L.grid = grid_for(s, n);
    launch_ray_test(s->dev, n, dr, dh, L, s->stream);
    CU_TRY(cudaMemcpyAsync(hit_out, dh, n, cudaMemcpyDeviceToHost, s->stream));
    CU_TRY(cudaStreamSynchronize(s->stream));
    return B200PT_OK;
}

b200pt_status b200pt_bsdf_eval_pdf_sample(b200pt_scene *s, uint32_t bsdf, uint32_t n, const float *in_host, float *out_host) {
    if (!s || (n && (!in_host || !out_host))) return fail(B200PT_ERR_INVALID, "null argument");
    if (bsdf >= s->dev.n_bsdfs) return fail(B200PT_ERR_INVALID, "BSDF index out of range");
    if (n == 0) return B200PT_OK;
    CU_TRY(cudaSetDevice(s->device));
    float *di, *dout; DevScratch tmp;
    CU_TRY(tmp.alloc(&di, (size_t) n * 44)); CU_TRY(tmp.alloc(&dout, (size_t) n * 56));
    CU_TRY(cudaMemcpyAsync(di, in_host, (size_t) n * 44, cudaMemcpyHostToDevice, s->stream));
    DevBsdf hb; CU_TRY(cudaMemcpy(&hb, s->dev.bsdfs + bsdf, sizeof(hb), cudaMemcpyDeviceToHost));
    launch_bsdf_eval(s->dev, bsdf, hb.type, n, di, dout, s->stream);
    CU_TRY(cudaMemcpyAsync(out_host, dout, (size_t) n * 56, cudaMemcpyDeviceToHost, s->stream));
    CU_TRY(cudaStreamSynchronize(s->stream));
    return B200PT_OK;
}

b200pt_status b200pt_env_query(b200pt_scene *s, uint32_t n, const float *in_host, float *out_host) {
    if (!s || (n && (!in_host || !out_host))) return fail(B200PT_ERR_INVALID, "null argument");
    if (s->dev.env_type < 0) return fail(B200PT_ERR_INVALID, "the scene has no environment emitter");
    if (n == 0) return B200PT_OK;
    CU_TRY(cudaSetDevice(s->device));
    float *di, *dout; DevScratch tmp;
    CU_TRY(tmp.alloc(&di, (size_t) n * 32)); CU_TRY(tmp.alloc(&dout, (size_t) n * 80));
    CU_TRY(cudaMemcpyAsync(di, in_host, (size_t) n * 32, cudaMemcpyHostToDevice, s->stream));
    launch_env_query(s->dev, n, di, dout, s->stream);
    CU_TRY(cudaMemcpyAsync(out_host, dout, (size_t) n * 80, cudaMemcpyDeviceToHost, s->stream));
    CU_TRY(cudaStreamSynchronize(s->stream));
    return B200PT_OK;
}

b200pt_status b200pt_get_stats(b200pt_scene *s, b200pt_stats *out) {
    if (!s || !out) return fail(B200PT_ERR_INVALID, "null argument");
    CU_TRY(cudaSetDevice(s->device));
    b200pt_status e = resolve_stats(s); if (e) return e;
    *out = s->stats;
    return B200PT_OK;
}

// size of the ABI structs as compiled (checked against the ctypes mirror by tests/test_abi.py)
size_t b200pt_abi_sizeof(int which) {
    switch (which) {
        case 0: return sizeof(b200pt_texture); case 1: return sizeof(b200pt_bsdf); case 2: return sizeof(b200pt_shape);
        case 3: return sizeof(b200pt_emitter); case 4: return sizeof(b200pt_sensor); case 5: return sizeof(b200pt_scene_desc);
        case 6: return sizeof(b200pt_render_params); case 7: return sizeof(b200pt_stats);
    }
    return 0;
}

} // extern "C"
