// kernels.cu -- the wavefront kernels of the B200 path tracer (sm_100a).
//
// One wavefront per bounce (SURVEY.md 8(a), DESIGN.md):
//
//   k_generate      lane -> pixel, TEA/PCG32 seeding, primary ray          (integrator.cpp:322-339,448-485)
//   k_trace_flat /  traversal (flat leaf-box kernel for scenes of <= 32 leaves, persistent BVH walk with dynamic
//   k_trace_dyn     work fetch otherwise): resolves the pending NEE shadow ray of
//                   every slot (Scene::ray_test), then the closest hit of its path ray
//                   (Scene::ray_intersect_preliminary) and bins the slot into the
//                   queue of the material it hit, or into the queue of the rays that
//                   left the scene (warp-ballot bucket pass)
//   k_shade_env     escaped rays: environment emitter (envmap / constant) x MIS, path ends
//   k_shade<TYPE>   one branch-flattened kernel per BSDF model over its material
//                   queue: surface interaction, emitter hit + MIS, NEE sample, BSDF
//                   eval/sample, russian roulette; writes the survivors COMPACTED
//                   into the other state buffer (warp-aggregated slot allocation).
//                   <TYPE, true>: PRB replay -- adjoint (gradient scatter) or forward mode
//   k_splat_*       ImageBlock::put (box / gaussian), k_develop: HDRFilm::develop
//
// The path state lives in HBM as structure-of-arrays float4 vectors (kernels.cuh).
// BVH nodes/triangles of the top of the tree are staged into shared memory with a
// bulk asynchronous copy (TMA, cp.async.bulk + mbarrier) once per persistent CTA.
#include "kernels.cuh"
#include <mutex>
#include <algorithm>

namespace pt {

// ---------------------------------------------------------------------------
// TMA bulk copy global -> shared, completion on an mbarrier
// ---------------------------------------------------------------------------
PT_DEV uint32_t smem_u32(const void *p) { return (uint32_t) __cvta_generic_to_shared(p); }
PT_DEV void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
PT_DEV void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
PT_DEV void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
#ifdef B200PT_WATCHDOG
// debugging build only: counters of loops that ran past any plausible bound (0: mbarrier wait, 1: BVH walk of one ray, 2: rounds of a warp)
__device__ unsigned long long g_watchdog[4];
#endif
PT_DEV void mbar_wait(uint64_t *bar, uint32_t phase) {
    uint32_t done = 0;
#ifdef B200PT_WATCHDOG
    uint32_t spins = 0;
#endif
    while (!done) {
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n" : "=r"(done) : "r"(smem_u32(bar)), "r"(phase) : "memory");
#ifdef B200PT_WATCHDOG
        if (++spins > (1u << 22)) { atomicAdd(&g_watchdog[0], 1ull); break; }
#endif
    }
}

// Stage `n_nodes` BVH nodes (64 B each) and `n_tris` triangles (48 B each) into
// shared memory. One elected thread arms the barrier and issues the copies in
// <= 32 KiB pieces; everybody waits on the barrier's phase 0.
PT_DEV void stage_bvh(const DevScene &sc, float4 *s_nodes, float4 *s_tris, uint32_t n_nodes, uint32_t n_tris, uint64_t *bar) {
    if (threadIdx.x == 0) {
        uint32_t nb = n_nodes * 64u, tb = n_tris * 48u;
        mbar_expect_tx(bar, nb + tb);
        const char *src = (const char *) sc.nodes; char *dst = (char *) s_nodes;
        for (uint32_t off = 0; off < nb; off += 32768u) bulk_g2s(dst + off, src + off, min(32768u, nb - off), bar);
        src = (const char *) sc.tris; dst = (char *) s_tris;
        for (uint32_t off = 0; off < tb; off += 32768u) bulk_g2s(dst + off, src + off, min(32768u, tb - off), bar);
    }
    mbar_wait(bar, 0);
    // Every thread must have seen phase 0 complete before thread 0 arms phase 1 (stage_tables): a thread that still polls
    // parity 0 after phase 1 has completed as well waits for phase 2, which nobody arms -- the block spins forever. It takes
    // a busy SM to delay a warp that long (blocks that become resident while other blocks keep the issue slots busy:
    // grids larger than one wave, kernels of another stream); measured as hangs, profiles/r02_summary.md.
    __syncthreads();
}

// Scene tables (shapes, BSDFs, emitters, textures) and -- for small scenes -- the shading
// geometry (prim_verts + packed vertices) are staged into shared memory as well: the
// shading kernels chase slot -> hit -> primitive -> vertex -> shape -> BSDF -> texture,
// and every hop that stays on chip removes an L2 round trip from that dependent chain.
constexpr uint32_t TABLES_SMEM_MAX = 12288, GEOM_SMEM_MAX = 20480;
PT_DEV uint32_t tables_smem_bytes(const DevScene &sc) {
    return (sc.tables_bytes <= TABLES_SMEM_MAX ? sc.tables_bytes : 0u) + (sc.geom_bytes <= GEOM_SMEM_MAX ? sc.geom_bytes : 0u);
}
// `sc` is the kernel's private copy of the scene descriptor; its pointers are redirected.
PT_DEV void stage_tables(DevScene &sc, unsigned char *smem, uint64_t *bar, uint32_t phase) {
    bool st = sc.tables_bytes <= TABLES_SMEM_MAX, sg = sc.geom_bytes <= GEOM_SMEM_MAX;
    if (!st && !sg) return;
    uint32_t tb = st ? sc.tables_bytes : 0u, gb = sg ? sc.geom_bytes : 0u;
    if (threadIdx.x == 0) {
        mbar_expect_tx(bar, tb + gb);
        if (st) bulk_g2s(smem, sc.tables, tb, bar);
        if (sg) {
            uint32_t pvb = sc.n_tris * 16u;
            bulk_g2s(smem + tb, sc.prim_verts, pvb, bar);
            bulk_g2s(smem + tb + pvb, sc.vertices, gb - pvb, bar);
        }
    }
    mbar_wait(bar, phase);
    if (st) {
        sc.shapes = (const DevShape *) smem; sc.bsdfs = (const DevBsdf *) (smem + sc.off_bsdfs);
        sc.emitters = (const DevEmitter *) (smem + sc.off_emitters); sc.textures = (const DevTexture *) (smem + sc.off_textures);
    }
    if (sg) { sc.prim_verts = (const uint4 *) (smem + tb); sc.vertices = (const float4 *) (smem + tb + sc.n_tris * 16u); }
}

// ---------------------------------------------------------------------------
// BVH traversal (bvh.h layout). The ray/triangle test is the reference's
// Moeller-Trumbore (mesh.h:1132-1153); boxes only cull.
// ---------------------------------------------------------------------------
struct Hit { float t, u, v; uint32_t prim; };

struct TraceCtx {
    const float4 *s_nodes, *s_tris;   // shared-memory copies (top of the tree / all triangles)
    const float4 *g_nodes, *g_tris;
    uint32_t n_smem_nodes, n_smem_tris;
};

// SMEM_ALL: the whole BVH and all triangles are staged (small scenes) -> plain LDS, no
// per-access shared/global selection (it costs ~12 address instructions per node visit).
template <bool SMEM_ALL>
PT_DEV float4 ld_node(const TraceCtx &c, uint32_t node, int k) {
    if (SMEM_ALL) return c.s_nodes[4 * node + k];
    return node < c.n_smem_nodes ? c.s_nodes[4 * node + k] : __ldg(&c.g_nodes[4 * (size_t) node + k]);
}
template <bool SMEM_ALL>
PT_DEV float4 ld_tri(const TraceCtx &c, uint32_t tri, int k) {
    if (SMEM_ALL) return c.s_tris[3 * tri + k];
    return tri < c.n_smem_tris ? c.s_tris[3 * tri + k] : __ldg(&c.g_tris[3 * (size_t) tri + k]);
}

PT_DEV float safe_inv(float d) { return fabsf(d) > 1e-30f ? __frcp_rn(d) : copysignf(1e30f, d); }

// Slab test of the tree walk, subtraction first (no cancellation against o * inv); the ray origin is live for the triangle
// test anyway, so this form costs the walk three registers (inv) where the fused one below costs seven.
PT_DEV bool box_hit(float lox, float loy, float loz, float hix, float hiy, float hiz, float3 o, float3 inv, float tmax, float &tnear) {
    float t0x = (lox - o.x) * inv.x, t1x = (hix - o.x) * inv.x;
    float t0y = (loy - o.y) * inv.y, t1y = (hiy - o.y) * inv.y;
    float t0z = (loz - o.z) * inv.z, t1z = (hiz - o.z) * inv.z;
    float tmin = fmaxf(fmaxf(fminf(t0x, t1x), fminf(t0y, t1y)), fmaxf(fminf(t0z, t1z), 0.f));
    float tmx = fminf(fminf(fmaxf(t0x, t1x), fmaxf(t0y, t1y)), fminf(fmaxf(t0z, t1z), tmax));
    tnear = tmin;
    return tmin <= tmx * 1.0000004f;
}

// Slab test in fused form (flat traversal, flat_phase: 18+ boxes per ray, registers to spare): t = lo * inv - (o * inv), one FFMA per
// plane instead of a subtraction and a multiplication. The product o * inv is rounded once per ray, so a plane distance is off
// by up to 2^-24 |o * inv| against the exact (lo - o) * inv; `slack` = 2^-22 max |o * inv| widens the interval test by more
// than twice that. The boxes only cull -- a hit is only ever decided by the reference's Moeller-Trumbore arithmetic -- so a
// wider test costs candidates (rays almost parallel to an axis stop culling on it), never a result.
// (In k_trace_dyn the four extra live registers of this form spill at its 48-register budget: Cornell 3.45 -> 3.34 ms per
//  launch, but the 205k-triangle scene 7.3 -> 8.2 ms; the walk keeps the form above. profiles/r02_summary.md)
struct RaySlabs { float3 inv, oi; float slack; };
PT_DEV RaySlabs make_slabs(float3 o, float3 d) {
    RaySlabs r;
    r.inv = V(safe_inv(d.x), safe_inv(d.y), safe_inv(d.z));
    r.oi = V(o.x * r.inv.x, o.y * r.inv.y, o.z * r.inv.z);
    r.slack = fmaxf(fmaxf(fabsf(r.oi.x), fabsf(r.oi.y)), fabsf(r.oi.z)) * 2.3841858e-7f;
    return r;
}

// Speculative while-while traversal (Aila & Laine, "Understanding the Efficiency of Ray
// Traversal on GPUs"): every lane walks inner nodes until it has found a leaf, postpones
// it and keeps walking until ALL lanes of the warp hold a leaf; then the warp tests
// triangles together. This keeps the two instruction streams (box tests / triangle
// tests) converged instead of interleaving them per lane.
constexpr int32_t TRAV_SENTINEL = 0x76543210;

template <bool ANY, bool SMEM_ALL>
PT_DEV bool traverse(const TraceCtx &c, float3 o, float3 d, float maxt, Hit &hit) {
    hit.t = PT_INF; hit.u = hit.v = 0.f; hit.prim = 0xffffffffu;
    float3 inv = V(safe_inv(d.x), safe_inv(d.y), safe_inv(d.z));
    int32_t stack[64]; stack[0] = TRAV_SENTINEL; int sp = 0;
    int32_t node = 0, leaf = 0;     // leaf >= 0: none postponed
    bool any = false;
    while (node != TRAV_SENTINEL) {
        bool searching = true;
        while (node >= 0 && node != TRAV_SENTINEL) {
            float4 n0 = ld_node<SMEM_ALL>(c, node, 0), n1 = ld_node<SMEM_ALL>(c, node, 1), n2 = ld_node<SMEM_ALL>(c, node, 2), n3 = ld_node<SMEM_ALL>(c, node, 3);
            int32_t cl = __float_as_int(n3.x), cr = __float_as_int(n3.y);
            float tl, tr;
            // both slab tests are evaluated unconditionally (no short-circuit branches); the
            // "no child" marker only exists in the synthetic root of a <= 2-triangle scene
            bool hl = box_hit(n0.x, n0.y, n0.z, n0.w, n1.x, n1.y, o, inv, maxt, tl) & (cl != 0x7fffffff);
            bool hr = box_hit(n1.z, n1.w, n2.x, n2.y, n2.z, n2.w, o, inv, maxt, tr) & (cr != 0x7fffffff);
            if (!hl && !hr) node = stack[sp--];
            else {
                node = hl ? cl : cr;
                if (hl && hr) {
                    int32_t far = cr;
                    if (tr < tl) { far = cl; node = cr; }
                    stack[++sp] = far;
                }
            }
            if (node < 0 && leaf >= 0) { searching = false; leaf = node; node = stack[sp--]; }   // postpone the first leaf
            if (!__any_sync(__activemask(), searching)) break;
        }
        while (leaf < 0) {
            uint32_t enc = (uint32_t) ~leaf, first = enc >> 3, count = (enc & 7u) + 1u;
            for (uint32_t i = first; i < first + count; ++i) {
                float4 a = ld_tri<SMEM_ALL>(c, i, 0), b = ld_tri<SMEM_ALL>(c, i, 1), e = ld_tri<SMEM_ALL>(c, i, 2);
                float t, u, v;
                if (moeller_trumbore(o, d, maxt, V(a.x, a.y, a.z), V(b.x, b.y, b.z), V(e.x, e.y, e.z), t, u, v)) {
                    if (ANY) return true;
                    uint32_t prim = __float_as_uint(a.w);
                    // closest hit; ties keep the smallest (shape, prim) index like a linear scan would
                    if (t < hit.t || (t == hit.t && prim < hit.prim)) { hit.t = t; hit.u = u; hit.v = v; hit.prim = prim; maxt = t; any = true; }
                }
            }
            leaf = node;
            if (node < 0) node = stack[sp--];
        }
    }
    return any;
}

// ---------------------------------------------------------------------------
// Flat traversal for scenes of at most FLAT_MAX_LEAVES leaves (the Cornell box: 36 triangles in 18 leaves). In a closed
// room the top of a binary tree culls nothing -- every inner box near the root spans the room -- so a walk spends ~10
// divergent node steps per ray before it reaches the two or three leaves that matter. Here every lane tests the boxes of
// ALL leaves in the same order instead (32 of 32 threads active, no stack), keeps the hit boxes as a bit mask, and then runs
// the reference's Moeller-Trumbore on the candidate leaves only (k_trace_flat, flat_phase). Results are those of any other
// traversal order: closest hit with ties resolved towards the smaller primitive index, any-hit a boolean.
// ---------------------------------------------------------------------------
constexpr uint32_t FLAT_MAX_LEAVES = 32;
constexpr uint32_t FLAT_UNROLL = 3;                 // leaves per iteration of the box pass; the list is padded to a multiple
constexpr uint32_t FLAT_LEAF_SLOTS = (FLAT_MAX_LEAVES + FLAT_UNROLL - 1) / FLAT_UNROLL * FLAT_UNROLL;
constexpr uint32_t FLAT_MAX_TRIS = 256;

// Leaf boxes ordered by direction octant: box[l][0][oct] holds the near-plane coordinates of leaf l for a ray whose inv
// has the sign bits oct (bit 0: x, 1: y, 2: z; a set bit makes `hi` the near plane of that axis), box[l][1][oct] the far
// ones. For inv >= 0, fma(lo, inv, -oi) <= fma(hi, inv, -oi) because rounding is monotone, and the reverse for inv < 0, so
// the near/far values are exactly what fminf / fmaxf of the two plane distances would pick: the box pass needs no per-axis
// min/max. The 8 copies of one leaf's near (far) planes fill one 128-byte line, so a warp's loads of one leaf never
// conflict, whatever mix of octants its rays hold. `.w` of the near copies is the leaf code (bvh.h), of the far copies
// the leaf index. Slots n .. n_pad-1 are empty boxes (lo = +inf, hi = -inf: the near distance is +inf, the far -inf,
// never a hit).
struct FlatLeaves { float4 box[FLAT_LEAF_SLOTS][2][8]; uint32_t n; };

PT_DEV void put_flat_leaf(FlatLeaves &L, uint32_t k, float3 lo, float3 hi, uint32_t code) {
    for (uint32_t oc = 0; oc < 8; ++oc) {
        const bool sx = oc & 1u, sy = oc & 2u, sz = oc & 4u;
        L.box[k][0][oc] = make_float4(sx ? hi.x : lo.x, sy ? hi.y : lo.y, sz ? hi.z : lo.z, __uint_as_float(code));
        L.box[k][1][oc] = make_float4(sx ? lo.x : hi.x, sy ? lo.y : hi.y, sz ? lo.z : hi.z, __uint_as_float(k));
    }
}

// Leaf list from the staged nodes (every negative child of an inner node is a leaf), padded to a multiple of FLAT_UNROLL,
// and the map primitive id -> staged triangle. Returns the padded leaf count.
PT_DEV uint32_t build_leaf_list(const float4 *s_nodes, uint32_t n_nodes, const float4 *s_tris, uint32_t n_tris, FlatLeaves &L, uint8_t *s_primmap) {
    if (threadIdx.x == 0) L.n = 0;
    __syncthreads();
    for (uint32_t node = threadIdx.x; node < n_nodes; node += blockDim.x) {
        float4 n0 = s_nodes[4 * node], n1 = s_nodes[4 * node + 1], n2 = s_nodes[4 * node + 2], n3 = s_nodes[4 * node + 3];
        int32_t cl = __float_as_int(n3.x), cr = __float_as_int(n3.y);
        if (cl < 0) { uint32_t k = atomicAdd(&L.n, 1u); if (k < FLAT_MAX_LEAVES) put_flat_leaf(L, k, V(n0.x, n0.y, n0.z), V(n0.w, n1.x, n1.y), (uint32_t) ~cl); }
        if (cr < 0) { uint32_t k = atomicAdd(&L.n, 1u); if (k < FLAT_MAX_LEAVES) put_flat_leaf(L, k, V(n1.z, n1.w, n2.x), V(n2.y, n2.z, n2.w), (uint32_t) ~cr); }
    }
    for (uint32_t i = threadIdx.x; i < n_tris; i += blockDim.x) s_primmap[__float_as_uint(s_tris[3 * i].w) & (FLAT_MAX_TRIS - 1u)] = (uint8_t) i;
    __syncthreads();
    const uint32_t n = min(L.n, FLAT_MAX_LEAVES), n_pad = (n + FLAT_UNROLL - 1) / FLAT_UNROLL * FLAT_UNROLL;
    if (threadIdx.x >= n && threadIdx.x < n_pad) put_flat_leaf(L, threadIdx.x, V(PT_INF, PT_INF, PT_INF), V(-PT_INF, -PT_INF, -PT_INF), 0u);
    __syncthreads();
    return n_pad;
}

// ---------------------------------------------------------------------------
// k_generate -- SamplingIntegrator::render JIT branch (integrator.cpp:322-339) +
// render_sample up to the sensor ray (integrator.cpp:461-485).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(BLOCK) k_generate(DevScene sc, RenderCfg cfg, const uint32_t *__restrict__ pix_ids, PathBuf buf,
                                                    const float4 *__restrict__ adj_dL_lane, const float4 *__restrict__ adj_L_lane) {
    uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < cfg.chunk_lanes; i += stride) {
        uint32_t lp = cfg.chunk_pix0 + i / cfg.spp, s = i % cfg.spp;
        uint32_t pixel = __ldg(&pix_ids[lp]);
        uint32_t lane = pixel * cfg.spp + s;
        uint32_t py = pixel / sc.crop_w, px = pixel - py * sc.crop_w;
        Pcg32 rng; rng.seed_lane(cfg.seed_value, lane);
        float u1 = rng.next_f32(), u2 = rng.next_f32();
        float posx = (float) (px + sc.crop_x) + u1, posy = (float) (py + sc.crop_y) + u2;
        float scx = fdiv(1.f, (float) sc.crop_w), scy = fdiv(1.f, (float) sc.crop_h);
        float ax = __fmaf_rn(posx, scx, -(float) sc.crop_x * scx), ay = __fmaf_rn(posy, scy, -(float) sc.crop_y * scy);
        Ray ray = sample_camera_ray(sc, ax, ay);
        buf.ray_o[i] = make_float4(ray.o.x, ray.o.y, ray.o.z, ray.maxt);
        buf.ray_d[i] = make_float4(ray.d.x, ray.d.y, ray.d.z, 1.f);        // prev_bsdf_pdf = 1
        buf.thr[i] = make_float4(1.f, 1.f, 1.f, 1.f);                      // throughput, eta
        buf.prev[i] = make_float4(0.f, 0.f, 0.f, __uint_as_float(PF_PREV_DELTA | PF_ALIVE));
        buf.rng[i] = make_uint4((uint32_t) rng.state, (uint32_t) (rng.state >> 32), lane, i);
        buf.result[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (buf.vis && !cfg.adjoint) buf.vis[i] = 0u;       // primal pass of a gradient call: NEE visibility bits for the replay
        if (cfg.adjoint) { buf.adj_L[i] = adj_L_lane[i]; buf.adj_dL[i] = cfg.forward ? make_float4(1.f, 1.f, 1.f, 0.f) : adj_dL_lane[i]; }
    }
}

// ---------------------------------------------------------------------------
// Traversal kernels. Per slot of the current buffer:
//   1. pending NEE shadow ray (Scene::ray_test, scene.cpp:232/344): unoccluded ->
//      result += contribution (path.cpp:279-280)
//   2. if the lane is alive: closest hit (scene.cpp:216) -> hit record, bin the slot
//      into the queue of the BSDF model it hit; a miss ends the path
//   3. finished lanes write their radiance to lane_result (consumed by k_splat)
// ---------------------------------------------------------------------------
// ---------------------------------------------------------------------------
// k_trace_flat -- the traversal kernel of scenes with at most FLAT_MAX_LEAVES leaves (see FlatLeaves). Same work per
// slot as k_trace, organised in warp-wide phases so that the exact triangle tests are shared by the whole warp:
//   box pass    every lane tests its own ray against all leaf boxes (32 of 32 threads, the octant's near / far planes:
//               2 LDS.128, 6 FFMA, 4 FMNMX, 1 FFMA, 1 FSETP and one predicated LOP3 per leaf) -> candidate mask
//   pair list   the (ray, leaf) candidates of the 32 rays are written to one list in shared memory (warp prefix sum)
//   test rounds lane j tests pairs j, j + 32, ...: the reference's Moeller-Trumbore on another lane's ray (the rays sit in
//               shared memory); closest hit = 64-bit atomicMin on (t bits, primitive id) per ray -- the same minimum and
//               the same tie-break as a serial scan, in any order; any-hit = a flag
//   winner      every lane repeats the test on its winning triangle to get (t, u, v): same inputs, same bits
// A serial per-lane candidate loop (ncu, profiles/r02_summary.md) ran the triangle tests at 4-9 of 32 threads and took 56 %
// of the kernel's instructions; the rounds run them at ~30 of 32.
// ---------------------------------------------------------------------------
constexpr uint32_t FLAT_PAIR_CAP = 32 * FLAT_MAX_LEAVES;      // candidate (ray, leaf) pairs of one warp and phase: every pair fits

struct FlatWarp {          // per-warp scratch in shared memory
    float4 ray[64];                        // (o, maxt), (d, -) of the 32 rays of the phase
    unsigned long long key[32];            // closest hit so far: (t bits << 32) | primitive id
    uint32_t occ[32];                      // any-hit flag
    uint16_t pairs[FLAT_PAIR_CAP];         // (ray << 8) | leaf
};

// One phase for the 32 rays of a warp; called by all 32 lanes at a converged point. ANY: returns "occluded"; otherwise the
// closest hit in `hit`.
// Closest hit tests the lane's nearest candidate leaf (smallest box entry distance) on the lane itself first and hands
// to the shared rounds only the candidates whose entry distance is at most lim = t * (1 + 2^-10) + slack, t the hit found
// there. A leaf beyond lim holds no hit at t or closer: the box pass culls against maxt with a margin of 4e-7 relative
// plus the same slack, and 2^-10 is more than 2000 times that. Hits at an equal t in a neighbouring leaf (shared edges,
// the corners of a room) stay inside the margin and meet the own hit in the same (t bits, primitive) minimum.
template <bool ANY>
PT_DEV bool flat_phase(FlatWarp &w, const FlatLeaves &L, uint32_t n_pad, const float4 *s_tris, const uint8_t *s_primmap,
                       bool active, float3 o, float3 d, float maxt, Hit &hit) {
    const uint32_t lane_id = threadIdx.x & 31u;
    hit.t = PT_INF; hit.u = hit.v = 0.f; hit.prim = 0xffffffffu;
    uint32_t mask = 0;
    unsigned long long own = ~0ull;            // closest hit in the nearest candidate leaf: (t bits << 32) | primitive id
    float own_t = 0.f, own_u = 0.f, own_v = 0.f;
    if (active) {
        const RaySlabs rs = make_slabs(o, d);
        const uint32_t oct = (__float_as_uint(rs.inv.x) >> 31) | (__float_as_uint(rs.inv.y) >> 31 << 1) | (__float_as_uint(rs.inv.z) >> 31 << 2);
        const float4 *bx = &L.box[0][0][oct];
        uint32_t nearest = ~0u;                // entry distance bits with the leaf index in the low 5 bits: the smallest wins
#pragma unroll 1
        for (uint32_t l = 0; l < n_pad; l += FLAT_UNROLL, bx += FLAT_UNROLL * 16) {
            uint32_t g = 0;
#pragma unroll
            for (uint32_t j = 0; j < FLAT_UNROLL; ++j) {
                // box_hit with the near / far plane of every axis known in advance: the same values, the same predicate
                const float4 nr = bx[16 * j], fr = bx[16 * j + 8];
                const float nx = __fmaf_rn(nr.x, rs.inv.x, -rs.oi.x), ny = __fmaf_rn(nr.y, rs.inv.y, -rs.oi.y), nz = __fmaf_rn(nr.z, rs.inv.z, -rs.oi.z);
                const float fx = __fmaf_rn(fr.x, rs.inv.x, -rs.oi.x), fy = __fmaf_rn(fr.y, rs.inv.y, -rs.oi.y), fz = __fmaf_rn(fr.z, rs.inv.z, -rs.oi.z);
                const float tmin = fmaxf(fmaxf(nx, ny), fmaxf(nz, 0.f)), tmx = fminf(fminf(fx, fy), fminf(fz, maxt));
                if (tmin <= __fmaf_rn(tmx, 1.0000004f, rs.slack)) {
                    g |= 1u << j;
                    if (!ANY) nearest = min(nearest, (__float_as_uint(tmin) & 0x7fffffe0u) | __float_as_uint(fr.w));
                }
            }
            mask |= g << l;
        }
        if (!ANY && mask) {
            const uint32_t l0 = nearest & 31u, enc = __float_as_uint(L.box[l0][0][0].w), t0 = enc >> 3, count = (enc & 7u) + 1u;
            mask &= ~(1u << l0);
            for (uint32_t ti = t0; ti < t0 + count; ++ti) {
                const float4 ta = s_tris[3 * ti], tb = s_tris[3 * ti + 1], te = s_tris[3 * ti + 2];
                float t, u, v;
                if (moeller_trumbore(o, d, maxt, V(ta.x, ta.y, ta.z), V(tb.x, tb.y, tb.z), V(te.x, te.y, te.z), t, u, v)) {
                    const unsigned long long k = ((unsigned long long) __float_as_uint(t + 0.f) << 32) | __float_as_uint(ta.w);
                    if (k < own) { own = k; own_t = t; own_u = u; own_v = v; }
                }
            }
            if (own != ~0ull) {
                const float lim = __fmaf_rn(__uint_as_float((uint32_t) (own >> 32)), 1.0009765625f, rs.slack);
                for (uint32_t m = mask; m; m &= m - 1u) {
                    const uint32_t l = (uint32_t) __ffs((int) m) - 1u;
                    const float4 nr = L.box[l][0][oct];
                    const float nx = __fmaf_rn(nr.x, rs.inv.x, -rs.oi.x), ny = __fmaf_rn(nr.y, rs.inv.y, -rs.oi.y), nz = __fmaf_rn(nr.z, rs.inv.z, -rs.oi.z);
                    if (fmaxf(fmaxf(nx, ny), fmaxf(nz, 0.f)) > lim) mask &= ~(1u << l);
                }
            }
        }
    }
    unsigned long long key = own;
    if (__any_sync(0xffffffffu, mask != 0u)) {
        if (mask) { w.ray[2 * lane_id] = make_float4(o.x, o.y, o.z, maxt); w.ray[2 * lane_id + 1] = make_float4(d.x, d.y, d.z, 0.f); }
        if (ANY) w.occ[lane_id] = 0u; else w.key[lane_id] = own;
        // exclusive prefix sum of the candidate counts
        const uint32_t cnt = (uint32_t) __popc(mask);
        uint32_t incl = cnt;
#pragma unroll
        for (int of = 1; of < 32; of <<= 1) { uint32_t v = __shfl_up_sync(0xffffffffu, incl, of); if ((int) lane_id >= of) incl += v; }
        const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
        {   // pair list: (ray << 8) | leaf
            uint32_t k = incl - cnt, m = mask;
            while (m) { uint32_t l = (uint32_t) __ffs((int) m) - 1u; m &= m - 1u; w.pairs[k++] = (uint16_t) ((lane_id << 8) | l); }
        }
        __syncwarp();
        for (uint32_t p = lane_id; p < total; p += 32u) {
            const uint32_t e = w.pairs[p], r = e >> 8, l = e & 255u;
            const float4 ro = w.ray[2 * r], rd = w.ray[2 * r + 1];
            const uint32_t enc = __float_as_uint(L.box[l][0][0].w), t0 = enc >> 3, count = (enc & 7u) + 1u;
            for (uint32_t ti = t0; ti < t0 + count; ++ti) {
                const float4 ta = s_tris[3 * ti], tb = s_tris[3 * ti + 1], te = s_tris[3 * ti + 2];
                float t, u, v;
                if (moeller_trumbore(V(ro.x, ro.y, ro.z), V(rd.x, rd.y, rd.z), ro.w, V(ta.x, ta.y, ta.z), V(tb.x, tb.y, tb.z), V(te.x, te.y, te.z), t, u, v)) {
                    if (ANY) w.occ[r] = 1u;
                    else atomicMin(&w.key[r], ((unsigned long long) __float_as_uint(t + 0.f) << 32) | __float_as_uint(ta.w));   // t >= 0: its bits order like its value; -0 -> +0
                }
            }
        }
        __syncwarp();
        if (ANY) return active && w.occ[lane_id] != 0u;
        key = w.key[lane_id];
    }
    if (ANY || !active || key == ~0ull) return false;
    if (key == own) { hit.t = own_t; hit.u = own_u; hit.v = own_v; hit.prim = (uint32_t) key; return true; }
    const uint32_t ti = s_primmap[(uint32_t) key];
    const float4 ta = s_tris[3 * ti], tb = s_tris[3 * ti + 1], te = s_tris[3 * ti + 2];
    float t, u, v;
    moeller_trumbore(o, d, maxt, V(ta.x, ta.y, ta.z), V(tb.x, tb.y, tb.z), V(te.x, te.y, te.z), t, u, v);     // the winner's (t, u, v): same inputs, same bits
    hit.t = t; hit.u = u; hit.v = v; hit.prim = (uint32_t) key;
    return true;
}

template <bool FIRST>
__global__ void __launch_bounds__(BLOCK, 4) k_trace_flat(const __grid_constant__ DevScene sc_in, RenderCfg cfg, PathBuf cur, float4 *__restrict__ hit_out, const uint32_t *__restrict__ n_in,
                                                         Queues q, uint32_t *__restrict__ qcounts, float4 *__restrict__ lane_result,
                                                         unsigned long long *__restrict__ stats, uint32_t n_smem_nodes, uint32_t n_smem_tris) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ uint64_t bar;
    __shared__ FlatLeaves s_leaves;
    __shared__ uint8_t s_primmap[FLAT_MAX_TRIS];
    __shared__ FlatWarp s_warp[BLOCK / 32];
    DevScene sc = sc_in;
    float4 *s_nodes = (float4 *) smem_raw;
    float4 *s_tris = s_nodes + 4 * (size_t) n_smem_nodes;
    if (threadIdx.x == 0) mbar_init(&bar, 1);
    __syncthreads();
    stage_bvh(sc, s_nodes, s_tris, n_smem_nodes, n_smem_tris, &bar);
    stage_tables(sc, smem_raw + ((n_smem_nodes * 64u + n_smem_tris * 48u + 127u) & ~127u), &bar, 1u);
    const uint32_t n_pad = build_leaf_list(s_nodes, n_smem_nodes, s_tris, n_smem_tris, s_leaves, s_primmap);
    FlatWarp &w = s_warp[threadIdx.x >> 5];

    const uint32_t n = FIRST ? cfg.chunk_lanes : *n_in;
    const uint32_t lane_id = threadIdx.x & 31u;
    const uint32_t warp_stride = gridDim.x * blockDim.x;
    uint32_t n_shadow = 0, n_closest = 0;
    for (uint32_t base = blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < n; base += warp_stride) {
        const uint32_t i = base + lane_id;
        const bool valid = i < n;
        const uint32_t flags = valid ? (FIRST ? PF_ALIVE : __float_as_uint(cur.prev[i].w)) : 0u;
        // ---- 1. pending NEE shadow rays (Scene::ray_test) ------------------------------------------------------------------
        const bool has_shadow = !FIRST && (flags & PF_HAS_SHADOW);
        float4 res = make_float4(0.f, 0.f, 0.f, 0.f);
        bool res_loaded = false;
        if (!FIRST && __any_sync(0xffffffffu, has_shadow)) {
            float4 so = make_float4(0.f, 0.f, 0.f, 0.f), sd = make_float4(0.f, 0.f, 1.f, 0.f);
            if (has_shadow) { so = cur.sh_o[i]; sd = cur.sh_d[i]; n_shadow++; }
            Hit hs;
            const bool occluded = flat_phase<true>(w, s_leaves, n_pad, s_tris, s_primmap, has_shadow, V(so.x, so.y, so.z), V(sd.x, sd.y, sd.z), so.w, hs);
            if (has_shadow && !occluded) {
                if (cur.vis) { uint32_t bit = (flags & PF_DEPTH_MASK) - 1u; if (bit < 32u) cur.vis[cur.rng[i].w] |= 1u << bit; }
                float2 c = cur.sh_c[i];
                res = cur.result[i]; res_loaded = true;
                res.x += sd.w; res.y += c.x; res.z += c.y;
                cur.result[i] = res;
            }
            __syncwarp();
        }
        // ---- 2. closest hit of the path rays (Scene::ray_intersect_preliminary) --------------------------------------------------
        bool alive = valid && (flags & PF_ALIVE);
        bool finished = valid && !alive;
        int mytype = -1;
        if (__any_sync(0xffffffffu, alive)) {
            float3 o = V(0.f, 0.f, 0.f), d = V(0.f, 0.f, 1.f); float maxt = 0.f;
            if (alive) { float4 ro = cur.ray_o[i], rd = cur.ray_d[i]; o = V(ro.x, ro.y, ro.z); d = V(rd.x, rd.y, rd.z); maxt = ro.w; n_closest++; }
            Hit h;
            bool found = flat_phase<false>(w, s_leaves, n_pad, s_tris, s_primmap, alive, o, d, maxt, h);
            if (FIRST && cfg.hide_emitters) {
                // skip_area_emitters (integrator.cpp:96-123): continue through directly visible emitters
                bool again = alive && found && sc.shapes[sc.prim_verts[h.prim].w].emitter >= 0;
                while (__any_sync(0xffffffffu, again)) {
                    if (again) {
                        SurfaceInteraction si = compute_si(sc, h.t, h.u, h.v, h.prim, d);
                        Ray r = spawn_ray(si.p, si.n, d);
                        o = r.o; maxt = r.maxt;
                        cur.ray_o[i] = make_float4(o.x, o.y, o.z, maxt);
                    }
                    __syncwarp();
                    Hit h2;
                    bool f2 = flat_phase<false>(w, s_leaves, n_pad, s_tris, s_primmap, again, o, d, maxt, h2);
                    if (again) { found = f2; h = h2; again = found && sc.shapes[sc.prim_verts[h.prim].w].emitter >= 0; }
                    __syncwarp();
                }
            }
            if (alive) {
                if (found) {
                    hit_out[i] = make_float4(h.t, h.u, h.v, __uint_as_float(h.prim));
                    const DevShape &sh = sc.shapes[sc.prim_verts[h.prim].w];
                    mytype = sc.bsdfs[sh.bsdf].type;
                } else if (sc.env_type >= 0) mytype = Q_ENV;   // the ray left the scene: environment emitter (k_shade_env)
                else finished = true;      // path.cpp:225: si invalid, no environment emitter
            }
        }
        if (finished) {
            if (!res_loaded) res = cur.result[i];
            lane_result[cur.rng[i].w] = res;
        }
        __syncwarp();
        // bucket pass: bin the slot by material id (one atomic per warp and material)
#pragma unroll
        for (int t = 0; t < N_QUEUES; ++t) {
            uint32_t m = __ballot_sync(0xffffffffu, mytype == t);
            if (m) {
                uint32_t leader = __ffs(m) - 1, off = 0;
                if (lane_id == leader) off = atomicAdd(&qcounts[t == Q_ENV ? QCOUNT_ENV : t], __popc(m));
                off = __shfl_sync(0xffffffffu, off, leader);
                if (mytype == t) q.slots[t][off + __popc(m & ((1u << lane_id) - 1u))] = i;
            }
        }
    }
    for (int o = 16; o; o >>= 1) { n_shadow += __shfl_xor_sync(0xffffffffu, n_shadow, o); n_closest += __shfl_xor_sync(0xffffffffu, n_closest, o); }
    if (lane_id == 0) {
        if (n_shadow) atomicAdd(&stats[ST_SHADOW], (unsigned long long) n_shadow);
        if (n_closest) atomicAdd(&stats[ST_CLOSEST], (unsigned long long) n_closest);
    }
}

// ---------------------------------------------------------------------------
// k_trace_dyn -- persistent-threads variant with dynamic work fetch (Aila & Laine).
// A warp keeps a pool of up to 32 "ray jobs" (one per lane). A job is a slot of the
// current buffer: its NEE shadow ray first (if any), then its path ray. Lanes that
// finish a job become idle; when enough lanes are idle the warp claims the next slots
// from a global counter (one atomicAdd per refill) instead of waiting for the slowest
// ray of the batch. The traversal itself is the same speculative while-while walk,
// resumable across refills (node / leaf / stack live in registers + local memory).
// Semantics per slot are those of k_trace_flat.
// ---------------------------------------------------------------------------

#ifndef TRACE_MIN_BLOCKS
#define TRACE_MIN_BLOCKS 5
#endif
template <bool FIRST, bool SMEM_ALL>
__global__ void __launch_bounds__(BLOCK, TRACE_MIN_BLOCKS) k_trace_dyn(const __grid_constant__ DevScene sc_in, RenderCfg cfg, PathBuf cur, float4 *__restrict__ hit_out,
                                                     const uint32_t *__restrict__ n_in, Queues q, uint32_t *__restrict__ qcounts, uint32_t *__restrict__ work_counter,
                                                     float4 *__restrict__ lane_result, unsigned long long *__restrict__ stats, uint32_t n_smem_nodes, uint32_t n_smem_tris, int DYN_REFILL_IDLE) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ uint64_t bar;
    __shared__ uint32_t s_pool_open;
    DevScene sc = sc_in;
    float4 *s_nodes = (float4 *) smem_raw;
    float4 *s_tris = s_nodes + 4 * (size_t) n_smem_nodes;
    const uint32_t n = FIRST ? cfg.chunk_lanes : *n_in;
    if (threadIdx.x == 0) {
        mbar_init(&bar, 1);
        // a block that becomes resident late (another stream's kernels held the SM) finds the pool already claimed: it
        // leaves before staging anything
        s_pool_open = *(volatile uint32_t *) work_counter < n ? 1u : 0u;
    }
    __syncthreads();
    if (!s_pool_open) return;
    stage_bvh(sc, s_nodes, s_tris, n_smem_nodes, n_smem_tris, &bar);
    stage_tables(sc, smem_raw + ((n_smem_nodes * 64u + n_smem_tris * 48u + 127u) & ~127u), &bar, 1u);
    TraceCtx c = { s_nodes, s_tris, sc.nodes, sc.tris, n_smem_nodes, n_smem_tris };

    const uint32_t lane_id = threadIdx.x & 31u;
    uint32_t n_shadow = 0, n_closest = 0;

    // job state of this lane
    int kind = 0;                     // 0 idle, 1 shadow ray, 2 path ray
    uint32_t slot = 0, flags = 0;
    float3 o = V(0.f, 0.f, 0.f), d = V(0.f, 0.f, 1.f), inv = V(0.f, 0.f, 0.f);
    float maxt = 0.f;
    Hit hit; hit.t = PT_INF; hit.u = hit.v = 0.f; hit.prim = 0xffffffffu;
    int32_t stack[64]; int sp = 0; int32_t node = TRAV_SENTINEL, leaf = 0;
    bool occluded = false;
    bool exhausted = false;           // the global pool is empty
#ifdef B200PT_WATCHDOG
    uint32_t wd_steps = 0;
#endif

    auto start_ray = [&](float3 ro, float3 rd, float rmaxt) {
        o = ro; d = rd; maxt = rmaxt;
        inv = V(safe_inv(d.x), safe_inv(d.y), safe_inv(d.z));
        hit.t = PT_INF; hit.u = hit.v = 0.f; hit.prim = 0xffffffffu;
        stack[0] = TRAV_SENTINEL; sp = 0; node = 0; leaf = 0; occluded = false;
#ifdef B200PT_WATCHDOG
        wd_steps = 0;
#endif
    };
#ifdef B200PT_WATCHDOG
    uint32_t wd_rounds = 0;
#endif

    while (true) {
#ifdef B200PT_WATCHDOG
        if (++wd_rounds > (1u << 24)) { if (lane_id == 0) atomicAdd(&g_watchdog[2], 1ull); break; }
#endif
        // ---- refill idle lanes from the global pool --------------------------------------
        uint32_t idle_mask = __ballot_sync(0xffffffffu, kind == 0);
        if (!exhausted && (__popc(idle_mask) >= DYN_REFILL_IDLE)) {
            uint32_t cnt = __popc(idle_mask), base = 0;
            if (lane_id == 0) base = atomicAdd(work_counter, cnt);
            base = __shfl_sync(0xffffffffu, base, 0);
            if (base + cnt >= n) exhausted = true;
            if (kind == 0) {
                uint32_t i = base + __popc(idle_mask & ((1u << lane_id) - 1u));
                if (i < n) {
                    const uint32_t si = i;
                    slot = si;
                    flags = FIRST ? PF_ALIVE : __float_as_uint(cur.prev[si].w);
                    if (!FIRST && (flags & PF_HAS_SHADOW)) {
                        float4 so = cur.sh_o[si], sd = cur.sh_d[si];
                        kind = 1; n_shadow++;
                        start_ray(V(so.x, so.y, so.z), V(sd.x, sd.y, sd.z), so.w);
                    } else {       // every queued slot is alive or has a shadow ray
                        float4 ro = cur.ray_o[si], rd = cur.ray_d[si];
                        kind = 2; n_closest++;
                        start_ray(V(ro.x, ro.y, ro.z), V(rd.x, rd.y, rd.z), ro.w);
                    }
                }
            }
        }
        if (!__any_sync(0xffffffffu, kind != 0)) break;

        // ---- traverse until this lane's ray is done or the warp wants to refill -----------
        // (lanes run these loops divergently on purpose: with a full-mask vote per node step -- measured, profiles/r02_summary.md --
        //  every step waits for the slowest lane's node fetch, 11 % slower on the 205k-triangle scene whose nodes come from L2)
        if (kind != 0) {
            while (node != TRAV_SENTINEL) {
                bool searching = true;
                while (node >= 0 && node != TRAV_SENTINEL) {
                    float4 n0 = ld_node<SMEM_ALL>(c, node, 0), n1 = ld_node<SMEM_ALL>(c, node, 1), n2 = ld_node<SMEM_ALL>(c, node, 2), n3 = ld_node<SMEM_ALL>(c, node, 3);
                    int32_t cl = __float_as_int(n3.x), cr = __float_as_int(n3.y);
                    float tl, tr;
                    bool hl = box_hit(n0.x, n0.y, n0.z, n0.w, n1.x, n1.y, o, inv, maxt, tl) & (cl != 0x7fffffff);
                    bool hr = box_hit(n1.z, n1.w, n2.x, n2.y, n2.z, n2.w, o, inv, maxt, tr) & (cr != 0x7fffffff);
                    if (!hl && !hr) node = stack[sp--];
                    else {
                        node = hl ? cl : cr;
                        if (hl && hr) {
                            int32_t far = cr;
                            if (tr < tl) { far = cl; node = cr; }
                            stack[++sp] = far;
                        }
                    }
                    if (node < 0 && leaf >= 0) { searching = false; leaf = node; node = stack[sp--]; }
#ifdef B200PT_WATCHDOG
                    if (++wd_steps > 200000u) { atomicAdd(&g_watchdog[1], 1ull); node = TRAV_SENTINEL; leaf = 0; wd_steps = 0; }
#endif
                    if (!__any_sync(__activemask(), searching)) break;
                }
                while (leaf < 0) {
                    uint32_t enc = (uint32_t) ~leaf, first = enc >> 3, count = (enc & 7u) + 1u;
                    for (uint32_t i = first; i < first + count; ++i) {
                        float4 a = ld_tri<SMEM_ALL>(c, i, 0), b = ld_tri<SMEM_ALL>(c, i, 1), e = ld_tri<SMEM_ALL>(c, i, 2);
                        float t, u, v;
                        if (moeller_trumbore(o, d, maxt, V(a.x, a.y, a.z), V(b.x, b.y, b.z), V(e.x, e.y, e.z), t, u, v)) {
                            uint32_t prim = __float_as_uint(a.w);
                            if (kind == 1) { occluded = true; }
                            else if (t < hit.t || (t == hit.t && prim < hit.prim)) { hit.t = t; hit.u = u; hit.v = v; hit.prim = prim; maxt = t; }
                        }
                    }
                    leaf = node;
                    if (node < 0) node = stack[sp--];
                    if (occluded) { node = TRAV_SENTINEL; leaf = 0; }     // any-hit: stop at the first occluder
                }
                // dynamic fetch: leave the loop when too few lanes of the warp are still walking
                if (!exhausted && __popc(__activemask()) < 32 - DYN_REFILL_IDLE) break;
            }
        }
        __syncwarp();

        // ---- retire finished rays -----------------------------------------------------------
        int mytype = -1;
        if (kind != 0 && node == TRAV_SENTINEL) {
            if (kind == 1) {
                if (!occluded) {
                    if (cur.vis) { uint32_t bit = (flags & PF_DEPTH_MASK) - 1u; if (bit < 32u) cur.vis[cur.rng[slot].w] |= 1u << bit; }
                    float4 sd = cur.sh_d[slot]; float2 cc = cur.sh_c[slot]; float4 res = cur.result[slot];
                    res.x += sd.w; res.y += cc.x; res.z += cc.y;
                    cur.result[slot] = res;
                }
                if (flags & PF_ALIVE) {
                    float4 ro = cur.ray_o[slot], rd = cur.ray_d[slot];
                    kind = 2; n_closest++;
                    start_ray(V(ro.x, ro.y, ro.z), V(rd.x, rd.y, rd.z), ro.w);
                } else {
                    lane_result[cur.rng[slot].w] = cur.result[slot];
                    kind = 0;
                }
            } else {
                bool found = hit.prim != 0xffffffffu;
                if (FIRST && cfg.hide_emitters && found && sc.shapes[sc.prim_verts[hit.prim].w].emitter >= 0) {
                    // skip_area_emitters (integrator.cpp:96-123)
                    SurfaceInteraction si = compute_si(sc, hit.t, hit.u, hit.v, hit.prim, d);
                    Ray r = spawn_ray(si.p, si.n, d);
                    cur.ray_o[slot] = make_float4(r.o.x, r.o.y, r.o.z, r.maxt);
                    start_ray(r.o, d, r.maxt);
                } else {
                    if (found) {
                        hit_out[slot] = make_float4(hit.t, hit.u, hit.v, __uint_as_float(hit.prim));
                        mytype = sc.bsdfs[sc.shapes[sc.prim_verts[hit.prim].w].bsdf].type;
                    } else if (sc.env_type >= 0) mytype = Q_ENV;     // the ray left the scene: environment emitter (k_shade_env)
                    else lane_result[cur.rng[slot].w] = cur.result[slot];
                    kind = 0;
                }
            }
        }
        __syncwarp();
#pragma unroll
        for (int t = 0; t < N_QUEUES; ++t) {
            uint32_t m = __ballot_sync(0xffffffffu, mytype == t);
            if (m) {
                uint32_t leader = __ffs(m) - 1, off = 0;
                if (lane_id == leader) off = atomicAdd(&qcounts[t == Q_ENV ? QCOUNT_ENV : t], __popc(m));
                off = __shfl_sync(0xffffffffu, off, leader);
                if (mytype == t) q.slots[t][off + __popc(m & ((1u << lane_id) - 1u))] = slot;
            }
        }
    }
    for (int of = 16; of; of >>= 1) { n_shadow += __shfl_xor_sync(0xffffffffu, n_shadow, of); n_closest += __shfl_xor_sync(0xffffffffu, n_closest, of); }
    if (lane_id == 0) {
        if (n_shadow) atomicAdd(&stats[ST_SHADOW], (unsigned long long) n_shadow);
        if (n_closest) atomicAdd(&stats[ST_CLOSEST], (unsigned long long) n_closest);
    }
}

// ---------------------------------------------------------------------------
// Warp-cooperative fp32 gradient scatter (adjoint of tex_eval3). Called by all 32
// lanes at a converged point; lanes without a request pass tex = -1. Lanes that
// target the same texel are combined with __match_any_sync + shuffles so that the
// texture receives ONE atomicAdd per distinct (texel, channel) and warp -- the
// contention fix for few-texel parameters (constant albedo = 3 floats).
// (Measured in round 2 and NOT kept: a butterfly reduction per distinct single-target texture plus plain atomics for bitmap taps
//  45.2 ms, the same with the match/shuffle path kept for bitmaps 44.2 ms, against 39.7 ms for this version on the configs[2]
//  gradient step -- the adjoint kernel runs at its 128-register budget with spills, and the longer code costs more there than the
//  32-step peer loop of the all-lanes-one-target case. profiles/r02_summary.md section 6.)
// ---------------------------------------------------------------------------
PT_DEV void warp_scatter3(const DevScene &sc, int32_t tex, float2 uv, float3 g) {
    const uint32_t lane_id = threadIdx.x & 31u;
    bool has = tex >= 0 && sc.textures[tex >= 0 ? tex : 0].differentiable && (g.x != 0.f || g.y != 0.f || g.z != 0.f);
    if (!__any_sync(0xffffffffu, has)) return;
    TexTaps tp; tp.n = 0;
    int C = 3; float *grad = nullptr; bool is_const = false;
    if (has) {
        const DevTexture &t = sc.textures[tex];
        C = t.channels; grad = sc.grad + t.grad_offset;
        if (t.kind == B200PT_TEX_CONST) { tp.n = 1; tp.idx[0] = 0; tp.w[0] = 1.f; is_const = true; }
        else if (t.kind == B200PT_TEX_CHECKERBOARD) { tp.n = 1; tp.idx[0] = checker_masks_equal(t, uv) ? 0 : 1; tp.w[0] = 1.f; }
        else tex_lookup(t, uv, tp);
    }
    for (int k = 0; k < 4; ++k) {
        bool hk = has && k < tp.n;
        if (!__any_sync(0xffffffffu, hk)) break;
        unsigned long long key = hk ? (((unsigned long long) (uint32_t) tex << 32) | (uint32_t) tp.idx[k]) : ~0ull;
        uint32_t peers = __match_any_sync(0xffffffffu, key);
        float w = hk ? tp.w[k] : 0.f;
        float v0 = g.x * w, v1 = g.y * w, v2 = g.z * w;
        uint32_t leader = __ffs(peers) - 1;
        float s0 = 0.f, s1 = 0.f, s2 = 0.f;
        for (uint32_t m = peers; m; m &= m - 1) {
            int src = __ffs(m) - 1;
            s0 += __shfl_sync(peers, v0, src); s1 += __shfl_sync(peers, v1, src); s2 += __shfl_sync(peers, v2, src);
        }
        if (hk && lane_id == leader) {
            if (C == 1) atomicAdd(grad + (is_const ? 0 : tp.idx[k]), s0 + s1 + s2);
            else { float *gp = grad + (size_t) tp.idx[k] * 3; atomicAdd(gp, s0); atomicAdd(gp + 1, s1); atomicAdd(gp + 2, s2); }
        }
    }
}

// Forward mode: the contraction of a scatter request (tex, uv, g) with the parameter tangents,
// i.e. sum_texels w * g (.) d(parameter)[texel] -- the transpose of warp_scatter3.
PT_DEV float3 tangent_dot(const DevScene &sc, int32_t tex, float2 uv, float3 g) {
    if (tex < 0) return V(0.f, 0.f, 0.f);
    const DevTexture &t = sc.textures[tex];
    if (!t.differentiable) return V(0.f, 0.f, 0.f);
    TexTaps tp; tp.n = 0;
    if (t.kind == B200PT_TEX_CONST) { tp.n = 1; tp.idx[0] = 0; tp.w[0] = 1.f; }
    else if (t.kind == B200PT_TEX_CHECKERBOARD) { tp.n = 1; tp.idx[0] = checker_masks_equal(t, uv) ? 0 : 1; tp.w[0] = 1.f; }
    else tex_lookup(t, uv, tp);
    const float *tg = sc.tangent + t.grad_offset;
    int C = t.channels;
    float3 acc = V(0.f, 0.f, 0.f);
    for (int k = 0; k < tp.n; ++k) {
        const float *q = tg + (size_t) tp.idx[k] * C;
        float3 tv = C == 1 ? V(q[0], q[0], q[0]) : V(q[0], q[1], q[2]);
        acc = V(__fmaf_rn(tp.w[k] * tv.x, g.x, acc.x), __fmaf_rn(tp.w[k] * tv.y, g.y, acc.y), __fmaf_rn(tp.w[k] * tv.z, g.z, acc.z));
    }
    return acc;
}

// BSDF parameter adjoint at one vertex (prb.py:263-313 restricted to texture parameters):
//   d/dtheta [ g_dir . f(wo_em; theta) + g_ind . f(wo_s; theta) / f(wo_s) ]
// Returns the gradient w.r.t. the (single) differentiable colour texture of the model and its slot.
template <int TYPE>
PT_DEV float3 bsdf_backward(const DevScene &sc, const DevBsdf &b, float2 uv, float3 wi, float3 wo_em, float3 wo_s, float3 g_dir, float3 g_ind, int32_t &tex) {
    tex = -1;
    if (b.twosided && wi.z < 0.f) { wi.z = -wi.z; wo_em.z = -wo_em.z; wo_s.z = -wo_s.z; }
    if (TYPE == B200PT_BSDF_DIFFUSE) {
        tex = b.tex[B200PT_SLOT_REFLECTANCE];
        float3 rho = tex_eval3(sc, tex, uv);
        float3 g = V(0.f, 0.f, 0.f);
        if (wi.z > 0.f && wo_em.z > 0.f) g = g_dir * (PT_INV_PI * wo_em.z);
        if (wi.z > 0.f && wo_s.z > 0.f)
            g = g + V(rho.x != 0.f ? fdiv(g_ind.x, rho.x) : 0.f, rho.y != 0.f ? fdiv(g_ind.y, rho.y) : 0.f, rho.z != 0.f ? fdiv(g_ind.z, rho.z) : 0.f);
        return g;
    }
    return V(0.f, 0.f, 0.f);
}

// ---------------------------------------------------------------------------
// k_shade<TYPE> -- loop body of PathIntegrator::sample (path.cpp:193-340) /
// PRBIntegrator.sample (prb.py:125-333) for the lanes whose hit has BSDF model
// TYPE. ADJOINT = PRB backward pass: replays the path, resolves the NEE
// visibility inline and scatters the parameter gradients (prb.py:263-313).
// ---------------------------------------------------------------------------
#ifndef SHADE_MIN_BLOCKS
#define SHADE_MIN_BLOCKS 4
#endif
// ADJ: 0 primal; 1 adjoint / forward replay that resolves the NEE visibility with an inline any-hit walk; 2 replay that
// reads the visibility bits the primal pass of the same call recorded (PathBuf::vis, one bit per bounce, max_depth <= 32):
// no walk, no BVH in shared memory, twice the occupancy.
template <int TYPE, int ADJ, bool EXT>
__global__ void __launch_bounds__(BLOCK_SHADE, ADJ == 1 ? 2 : (ADJ == 2 ? (TYPE == B200PT_BSDF_DIFFUSE ? 4 : 2) : SHADE_MIN_BLOCKS)) k_shade(const __grid_constant__ DevScene sc_in, RenderCfg cfg, PathBuf cur, const float4 *__restrict__ hit_in,
                                                 const uint32_t *__restrict__ queue, const uint32_t *__restrict__ qcount, PathBuf nxt,
                                                 uint32_t *__restrict__ nxt_count, float4 *__restrict__ lane_result,
                                                 unsigned long long *__restrict__ stats, uint32_t n_smem_nodes, uint32_t n_smem_tris) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ uint64_t bar;
    constexpr bool ADJOINT = ADJ != 0;
    DevScene sc = sc_in;
    TraceCtx ctx = { nullptr, nullptr, sc.nodes, sc.tris, 0, 0 };
    if (threadIdx.x == 0) mbar_init(&bar, 1);
    __syncthreads();
    uint32_t bvh_bytes = 0;
    if (ADJ == 1) {
        float4 *s_nodes = (float4 *) smem_raw;
        float4 *s_tris = s_nodes + 4 * (size_t) n_smem_nodes;
        stage_bvh(sc, s_nodes, s_tris, n_smem_nodes, n_smem_tris, &bar);
        ctx.s_nodes = s_nodes; ctx.s_tris = s_tris; ctx.n_smem_nodes = n_smem_nodes; ctx.n_smem_tris = n_smem_tris;
        bvh_bytes = (n_smem_nodes * 64u + n_smem_tris * 48u + 127u) & ~127u;
    }
    stage_tables(sc, smem_raw + bvh_bytes, &bar, ADJ == 1 ? 1u : 0u);
    const uint32_t n = *qcount;
    const uint32_t lane_id = threadIdx.x & 31u;
    const uint32_t warp_stride = gridDim.x * blockDim.x;
    const bool prb = cfg.prb != 0;
    const bool fwd = ADJOINT && cfg.forward != 0;     // forward-mode replay: `result` carries the sample's dL
    uint32_t n_bounces = 0, n_shadow = 0;
    for (uint32_t base = blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < n; base += warp_stride) {
        uint32_t qi = base + lane_id;
        bool valid = qi < n;
        bool write_next = false;
        // state of the lane after this vertex
        float4 o_ro, o_rd, o_thr, o_prev, o_res, o_sho, o_shd, o_L, o_dL; float2 o_shc; uint4 o_rng;
        // gradient scatter requests of this vertex (adjoint)
        int32_t gt0 = -1, gt1 = -1, gt2 = -1; float2 guv0 = make_float2(0.f, 0.f), guv1 = guv0, guv2 = guv0;
        float3 gv0 = V(0.f, 0.f, 0.f), gv1 = gv0, gv2 = gv0;
        // non-diffuse models: the BSDF-parameter derivatives of this vertex are evaluated slot by slot at the converged
        // point below (pt_bsdf_grad.cuh); what they need is kept here
        int32_t pg_bsdf = -1; bool pg_dir = false, pg_ind = false;
        float3 pg_wi = V(0.f, 0.f, 1.f), pg_wo_em = pg_wi, pg_wo_s = pg_wi, pg_adir = V(0.f, 0.f, 0.f), pg_aind = pg_adir;
        if (valid) {
            n_bounces++;
            uint32_t slot = __ldg(&queue[qi]);
            float4 rd = cur.ray_d[slot], th = cur.thr[slot], pv = cur.prev[slot], hr = hit_in[slot], res = cur.result[slot];
            uint4 rs = cur.rng[slot];
            float3 ray_d = V(rd.x, rd.y, rd.z);
            float prev_bsdf_pdf = rd.w;
            float3 throughput = V(th.x, th.y, th.z); float eta = th.w;
            float3 prev_p = V(pv.x, pv.y, pv.z);
            uint32_t flags = __float_as_uint(pv.w), depth = flags & PF_DEPTH_MASK;
            bool prev_delta = (flags & PF_PREV_DELTA) != 0;
            float3 result = V(res.x, res.y, res.z);
            Pcg32 rng; rng.restore(cfg.seed_value, rs.z, ((uint64_t) rs.y << 32) | rs.x);
            float3 L = V(0.f, 0.f, 0.f), dL = V(0.f, 0.f, 0.f);
            if (ADJOINT) { float4 a = cur.adj_L[slot], b = cur.adj_dL[slot]; L = V(a.x, a.y, a.z); dL = V(b.x, b.y, b.z); }

            SurfaceInteraction si = compute_si(sc, hr.x, hr.y, hr.z, __float_as_uint(hr.w), ray_d);
            const DevShape &sh = sc.shapes[si.shape];
            const DevBsdf &bsdf = sc.bsdfs[sh.bsdf];

            // ---- direct emission (path.cpp:206-222, prb.py:151-163)
            float3 Le = V(0.f, 0.f, 0.f);
            if (sh.emitter >= 0) {
                float3 rel = si.p - prev_p;
                float dist = __fsqrt_rn(vsqnorm(rel));
                float3 d = V(fdiv(rel.x, dist), fdiv(rel.y, dist), fdiv(rel.z, dist));
                float em_pdf = prev_delta ? 0.f : pdf_emitter_direction(sc, sh.emitter, d, si.sh_n, dist);
                float mis_bsdf = mis_weight(prev_bsdf_pdf, em_pdf);
                bool em_active = si.wi.z > 0.f && (prb || prev_bsdf_pdf > 0.f);
                float3 rad = em_active ? tex_eval3(sc, sc.emitters[sh.emitter].radiance_tex, si.uv) : V(0.f, 0.f, 0.f);
                if (prb) { Le = (throughput * mis_bsdf) * rad; if (!fwd) result = result + Le; }
                else { Le = throughput * (rad * mis_bsdf); result = vfma(throughput, rad * mis_bsdf, result); }
                if (ADJOINT && em_active) { gt0 = sc.emitters[sh.emitter].radiance_tex; guv0 = si.uv; gv0 = dL * (throughput * mis_bsdf); }
            }
            bool active_next = depth + 1 < cfg.max_depth;
            if (!active_next) {
                if (fwd) result = result + tangent_dot(sc, gt0, guv0, gv0);     // forward mode: dLe
                if (!ADJOINT || fwd) lane_result[rs.w] = make_float4(result.x, result.y, result.z, 0.f);
                if (fwd) gt0 = -1;
            } else {
                // ---- emitter sampling (path.cpp:238-259): the two randoms are always drawn (JIT semantics)
                const bool smooth = TYPE == B200PT_BSDF_DIFFUSE || TYPE == B200PT_BSDF_PRINCIPLED || (bsdf.flags & (B200PT_M_ROUGH | PT_M_PLASTIC));   // BSDFFlags::Smooth (path.cpp:238)
                float ex = rng.next_f32(), ey = rng.next_f32();
                DirectionSample ds; ds.pdf = 0.f; ds.emitter = -1; ds.uv = make_float2(0.f, 0.f);
                float3 em_weight = V(0.f, 0.f, 0.f), wo = V(0.f, 0.f, 0.f);
                bool active_em = false;
                Ray sray; sray.o = V(0.f, 0.f, 0.f); sray.d = V(0.f, 0.f, 0.f); sray.maxt = 0.f;
                if (smooth) {
                    em_weight = sample_emitter_direction<EXT>(sc, si.p, ex, ey, ds);
                    active_em = ds.pdf != 0.f;
                    wo = si.to_local(ds.d);
                    if (ADJOINT && active_em) {
                        // the adjoint needs Lr_dir now (prb.py:227)
                        bool occluded;
                        if (ADJ == 2) occluded = !((cur.vis[rs.w] >> depth) & 1u);      // recorded by the primal pass of this call (k_trace*)
                        else {                                                           // resolve the visibility inline
                            sray = spawn_ray_to(si.p, si.n, ds.p);
                            Hit h; n_shadow++;
                            occluded = traverse<true, false>(ctx, sray.o, sray.d, sray.maxt, h);
                        }
                        if (occluded) { em_weight = V(0.f, 0.f, 0.f); ds.pdf = 0.f; active_em = false; }
                    }
                }
                // ---- BSDF (path.cpp:263-267)
                float s1 = rng.next_f32(), s2x = rng.next_f32(), s2y = rng.next_f32();
                BsdfResult br = bsdf_eval_pdf_sample<TYPE>(sc, bsdf, si.uv, si.wi, wo, s1, s2x, s2y);
                // NEE contribution (path.cpp:271-281); in the primal passes its visibility is resolved by the next k_trace
                bool has_shadow = false; float3 contrib = V(0.f, 0.f, 0.f); float mis_em = 0.f;
                if (active_em) {
                    mis_em = mis_weight(ds.pdf, br.pdf);
                    contrib = prb ? ((throughput * mis_em) * br.value) * em_weight : throughput * ((br.value * em_weight) * mis_em);
                    if (!ADJOINT) {
                        // (a pass that records visibility for the replay traces every NEE ray: a zero contribution can
                        //  still have a non-zero parameter derivative)
                        has_shadow = contrib.x != 0.f || contrib.y != 0.f || contrib.z != 0.f || cur.vis != nullptr;
                        if (has_shadow) sray = spawn_ray_to(si.p, si.n, ds.p);
                    }
                }
                // ---- BSDF sampling (path.cpp:285-313)
                Ray next = spawn_ray(si.p, si.n, si.to_world(br.bs.wo));
                float3 beta_vertex = throughput;
                throughput = throughput * br.weight;
                eta *= br.bs.eta;
                // ---- russian roulette (path.cpp:317-331 / prb.py:241-252: prb tests the pre-increment depth)
                float tmax = vmaxc(throughput);
                float rr_prob = fminf(tmax * sqr(eta), .95f);
                bool rr_active = prb ? depth >= cfg.rr_depth : depth + 1 >= cfg.rr_depth;
                bool rr_continue;
                if (prb) { if (rr_active) throughput = throughput * rcp_(rr_prob); rr_continue = rng.next_f32() < rr_prob; }
                else { rr_continue = rng.next_f32() < rr_prob; if (rr_active) throughput = throughput * rcp_(rr_prob); }
                bool active = (!rr_active || rr_continue) && tmax != 0.f;
                if (ADJOINT) {
                    float3 Lr_dir = active_em ? contrib : V(0.f, 0.f, 0.f);
                    L = (L - Le) - Lr_dir;                                            // prb.py:227
                    float3 g_dir = active_em ? dL * ((beta_vertex * mis_em) * em_weight) : V(0.f, 0.f, 0.f);
                    float3 g_ind = active ? dL * L : V(0.f, 0.f, 0.f);
                    guv1 = si.uv;
                    if (TYPE == B200PT_BSDF_DIFFUSE) gv1 = bsdf_backward<TYPE>(sc, bsdf, si.uv, si.wi, wo, br.bs.wo, g_dir, g_ind, gt1);
                    else {
                        pg_bsdf = sh.bsdf; pg_dir = active_em; pg_ind = active; pg_adir = g_dir; pg_aind = g_ind;
                        pg_wi = si.wi; pg_wo_em = wo; pg_wo_s = br.bs.wo;
                        if (bsdf.twosided && si.wi.z < 0.f) { pg_wi.z = -pg_wi.z; pg_wo_em.z = -pg_wo_em.z; pg_wo_s.z = -pg_wo_s.z; }
                        if (fwd) {
                            // forward mode (dL = 1, so a_dir / a_ind are per-channel coefficients): d(radiance) of this vertex
                            // = sum over parameter channels of coefficient x the parameter's tangent at this texture position
                            for (int k = 0; k < B200PT_MAX_SLOTS; ++k) {
                                int32_t pt = bsdf_grad_slot(sc, bsdf, k);
                                if (pt < 0) continue;
                                const int nch = sc.textures[pt].channels;
                                for (int ch = 0; ch < nch; ++ch) {
                                    float3 cf = bsdf_param_coeff<TYPE>(sc, bsdf, si.uv, pg_wi, pg_wo_em, pg_wo_s, pg_adir, pg_aind, pg_dir, pg_ind, pt, ch);
                                    float3 e = V(ch == 0 ? 1.f : 0.f, ch == 1 ? 1.f : 0.f, ch == 2 ? 1.f : 0.f);
                                    float3 td = tangent_dot(sc, pt, si.uv, e);
                                    result = result + cf * (nch == 1 ? td.x : (ch == 0 ? td.x : ch == 1 ? td.y : td.z));
                                }
                            }
                            pg_bsdf = -1;
                        }
                    }
                    if (active_em) {
                        // emitter radiance inside em_weight = radiance / pdf (area.cpp:161, envmap.cpp:374-377;
                        // the sampling density is detached); envmap: rad = scale * sum_taps w * data[texel]
                        int32_t rt = sc.emitters[ds.emitter].radiance_tex;
                        bool is_env = sc.emitters[ds.emitter].type == B200PT_EMITTER_ENVMAP;
                        float3 rad = is_env ? env_eval_spectrum(*sc.env, ds.uv.x, ds.uv.y) : tex_eval3(sc, rt, ds.uv);
                        if (is_env) Lr_dir = Lr_dir * sc.env_scale;
                        gt2 = rt; guv2 = ds.uv;
                        gv2 = dL * V(rad.x != 0.f ? fdiv(Lr_dir.x, rad.x) : 0.f, rad.y != 0.f ? fdiv(Lr_dir.y, rad.y) : 0.f, rad.z != 0.f ? fdiv(Lr_dir.z, rad.z) : 0.f);
                    }
                }
                if (fwd) {
                    // forward mode: dL of this vertex = <derivative coefficients, parameter tangents>
                    result = result + tangent_dot(sc, gt0, guv0, gv0) + tangent_dot(sc, gt1, guv1, gv1) + tangent_dot(sc, gt2, guv2, gv2);
                    gt0 = gt1 = gt2 = -1;
                }
                if (!active && !has_shadow) {
                    if (!ADJOINT || fwd) lane_result[rs.w] = make_float4(result.x, result.y, result.z, 0.f);
                } else {
                    write_next = true;
                    uint32_t nf = (depth + 1) | ((br.bs.sampled_type & F_DELTA) ? PF_PREV_DELTA : 0u) | (has_shadow ? PF_HAS_SHADOW : 0u) | (active ? PF_ALIVE : 0u);
                    o_ro = make_float4(next.o.x, next.o.y, next.o.z, next.maxt);
                    o_rd = make_float4(next.d.x, next.d.y, next.d.z, br.bs.pdf);
                    o_thr = make_float4(throughput.x, throughput.y, throughput.z, eta);
                    o_prev = make_float4(si.p.x, si.p.y, si.p.z, __uint_as_float(nf));
                    o_res = make_float4(result.x, result.y, result.z, 0.f);
                    o_sho = make_float4(sray.o.x, sray.o.y, sray.o.z, sray.maxt);
                    o_shd = make_float4(sray.d.x, sray.d.y, sray.d.z, contrib.x);
                    o_shc = make_float2(contrib.y, contrib.z);
                    o_rng = make_uint4((uint32_t) rng.state, (uint32_t) (rng.state >> 32), rs.z, rs.w);
                    if (ADJOINT) { o_L = make_float4(L.x, L.y, L.z, 0.f); o_dL = make_float4(dL.x, dL.y, dL.z, 0.f); }
                }
            }
        }
        __syncwarp();
        if (ADJOINT) {
            // fp32 atomicAdd scatter into the parameter gradients, combined per warp and texel
            warp_scatter3(sc, gt0, guv0, gv0);
            warp_scatter3(sc, gt1, guv1, gv1);
            warp_scatter3(sc, gt2, guv2, gv2);
            if (TYPE != B200PT_BSDF_DIFFUSE && __any_sync(0xffffffffu, pg_bsdf >= 0)) {
                // the lanes of a material queue may hold different BSDFs of this model: the slot loop is uniform, a lane
                // without a differentiable texture in slot k passes -1
                for (int k = 0; k < B200PT_MAX_SLOTS; ++k) {
                    const int32_t pt = pg_bsdf >= 0 ? bsdf_grad_slot(sc, sc.bsdfs[pg_bsdf >= 0 ? pg_bsdf : 0], k) : -1;
                    if (!__any_sync(0xffffffffu, pt >= 0)) continue;
                    float3 g = V(0.f, 0.f, 0.f);
                    if (pt >= 0) {
                        const DevBsdf &pb = sc.bsdfs[pg_bsdf];
                        const int nch = sc.textures[pt].channels;
                        for (int ch = 0; ch < nch; ++ch) {
                            float3 cf = bsdf_param_coeff<TYPE>(sc, pb, guv1, pg_wi, pg_wo_em, pg_wo_s, pg_adir, pg_aind, pg_dir, pg_ind, pt, ch);
                            float sum = cf.x + cf.y + cf.z;      // a_dir / a_ind carry dL per colour channel
                            if (ch == 0) g.x = sum; else if (ch == 1) g.y = sum; else g.z = sum;
                        }
                    }
                    warp_scatter3(sc, pt, guv1, g);
                }
            }
        }
        // compaction: survivors get consecutive slots of the next buffer (one atomic per warp)
        uint32_t m = __ballot_sync(0xffffffffu, write_next);
        if (m) {
            uint32_t leader = __ffs(m) - 1, off = 0;
            if (lane_id == leader) off = atomicAdd(nxt_count, __popc(m));
            off = __shfl_sync(0xffffffffu, off, leader);
            if (write_next) {
                uint32_t dst = off + __popc(m & ((1u << lane_id) - 1u));
                nxt.ray_o[dst] = o_ro; nxt.ray_d[dst] = o_rd; nxt.thr[dst] = o_thr; nxt.prev[dst] = o_prev; nxt.result[dst] = o_res;
                nxt.rng[dst] = o_rng;
                if (__float_as_uint(o_prev.w) & PF_HAS_SHADOW) { nxt.sh_o[dst] = o_sho; nxt.sh_d[dst] = o_shd; nxt.sh_c[dst] = o_shc; }
                if (ADJOINT) { nxt.adj_L[dst] = o_L; nxt.adj_dL[dst] = o_dL; }
            }
        }
    }
    for (int o = 16; o; o >>= 1) { n_bounces += __shfl_xor_sync(0xffffffffu, n_bounces, o); n_shadow += __shfl_xor_sync(0xffffffffu, n_shadow, o); }
    if (lane_id == 0 && n_bounces) atomicAdd(&stats[ST_BOUNCES], (unsigned long long) n_bounces);
    if (lane_id == 0 && n_shadow) atomicAdd(&stats[ST_SHADOW], (unsigned long long) n_shadow);
}

// ---------------------------------------------------------------------------
// k_shade_env -- the rays of this bounce that left the scene: direct emission of the
// environment emitter with the MIS weight of the previous BSDF sample (path.cpp:115,
// 206-231,343; prb.py:148-163), then the path ends. One thread per queued slot.
// ---------------------------------------------------------------------------
template <bool ADJOINT>
__global__ void __launch_bounds__(BLOCK) k_shade_env(const __grid_constant__ DevScene sc, RenderCfg cfg, PathBuf cur, const uint32_t *__restrict__ queue,
                                                     const uint32_t *__restrict__ qcount, float4 *__restrict__ lane_result, unsigned long long *__restrict__ stats) {
    const uint32_t n = *qcount;
    const bool prb = cfg.prb != 0;
    const uint32_t stride = gridDim.x * blockDim.x;
    if (blockIdx.x == 0 && threadIdx.x == 0 && n) atomicAdd(&stats[ST_BOUNCES], (unsigned long long) n);   // loop iterations (path.cpp:193)
    for (uint32_t base = blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < n; base += stride) {
        uint32_t i = base + (threadIdx.x & 31u);
        int32_t gt = -1; float3 gv = V(0.f, 0.f, 0.f); float2 guv = make_float2(0.f, 0.f);
        if (i < n) {
            uint32_t slot = queue[i];
            float4 rd = cur.ray_d[slot], th = cur.thr[slot], pv = cur.prev[slot], rs4 = cur.result[slot];
            uint32_t flags = __float_as_uint(pv.w), depth = flags & PF_DEPTH_MASK;
            bool prev_delta = (flags & PF_PREV_DELTA) != 0;
            float3 d = V(rd.x, rd.y, rd.z), throughput = V(th.x, th.y, th.z), result = V(rs4.x, rs4.y, rs4.z);
            float prev_bsdf_pdf = rd.w;
            float em_pdf = prev_delta ? 0.f : env_pdf_direction(sc.env, d) * emitter_pmf(sc, sc.env_emitter);   // scene.cpp:378-389
            float mis_bsdf = mis_weight(prev_bsdf_pdf, em_pdf);
            bool em_active = prb ? !(cfg.hide_emitters && depth == 0) : prev_bsdf_pdf > 0.f;
            float3 crad = sc.env_type == B200PT_EMITTER_CONSTANT ? tex_eval3(sc, sc.env_radiance_tex, make_float2(0.f, 0.f)) : V(0.f, 0.f, 0.f);
            float3 rad = em_active ? env_eval(sc.env, crad, d) : V(0.f, 0.f, 0.f);
            const bool fwd = ADJOINT && cfg.forward != 0;
            if (fwd) {
                // forward mode: `result` carries dL; dLe = (beta * mis) (.) d(radiance) for the constant emitter
                if (em_active) {
                    bool is_map = sc.env_type == B200PT_EMITTER_ENVMAP;
                    float2 tuv = is_map ? env_direction_to_uv(env_xform(sc.env->mi, d)) : make_float2(0.f, 0.f);
                    result = result + tangent_dot(sc, sc.env_radiance_tex, tuv, (throughput * mis_bsdf) * (is_map ? sc.env_scale : 1.f));
                }
            } else if (prb) result = result + (throughput * mis_bsdf) * rad;
            else result = vfma(throughput, rad * mis_bsdf, result);
            // path.cpp:115,343: a primary ray that sees only the hidden environment is not a valid sample
            if (!prb && cfg.hide_emitters && depth == 0) result = V(0.f, 0.f, 0.f);
            if (!ADJOINT || fwd) lane_result[cur.rng[slot].w] = make_float4(result.x, result.y, result.z, 0.f);
            else if (em_active) {
                float4 dl = cur.adj_dL[slot];
                gt = sc.env_radiance_tex; gv = V(dl.x, dl.y, dl.z) * (throughput * mis_bsdf);
                if (sc.env_type == B200PT_EMITTER_ENVMAP) { guv = env_direction_to_uv(env_xform(sc.env->mi, d)); gv = gv * sc.env_scale; }
            }
        }
        if (ADJOINT) { __syncwarp(); warp_scatter3(sc, gt, guv, gv); }
    }
}

// Emitter::sample_direction / eval / pdf_direction tables of the environment emitter
// (b200pt_env_query): in n x 8 = ref point, sample, direction; out n x 20.
__global__ void k_env_query(const __grid_constant__ DevScene sc, uint32_t n, const float *__restrict__ in, float *__restrict__ out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float *q = in + 8 * (size_t) i; float *o = out + 20 * (size_t) i;
    DirectionSample ds; ds.pdf = 0.f; ds.emitter = -1; ds.uv = make_float2(0.f, 0.f);
    float3 crad = sc.env_type == B200PT_EMITTER_CONSTANT ? tex_eval3(sc, sc.env_radiance_tex, make_float2(0.f, 0.f)) : V(0.f, 0.f, 0.f);
    float3 w = env_sample_direction(sc.env, crad, V(q[0], q[1], q[2]), q[3], q[4], ds);
    o[0] = ds.d.x; o[1] = ds.d.y; o[2] = ds.d.z; o[3] = ds.pdf; o[4] = ds.dist; o[5] = ds.uv.x; o[6] = ds.uv.y;
    o[7] = w.x; o[8] = w.y; o[9] = w.z;
    float3 e = env_eval(sc.env, crad, ds.d);
    o[10] = e.x; o[11] = e.y; o[12] = e.z; o[13] = env_pdf_direction(sc.env, ds.d);
    float3 d = V(q[5], q[6], q[7]);
    e = env_eval(sc.env, crad, d);
    o[14] = e.x; o[15] = e.y; o[16] = e.z; o[17] = env_pdf_direction(sc.env, d);
    o[18] = 0.f; o[19] = 0.f;
}

// ---------------------------------------------------------------------------
// Film: ImageBlock::put (imageblock.cpp:192-574) + HDRFilm::develop (hdrfilm.cpp:393)
// ---------------------------------------------------------------------------
// Box filter: the spp samples of a pixel are consecutive lanes -> one warp per
// pixel sums them in a fixed order and owns the pixel (no atomics, deterministic).
__global__ void __launch_bounds__(BLOCK) k_splat_box(DevScene sc, RenderCfg cfg, const uint32_t *__restrict__ pix_ids,
                                                     const float4 *__restrict__ lane_result, float *__restrict__ film) {
    uint32_t n_pix = cfg.chunk_lanes / cfg.spp;
    uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane_id = threadIdx.x & 31u, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t p = warp; p < n_pix; p += n_warps) {
        float r = 0.f, g = 0.f, b = 0.f;
        for (uint32_t s = lane_id; s < cfg.spp; s += 32) {
            float4 v = lane_result[(size_t) p * cfg.spp + s];
            r += v.x; g += v.y; b += v.z;
        }
        for (int o = 16; o; o >>= 1) { r += __shfl_xor_sync(0xffffffffu, r, o); g += __shfl_xor_sync(0xffffffffu, g, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
        if (lane_id == 0) {
            uint32_t pixel = __ldg(&pix_ids[cfg.chunk_pix0 + p]);
            float4 *f = (float4 *) film + pixel;
            float4 a = *f; a.x += r; a.y += g; a.z += b; a.w += (float) cfg.spp; *f = a;
        }
    }
}

PT_DEV void sample_film_pos(const DevScene &sc, const RenderCfg &cfg, uint32_t pixel, uint32_t s, float &pfx, float &pfy) {
    uint32_t py = pixel / sc.crop_w, px = pixel - py * sc.crop_w;
    Pcg32 rng; rng.seed_lane(cfg.seed_value, pixel * cfg.spp + s);
    float u1 = rng.next_f32(), u2 = rng.next_f32();
    // position relative to the block: pos + (border - offset - .5) (imageblock.cpp:280)
    pfx = ((float) (px + sc.crop_x) + u1) + (0.f - (float) sc.crop_x - .5f);
    pfy = ((float) (py + sc.crop_y) + u2) + (0.f - (float) sc.crop_y - .5f);
}

// Gaussian (any non-box) filter. The samples of a pixel are consecutive lanes, so a warp
// usually holds 32 samples of ONE pixel whose footprints lie in the same 5x5 window
// (floor(pos) +- 2, imageblock.cpp:452-466): the warp reduces the 25 x 4 weighted values
// with shuffles and issues one fp32 atomicAdd per (tap, channel) instead of 32.
// WEIGHTS_ONLY accumulates only the weight channel (first pass of the adjoint).
//
// The reduction folds: SHFL issues at a quarter of the ALU rate and 100 butterfly reductions (500 shuffles per warp)
// bounded this kernel. A folding reduction sums 32 values per lane with 16 + 8 + 4 + 2 + 1 = 31 shuffles: at offset o
// the lane keeps the half of its values selected by its bit o and hands the other half to its partner. Lane L ends up
// with the warp total of value L, added in the same pairwise order as a butterfly (measured on the B200:
// +2.6 % of the whole frame, profiles/r02_switches.md). The weights-only pass (25 values) keeps the butterfly.
template <bool WEIGHTS_ONLY>
__global__ void __launch_bounds__(BLOCK) k_splat_gauss(DevScene sc, RenderCfg cfg, const uint32_t *__restrict__ pix_ids,
                                                       const float4 *__restrict__ lane_result, float *__restrict__ film) {
    const uint32_t lane_id = threadIdx.x & 31u;
    const uint32_t warp_stride = gridDim.x * blockDim.x;
    const int W = (int) sc.crop_w, H = (int) sc.crop_h;
    const int n = (int) ceilf(sc.gauss_radius - .5f);          // taps on either side (2 for the default radius)
    for (uint32_t base = blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < cfg.chunk_lanes; base += warp_stride) {
        uint32_t i = base + lane_id;
        bool valid = i < cfg.chunk_lanes;
        uint32_t pixel = 0xffffffffu; float pfx = 0.f, pfy = 0.f;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (valid) {
            pixel = __ldg(&pix_ids[cfg.chunk_pix0 + i / cfg.spp]);
            sample_film_pos(sc, cfg, pixel, i % cfg.spp, pfx, pfy);
            if (!WEIGHTS_ONLY) v = lane_result[i];
        }
        uint32_t pixel0 = __shfl_sync(0xffffffffu, pixel, 0);
        bool uniform = __all_sync(0xffffffffu, pixel == pixel0) && n <= 2;
        if (uniform) {
            int py = (int) (pixel0 / sc.crop_w), px = (int) (pixel0 - (uint32_t) py * sc.crop_w);
            // per-lane separable weights on the common window px-2..px+2; zero outside the
            // sample's own footprint [ceil(p - r), floor(p + r)] (imageblock.cpp:283-287)
            float wx[5], wy[5];
            int x0 = (int) ceilf(pfx - sc.gauss_radius), x1 = (int) floorf(pfx + sc.gauss_radius);
            int y0 = (int) ceilf(pfy - sc.gauss_radius), y1 = (int) floorf(pfy + sc.gauss_radius);
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                int x = px - 2 + k, y = py - 2 + k;
                wx[k] = (x >= x0 && x <= x1) ? rfilter_eval(sc, (float) x - pfx) : 0.f;
                wy[k] = (y >= y0 && y <= y1) ? rfilter_eval(sc, (float) y - pfy) : 0.f;
            }
            if (!WEIGHTS_ONLY) {
                // value m = tap * 4 + channel (tap = ky * 5 + kx; channels r, g, b, weight), 100 values in 4 batches of 32
                const bool b16 = (lane_id & 16u) != 0, b8 = (lane_id & 8u) != 0, b4 = (lane_id & 4u) != 0, b2 = (lane_id & 2u) != 0, b1 = (lane_id & 1u) != 0;
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    float a[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const int m = 32 * b + j, tap = m >> 2, ch = m & 3;
                        if (m < 100) { float w = wx[tap % 5] * wy[tap / 5]; a[j] = ch == 0 ? v.x * w : ch == 1 ? v.y * w : ch == 2 ? v.z * w : w; }
                        else a[j] = 0.f;
                    }
#pragma unroll
                    for (int j = 0; j < 16; ++j) { float keep = b16 ? a[j + 16] : a[j], send = b16 ? a[j] : a[j + 16]; a[j] = keep + __shfl_xor_sync(0xffffffffu, send, 16); }
#pragma unroll
                    for (int j = 0; j < 8; ++j) { float keep = b8 ? a[j + 8] : a[j], send = b8 ? a[j] : a[j + 8]; a[j] = keep + __shfl_xor_sync(0xffffffffu, send, 8); }
#pragma unroll
                    for (int j = 0; j < 4; ++j) { float keep = b4 ? a[j + 4] : a[j], send = b4 ? a[j] : a[j + 4]; a[j] = keep + __shfl_xor_sync(0xffffffffu, send, 4); }
#pragma unroll
                    for (int j = 0; j < 2; ++j) { float keep = b2 ? a[j + 2] : a[j], send = b2 ? a[j] : a[j + 2]; a[j] = keep + __shfl_xor_sync(0xffffffffu, send, 2); }
                    { float keep = b1 ? a[1] : a[0], send = b1 ? a[0] : a[1]; a[0] = keep + __shfl_xor_sync(0xffffffffu, send, 1); }
                    // this lane now holds the warp total of value 32 b + lane_id; adding a zero total changes nothing
                    const int m = 32 * b + (int) lane_id, tap = m >> 2;
                    const int x = px - 2 + tap % 5, y = py - 2 + tap / 5;
                    if (m < 100 && x >= 0 && y >= 0 && x < W && y < H && a[0] != 0.f) atomicAdd(film + 4 * ((size_t) y * W + x) + (m & 3), a[0]);
                }
                continue;
            }
            float mine3 = 0.f;
#pragma unroll
            for (int ky = 0; ky < 5; ++ky)
#pragma unroll
                for (int kx = 0; kx < 5; ++kx) {
                    float a3 = wx[kx] * wy[ky];      // weights-only pass: the weight channel
#pragma unroll
                    for (int o = 16; o; o >>= 1) a3 += __shfl_xor_sync(0xffffffffu, a3, o);
                    if ((int) lane_id == ky * 5 + kx) mine3 = a3;
                }
            if (lane_id < 25) {
                int x = px - 2 + (int) (lane_id % 5), y = py - 2 + (int) (lane_id / 5);
                if (x >= 0 && y >= 0 && x < W && y < H && mine3 != 0.f) {
                    atomicAdd(film + 4 * ((size_t) y * W + x) + 3, mine3);
                }
            }
        } else if (valid) {
            int x0 = max((int) ceilf(pfx - sc.gauss_radius), 0), y0 = max((int) ceilf(pfy - sc.gauss_radius), 0);
            int x1 = min((int) floorf(pfx + sc.gauss_radius), W - 1), y1 = min((int) floorf(pfy + sc.gauss_radius), H - 1);
            for (int y = y0; y <= y1; ++y) {
                float wy = rfilter_eval(sc, (float) y - pfy);
                for (int x = x0; x <= x1; ++x) {
                    float w = rfilter_eval(sc, (float) x - pfx) * wy;
                    float *f = film + 4 * ((size_t) y * W + x);
                    if (!WEIGHTS_ONLY) { atomicAdd(f + 0, v.x * w); atomicAdd(f + 1, v.y * w); atomicAdd(f + 2, v.z * w); }
                    atomicAdd(f + 3, w);
                }
            }
        }
    }
}

// Adjoint of splat + develop for one sample (common.py:696-746): dL = sum_pix w * grad_in / W
__global__ void __launch_bounds__(BLOCK) k_splat_adjoint(DevScene sc, RenderCfg cfg, const uint32_t *__restrict__ pix_ids,
                                                         const float *__restrict__ grad_in, const float *__restrict__ film_w, float4 *__restrict__ lane_dL) {
    uint32_t stride = gridDim.x * blockDim.x;
    int W = (int) sc.crop_w, H = (int) sc.crop_h;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < cfg.chunk_lanes; i += stride) {
        uint32_t pixel = __ldg(&pix_ids[cfg.chunk_pix0 + i / cfg.spp]), s = i % cfg.spp;
        float3 g = V(0.f, 0.f, 0.f);
        if (sc.rfilter == B200PT_RFILTER_BOX) {
            float w = (float) cfg.spp;
            g = V(fdiv(grad_in[3 * (size_t) pixel], w), fdiv(grad_in[3 * (size_t) pixel + 1], w), fdiv(grad_in[3 * (size_t) pixel + 2], w));
        } else {
            float pfx, pfy; sample_film_pos(sc, cfg, pixel, s, pfx, pfy);
            int x0 = max((int) ceilf(pfx - sc.gauss_radius), 0), y0 = max((int) ceilf(pfy - sc.gauss_radius), 0);
            int x1 = min((int) floorf(pfx + sc.gauss_radius), W - 1), y1 = min((int) floorf(pfy + sc.gauss_radius), H - 1);
            for (int y = y0; y <= y1; ++y) for (int x = x0; x <= x1; ++x) {
                float w = rfilter_eval(sc, (float) x - pfx) * rfilter_eval(sc, (float) y - pfy);
                size_t pi = (size_t) y * W + x;
                float ws = film_w[4 * pi + 3]; if (ws == 0.f) ws = 1.f;
                g.x = __fmaf_rn(w, fdiv(grad_in[3 * pi], ws), g.x); g.y = __fmaf_rn(w, fdiv(grad_in[3 * pi + 1], ws), g.y); g.z = __fmaf_rn(w, fdiv(grad_in[3 * pi + 2], ws), g.z);
            }
        }
        lane_dL[i] = make_float4(g.x, g.y, g.z, 0.f);
    }
}

__global__ void __launch_bounds__(BLOCK) k_develop(uint32_t n_pix, const float *__restrict__ film, float *__restrict__ out) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_pix; i += gridDim.x * blockDim.x) {
        float4 f = ((const float4 *) film)[i];
        float w = f.w == 0.f ? 1.f : f.w;
        out[3 * (size_t) i] = fdiv(f.x, w); out[3 * (size_t) i + 1] = fdiv(f.y, w); out[3 * (size_t) i + 2] = fdiv(f.z, w);
    }
}

// ---------------------------------------------------------------------------
// Operator kernels (parity tests through the C ABI)
// ---------------------------------------------------------------------------
template <bool ANY>
__global__ void __launch_bounds__(BLOCK) k_ray_query(DevScene sc, uint32_t n, const float *__restrict__ rays, float *__restrict__ t_out, float *__restrict__ uv_out,
                                                     uint32_t *__restrict__ prim_out, int32_t *__restrict__ shape_out, uint8_t *__restrict__ occ_out,
                                                     uint32_t n_smem_nodes, uint32_t n_smem_tris, bool flat) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ uint64_t bar;
    float4 *s_nodes = (float4 *) smem_raw;
    float4 *s_tris = s_nodes + 4 * (size_t) n_smem_nodes;
    if (threadIdx.x == 0) mbar_init(&bar, 1);
    __syncthreads();
    stage_bvh(sc, s_nodes, s_tris, n_smem_nodes, n_smem_tris, &bar);
    TraceCtx ctx = { s_nodes, s_tris, sc.nodes, sc.tris, n_smem_nodes, n_smem_tris };
    auto put = [&](uint32_t i, bool found, const Hit &h) {
        if (ANY) { occ_out[i] = found ? 1 : 0; return; }
        t_out[i] = found ? h.t : PT_INF; uv_out[2 * i] = found ? h.u : 0.f; uv_out[2 * i + 1] = found ? h.v : 0.f;
        if (found) {
            uint4 pv = sc.prim_verts[h.prim];
            shape_out[i] = (int32_t) pv.w; prim_out[i] = h.prim - sc.shapes[pv.w].first_prim;
        } else { shape_out[i] = -1; prim_out[i] = 0; }
    };
    if (flat) {         // the traversal the render kernels use for this scene, in the same warp-uniform loop as k_trace_flat
        __shared__ FlatLeaves s_leaves;
        __shared__ uint8_t s_primmap[FLAT_MAX_TRIS];
        __shared__ FlatWarp s_warp[BLOCK / 32];
        const uint32_t n_pad = build_leaf_list(s_nodes, n_smem_nodes, s_tris, n_smem_tris, s_leaves, s_primmap);
        FlatWarp &w = s_warp[threadIdx.x >> 5];
        for (uint32_t base = blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < n; base += gridDim.x * blockDim.x) {
            const uint32_t i = base + (threadIdx.x & 31u);
            const bool valid = i < n;
            float3 o = V(0.f, 0.f, 0.f), d = V(0.f, 0.f, 1.f); float maxt = 0.f;
            if (valid) { const float *r = rays + 7 * (size_t) i; o = V(r[0], r[1], r[2]); d = V(r[3], r[4], r[5]); maxt = r[6]; }
            Hit h;
            const bool found = flat_phase<ANY>(w, s_leaves, n_pad, s_tris, s_primmap, valid, o, d, maxt, h);
            if (valid) put(i, found, h);
            __syncwarp();
        }
        return;
    }
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float *r = rays + 7 * (size_t) i;
        Hit h;
        const bool found = traverse<ANY, false>(ctx, V(r[0], r[1], r[2]), V(r[3], r[4], r[5]), r[6], h);
        put(i, found, h);
    }
}

template <int TYPE>
__global__ void k_bsdf_eval(DevScene sc, uint32_t bsdf, uint32_t n, const float *__restrict__ in, float *__restrict__ out) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float *q = in + 11 * (size_t) i; float *o = out + 14 * (size_t) i;
        BsdfResult r = bsdf_eval_pdf_sample<TYPE>(sc, sc.bsdfs[bsdf], make_float2(q[6], q[7]), V(q[0], q[1], q[2]), V(q[3], q[4], q[5]), q[8], q[9], q[10]);
        o[0] = r.value.x; o[1] = r.value.y; o[2] = r.value.z; o[3] = r.pdf;
        o[4] = r.bs.wo.x; o[5] = r.bs.wo.y; o[6] = r.bs.wo.z; o[7] = r.bs.pdf; o[8] = r.bs.eta;
        o[9] = __uint_as_float(r.bs.sampled_type);
        o[10] = r.weight.x; o[11] = r.weight.y; o[12] = r.weight.z; o[13] = (float) r.bs.sampled_component;
    }
}

// ---------------------------------------------------------------------------
// host-side launchers
// ---------------------------------------------------------------------------
void read_watchdog(unsigned long long out[4]) {
#ifdef B200PT_WATCHDOG
    cudaMemcpyFromSymbol(out, g_watchdog, sizeof(unsigned long long) * 4);
#else
    out[0] = out[1] = out[2] = out[3] = 0;
#endif
}

void launch_generate(const DevScene &sc, const RenderCfg &cfg, const uint32_t *pix_ids, PathBuf buf, const float4 *adj_dL_lane,
                     const float4 *adj_L_lane, int grid, cudaStream_t st) {
    k_generate<<<grid, BLOCK, 0, st>>>(sc, cfg, pix_ids, buf, adj_dL_lane, adj_L_lane);
}

void launch_trace(const DevScene &sc, const RenderCfg &cfg, PathBuf cur, float4 *hit, const uint32_t *n_in, Queues q, uint32_t *qcounts,
                  float4 *lane_result, unsigned long long *stats, bool first, const Launch &L, cudaStream_t st) {
    bool all = L.n_smem_nodes == sc.n_nodes && L.n_smem_tris == sc.n_tris;
    if (L.flat) {       // <= FLAT_MAX_LEAVES leaves: every lane tests every leaf box, no tree walk (see k_trace_flat)
        int grid = L.grid_flat;
        if (first) k_trace_flat<true><<<grid, BLOCK, L.smem_trace + L.smem_tables, st>>>(sc, cfg, cur, hit, n_in, q, qcounts, lane_result, stats, L.n_smem_nodes, L.n_smem_tris);
        else k_trace_flat<false><<<grid, BLOCK, L.smem_trace + L.smem_tables, st>>>(sc, cfg, cur, hit, n_in, q, qcounts, lane_result, stats, L.n_smem_nodes, L.n_smem_tris);
        return;
    }
    {
#define LAUNCH_DYN(F, A) k_trace_dyn<F, A><<<L.grid, BLOCK, L.smem_trace + L.smem_tables, st>>>(sc, cfg, cur, hit, n_in, q, qcounts, qcounts + 5, lane_result, stats, L.n_smem_nodes, L.n_smem_tris, L.refill_idle)
        if (first) { if (all) LAUNCH_DYN(true, true); else LAUNCH_DYN(true, false); }
        else { if (all) LAUNCH_DYN(false, true); else LAUNCH_DYN(false, false); }
#undef LAUNCH_DYN
    }
}

template <int TYPE>
static void launch_shade_t(const DevScene &sc, const RenderCfg &cfg, PathBuf cur, const float4 *hit, const uint32_t *queue, const uint32_t *qcount,
                           PathBuf nxt, uint32_t *nxt_count, float4 *lane_result, unsigned long long *stats, const Launch &L, cudaStream_t st) {
    // EXT: environment emitter or non-uniform emitter selection present (pt_device.cuh: sample_emitter_direction)
    const bool ext = sc.env_type >= 0 || sc.em_cdf != nullptr;
    if (cfg.adjoint && cur.vis) k_shade<TYPE, 2, true><<<L.grid * (BLOCK / BLOCK_SHADE), BLOCK_SHADE, L.smem_tables, st>>>(sc, cfg, cur, hit, queue, qcount, nxt, nxt_count, lane_result, stats, 0, 0);
    else if (cfg.adjoint) k_shade<TYPE, 1, true><<<L.grid * (BLOCK / BLOCK_SHADE), BLOCK_SHADE, L.smem_trace + L.smem_tables, st>>>(sc, cfg, cur, hit, queue, qcount, nxt, nxt_count, lane_result, stats, L.n_smem_nodes, L.n_smem_tris);
    else if (ext) k_shade<TYPE, 0, true><<<L.grid * (BLOCK / BLOCK_SHADE), BLOCK_SHADE, L.smem_tables, st>>>(sc, cfg, cur, hit, queue, qcount, nxt, nxt_count, lane_result, stats, 0, 0);
    else k_shade<TYPE, 0, false><<<L.grid * (BLOCK / BLOCK_SHADE), BLOCK_SHADE, L.smem_tables, st>>>(sc, cfg, cur, hit, queue, qcount, nxt, nxt_count, lane_result, stats, 0, 0);
}

void launch_shade(int type, const DevScene &sc, const RenderCfg &cfg, PathBuf cur, const float4 *hit, const uint32_t *queue, const uint32_t *qcount,
                  PathBuf nxt, uint32_t *nxt_count, float4 *lane_result, unsigned long long *stats, const Launch &grid, cudaStream_t st) {
    switch (type) {
        case B200PT_BSDF_DIFFUSE: launch_shade_t<B200PT_BSDF_DIFFUSE>(sc, cfg, cur, hit, queue, qcount, nxt, nxt_count, lane_result, stats, grid, st); break;
        case B200PT_BSDF_CONDUCTOR: launch_shade_t<B200PT_BSDF_CONDUCTOR>(sc, cfg, cur, hit, queue, qcount, nxt, nxt_count, lane_result, stats, grid, st); break;
        case B200PT_BSDF_DIELECTRIC: launch_shade_t<B200PT_BSDF_DIELECTRIC>(sc, cfg, cur, hit, queue, qcount, nxt, nxt_count, lane_result, stats, grid, st); break;
        default: launch_shade_t<B200PT_BSDF_PRINCIPLED>(sc, cfg, cur, hit, queue, qcount, nxt, nxt_count, lane_result, stats, grid, st); break;
    }
}

void launch_shade_env(const DevScene &sc, const RenderCfg &cfg, PathBuf cur, const uint32_t *queue, const uint32_t *qcount,
                      float4 *lane_result, unsigned long long *stats, int grid, cudaStream_t st) {
    if (cfg.adjoint) k_shade_env<true><<<grid, BLOCK, 0, st>>>(sc, cfg, cur, queue, qcount, lane_result, stats);
    else k_shade_env<false><<<grid, BLOCK, 0, st>>>(sc, cfg, cur, queue, qcount, lane_result, stats);
}

// Lanes still queued when the per-chunk bounce counters run out (api.cu: MAX_BOUNCE_SLOTS, unbounded paths only) hand in
// the radiance gathered so far.
__global__ void __launch_bounds__(BLOCK) k_flush(PathBuf cur, Queues q, const uint32_t *__restrict__ qcounts, float4 *__restrict__ lane_result) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (int t = 0; t < N_QUEUES; ++t) {
        if (!q.slots[t]) continue;
        const uint32_t n = qcounts[t == Q_ENV ? QCOUNT_ENV : t];
        for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
            uint32_t slot = q.slots[t][i];
            lane_result[cur.rng[slot].w] = cur.result[slot];
        }
    }
}
void launch_flush(PathBuf cur, Queues q, const uint32_t *qcounts, float4 *lane_result, int grid, cudaStream_t st) {
    k_flush<<<grid, BLOCK, 0, st>>>(cur, q, qcounts, lane_result);
}

// ---------------------------------------------------------------------------
// Device-side BVH refit (geometry update with unchanged topology; the reference's Scene::parameters_changed ->
// accel update, scene.cpp:517-540, rebuilds or refits through Embree / OptiX). After new vertex positions have been
// uploaded: k_refit_tris regathers the leaf-ordered triangle records, k_refit_level recomputes the child boxes of
// one breadth-first level (deepest level first: children always have larger indices than their parent).
// `tight` keeps the un-inflated child boxes (12 floats per node) so that the inflation (bvh.cpp: inflate) is applied
// once per box, not once per level.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(BLOCK) k_refit_tris(uint32_t n_tris, float4 *__restrict__ tris, const uint4 *__restrict__ prim_verts, const float4 *__restrict__ vertices) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_tris; i += gridDim.x * blockDim.x) {
        const float4 t0 = tris[3 * (size_t) i];
        const uint4 pv = prim_verts[__float_as_uint(t0.w)];
        const float4 a = vertices[2 * (size_t) pv.x], b = vertices[2 * (size_t) pv.y], c = vertices[2 * (size_t) pv.z];
        tris[3 * (size_t) i] = make_float4(a.x, a.y, a.z, t0.w);
        tris[3 * (size_t) i + 1] = make_float4(b.x - a.x, b.y - a.y, b.z - a.z, 0.f);          // e1 = p1 - p0 (mesh.h:1139)
        tris[3 * (size_t) i + 2] = make_float4(c.x - a.x, c.y - a.y, c.z - a.z, 0.f);
    }
}

PT_DEV void refit_child(int32_t child, const float4 *tris, const uint4 *prim_verts, const float4 *vertices, const float *tight, float *out_tight, float *out_box) {
    float lo[3] = { PT_INF, PT_INF, PT_INF }, hi[3] = { -PT_INF, -PT_INF, -PT_INF };
    if (child == 0x7fffffff) { for (int a = 0; a < 3; ++a) { out_tight[a] = out_box[a] = PT_INF; out_tight[3 + a] = out_box[3 + a] = -PT_INF; } return; }
    if (child < 0) {          // leaf: the exact vertex positions of its triangles
        const uint32_t enc = (uint32_t) ~child, first = enc >> 3, count = (enc & 7u) + 1u;
        for (uint32_t i = first; i < first + count; ++i) {
            const uint4 pv = prim_verts[__float_as_uint(tris[3 * (size_t) i].w)];
            const uint32_t vi[3] = { pv.x, pv.y, pv.z };
            for (int k = 0; k < 3; ++k) {
                const float4 p = vertices[2 * (size_t) vi[k]];
                lo[0] = fminf(lo[0], p.x); lo[1] = fminf(lo[1], p.y); lo[2] = fminf(lo[2], p.z);
                hi[0] = fmaxf(hi[0], p.x); hi[1] = fmaxf(hi[1], p.y); hi[2] = fmaxf(hi[2], p.z);
            }
        }
    } else {                  // inner node: union of its two (tight) child boxes, already refitted (deeper level)
        const float *t = tight + 12 * (size_t) child;
        for (int a = 0; a < 3; ++a) { lo[a] = fminf(t[a], t[6 + a]); hi[a] = fmaxf(t[3 + a], t[9 + a]); }
    }
    for (int a = 0; a < 3; ++a) {
        out_tight[a] = lo[a]; out_tight[3 + a] = hi[a];
        const float m = fmaxf(fabsf(lo[a]), fabsf(hi[a])), pad = m * 4e-6f + 1e-7f;            // bvh.cpp: inflate
        out_box[a] = nextafterf(lo[a] - pad, -PT_INF); out_box[3 + a] = nextafterf(hi[a] + pad, PT_INF);
    }
}

__global__ void __launch_bounds__(BLOCK) k_refit_level(float4 *__restrict__ nodes, float *__restrict__ tight, const float4 *__restrict__ tris, const uint4 *__restrict__ prim_verts,
                                                       const float4 *__restrict__ vertices, uint32_t first, uint32_t count) {
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < count; k += gridDim.x * blockDim.x) {
        const uint32_t i = first + k;
        const float4 n3 = nodes[4 * (size_t) i + 3];
        float box[12];
        refit_child(__float_as_int(n3.x), tris, prim_verts, vertices, tight, tight + 12 * (size_t) i, box);
        refit_child(__float_as_int(n3.y), tris, prim_verts, vertices, tight, tight + 12 * (size_t) i + 6, box + 6);
        nodes[4 * (size_t) i] = make_float4(box[0], box[1], box[2], box[3]);
        nodes[4 * (size_t) i + 1] = make_float4(box[4], box[5], box[6], box[7]);
        nodes[4 * (size_t) i + 2] = make_float4(box[8], box[9], box[10], box[11]);
    }
}

void launch_refit(const DevScene &sc, float *tight, const uint32_t *level_start, uint32_t n_levels, int grid, cudaStream_t st) {
    k_refit_tris<<<grid, BLOCK, 0, st>>>(sc.n_tris, (float4 *) sc.tris, sc.prim_verts, sc.vertices);
    for (uint32_t l = n_levels; l-- > 0;) {
        const uint32_t first = level_start[l], count = level_start[l + 1] - first;
        if (count) k_refit_level<<<(int) std::min<uint32_t>((count + BLOCK - 1) / BLOCK, (uint32_t) grid), BLOCK, 0, st>>>((float4 *) sc.nodes, tight, sc.tris, sc.prim_verts, sc.vertices, first, count);
    }
}

void launch_env_query(const DevScene &sc, uint32_t n, const float *in, float *out, cudaStream_t st) {
    k_env_query<<<(int) ((n + 127) / 128), 128, 0, st>>>(sc, n, in, out);
}

void launch_splat(const DevScene &sc, const RenderCfg &cfg, const uint32_t *pix_ids, const float4 *lane_result, float *film, int grid, cudaStream_t st) {
    if (sc.rfilter == B200PT_RFILTER_BOX) k_splat_box<<<grid, BLOCK, 0, st>>>(sc, cfg, pix_ids, lane_result, film);
    else k_splat_gauss<false><<<grid, BLOCK, 0, st>>>(sc, cfg, pix_ids, lane_result, film);
}

void launch_weights(const DevScene &sc, const RenderCfg &cfg, const uint32_t *pix_ids, float *film, int grid, cudaStream_t st) {
    k_splat_gauss<true><<<grid, BLOCK, 0, st>>>(sc, cfg, pix_ids, nullptr, film);
}

void launch_splat_adjoint(const DevScene &sc, const RenderCfg &cfg, const uint32_t *pix_ids, const float *grad_in, const float *film_w,
                          float4 *lane_dL, int grid, cudaStream_t st) {
    k_splat_adjoint<<<grid, BLOCK, 0, st>>>(sc, cfg, pix_ids, grad_in, film_w, lane_dL);
}

void launch_develop(const DevScene &sc, const float *film, float *out, cudaStream_t st) {
    uint32_t n = sc.crop_w * sc.crop_h;
    k_develop<<<(n + BLOCK - 1) / BLOCK, BLOCK, 0, st>>>(n, film, out);
}

void launch_ray_intersect(const DevScene &sc, uint32_t n, const float *rays, float *t, float *uv, uint32_t *prim, int32_t *shape, const Launch &L, cudaStream_t st) {
    k_ray_query<false><<<L.grid, BLOCK, L.smem_trace, st>>>(sc, n, rays, t, uv, prim, shape, nullptr, L.n_smem_nodes, L.n_smem_tris, L.flat);
}
void launch_ray_test(const DevScene &sc, uint32_t n, const float *rays, uint8_t *hit, const Launch &L, cudaStream_t st) {
    k_ray_query<true><<<L.grid, BLOCK, L.smem_trace, st>>>(sc, n, rays, nullptr, nullptr, nullptr, nullptr, hit, L.n_smem_nodes, L.n_smem_tris, L.flat);
}
void launch_bsdf_eval(const DevScene &sc, uint32_t bsdf, int type, uint32_t n, const float *in, float *out, cudaStream_t st) {
    int grid = (int) ((n + 127) / 128); if (grid < 1) grid = 1;
    switch (type) {
        case B200PT_BSDF_DIFFUSE: k_bsdf_eval<B200PT_BSDF_DIFFUSE><<<grid, 128, 0, st>>>(sc, bsdf, n, in, out); break;
        case B200PT_BSDF_CONDUCTOR: k_bsdf_eval<B200PT_BSDF_CONDUCTOR><<<grid, 128, 0, st>>>(sc, bsdf, n, in, out); break;
        case B200PT_BSDF_DIELECTRIC: k_bsdf_eval<B200PT_BSDF_DIELECTRIC><<<grid, 128, 0, st>>>(sc, bsdf, n, in, out); break;
        default: k_bsdf_eval<B200PT_BSDF_PRINCIPLED><<<grid, 128, 0, st>>>(sc, bsdf, n, in, out); break;
    }
}

void set_trace_smem_attr(size_t bytes_wanted) {
    // the attribute is per kernel function (process-wide): never lower it, an earlier scene of this
    // process may need more dynamic shared memory than the one being created now
    // (and per device: the attribute belongs to the current device's context)
    static std::mutex mu;
    static size_t current[64] = { 0 };
    std::lock_guard<std::mutex> lock(mu);
    int dev = 0; cudaGetDevice(&dev); dev = dev < 0 ? 0 : dev % 64;
    if (bytes_wanted <= current[dev]) return;
    current[dev] = bytes_wanted;
    size_t bytes = bytes_wanted;
    cudaFuncSetAttribute(k_trace_dyn<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
    cudaFuncSetAttribute(k_trace_dyn<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
    cudaFuncSetAttribute(k_trace_dyn<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
    cudaFuncSetAttribute(k_trace_dyn<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
    cudaFuncSetAttribute(k_trace_flat<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
    cudaFuncSetAttribute(k_trace_flat<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
    cudaFuncSetAttribute(k_ray_query<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
    cudaFuncSetAttribute(k_ray_query<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
    cudaFuncSetAttribute(k_shade<B200PT_BSDF_DIFFUSE, 0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
    cudaFuncSetAttribute(k_shade<B200PT_BSDF_DIFFUSE, 0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
    cudaFuncSetAttribute(k_shade<B200PT_BSDF_CONDUCTOR, 0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
    cudaFuncSetAttribute(k_shade<B200PT_BSDF_CONDUCTOR, 0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
    cudaFuncSetAttribute(k_shade<B200PT_BSDF_DIELECTRIC, 0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
    cudaFuncSetAttribute(k_shade<B200PT_BSDF_DIELECTRIC, 0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
    cudaFuncSetAttribute(k_shade<B200PT_BSDF_PRINCIPLED, 0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
    cudaFuncSetAttribute(k_shade<B200PT_BSDF_PRINCIPLED, 0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
    cudaFuncSetAttribute(k_shade<B200PT_BSDF_DIFFUSE, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
    cudaFuncSetAttribute(k_shade<B200PT_BSDF_CONDUCTOR, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
    cudaFuncSetAttribute(k_shade<B200PT_BSDF_DIELECTRIC, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
    cudaFuncSetAttribute(k_shade<B200PT_BSDF_PRINCIPLED, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
}

} // namespace pt
