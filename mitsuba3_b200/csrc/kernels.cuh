// kernels.cuh -- wavefront state layout and kernel launch interface shared by
// kernels.cu (device code) and api.cu (host orchestration / C ABI).
#pragma once
#include "pt_device.cuh"

namespace pt {

// Path state of one wavefront buffer, structure-of-arrays, one 16-byte vector
// per field so that every access is a single 128-bit coalesced transaction.
// Two buffers ping-pong per bounce: the shading kernels read buffer A through
// the material queues and write the surviving lanes compacted into buffer B.
struct PathBuf {
    float4 *ray_o;    // o.xyz, maxt
    float4 *ray_d;    // d.xyz, prev_bsdf_pdf
    float4 *thr;      // throughput.xyz, eta
    float4 *prev;     // prev_si.p.xyz, flags (bits below)
    uint4  *rng;      // pcg state lo, hi, global lane (pixel*spp+s), chunk-local lane
    float4 *result;   // radiance accumulated so far (rgb), unused
    float4 *sh_o;     // pending NEE shadow ray: o.xyz, maxt
    float4 *sh_d;     // d.xyz, contribution.x
    float2 *sh_c;     // contribution.y, contribution.z
    // PRB adjoint pass only
    float4 *adj_L;    // radiance still to come (rgb), unused
    float4 *adj_dL;   // dLoss/dL of this sample (rgb), unused
    // gradient calls with max_depth <= 32: bit b of vis[chunk-local lane] = "the NEE ray of bounce b is unoccluded", written by
    // the traversal kernels in the call's primal pass, read by the replay (k_shade<.., 2, ..>); nullptr otherwise
    uint32_t *vis;
};

// flags word stored in prev.w
#define PF_DEPTH_MASK   0x0000ffffu
#define PF_PREV_DELTA   0x00010000u
#define PF_HAS_SHADOW   0x00020000u
#define PF_ALIVE        0x00040000u

constexpr int N_BSDF_TYPES = 4;
constexpr int N_QUEUES = N_BSDF_TYPES + 1;   // + the queue of the rays that left the scene (environment emitter)
constexpr int Q_ENV = N_BSDF_TYPES;
constexpr int QCOUNT_ENV = 6;                // index of the environment queue's size in a bounce's counter block

struct Queues {
    uint32_t *slots[N_QUEUES];      // material queues (+ environment queue): slot ids of the current buffer
    uint32_t *counts;               // [bounce][N_BSDF_TYPES] queue sizes, + in/out counters, see api.cu
};

struct RenderCfg {
    uint32_t seed_value;   // sampler base_seed + render seed
    uint32_t spp;
    uint32_t max_depth, rr_depth;
    int32_t hide_emitters, prb, adjoint;
    int32_t forward;       // with adjoint = 1: forward-mode replay (render_forward): dL = 1, the parameter
                           // derivatives are contracted with DevScene::tangent and summed into `result`
    uint32_t chunk_pix0;   // first local pixel of the chunk (index into pix_ids)
    uint32_t chunk_lanes;  // lanes in this chunk
};

// launch geometry
constexpr int BLOCK = 256;
constexpr int BLOCK_SHADE = 128;   // shading kernels: 128 threads x <=128 registers -> 4 blocks / SM

struct Launch { int grid; size_t smem_trace, smem_tables; uint32_t n_smem_nodes, n_smem_tris; int refill_idle;
    bool flat; int grid_flat;      // scenes of <= 32 leaves: flat traversal (kernels.cu: k_trace_flat), its own grid
};

// counters in the stats buffer
enum { ST_BOUNCES = 0, ST_SHADOW = 1, ST_CLOSEST = 2, ST_COUNT = 8 };

void launch_generate(const DevScene &sc, const RenderCfg &cfg, const uint32_t *pix_ids, PathBuf buf, const float4 *adj_dL_lane,
                     const float4 *adj_L_lane, int grid, cudaStream_t st);
void launch_trace(const DevScene &sc, const RenderCfg &cfg, PathBuf cur, float4 *hit, const uint32_t *n_in, Queues q, uint32_t *qcounts,
                  float4 *lane_result, unsigned long long *stats, bool first, const Launch &L, cudaStream_t st);
void launch_shade(int type, const DevScene &sc, const RenderCfg &cfg, PathBuf cur, const float4 *hit, const uint32_t *queue,
                  const uint32_t *qcount, PathBuf nxt, uint32_t *nxt_count, float4 *lane_result, unsigned long long *stats, const Launch &L, cudaStream_t st);
void launch_shade_env(const DevScene &sc, const RenderCfg &cfg, PathBuf cur, const uint32_t *queue, const uint32_t *qcount,
                      float4 *lane_result, unsigned long long *stats, int grid, cudaStream_t st);
void launch_flush(PathBuf cur, Queues q, const uint32_t *qcounts, float4 *lane_result, int grid, cudaStream_t st);
void launch_refit(const DevScene &sc, float *tight, const uint32_t *level_start, uint32_t n_levels, int grid, cudaStream_t st);
void launch_env_query(const DevScene &sc, uint32_t n, const float *in, float *out, cudaStream_t st);
void launch_splat(const DevScene &sc, const RenderCfg &cfg, const uint32_t *pix_ids, const float4 *lane_result, float *film, int grid, cudaStream_t st);
void launch_splat_adjoint(const DevScene &sc, const RenderCfg &cfg, const uint32_t *pix_ids, const float *grad_in, const float *film_w,
                          float4 *lane_dL, int grid, cudaStream_t st);
void launch_weights(const DevScene &sc, const RenderCfg &cfg, const uint32_t *pix_ids, float *film, int grid, cudaStream_t st);
void launch_develop(const DevScene &sc, const float *film, float *out, cudaStream_t st);
void launch_ray_intersect(const DevScene &sc, uint32_t n, const float *rays, float *t, float *uv, uint32_t *prim, int32_t *shape, const Launch &L, cudaStream_t st);
void launch_ray_test(const DevScene &sc, uint32_t n, const float *rays, uint8_t *hit, const Launch &L, cudaStream_t st);
void set_trace_smem_attr(size_t bytes);
void read_watchdog(unsigned long long out[4]);   // debugging builds (-DB200PT_WATCHDOG); zeros otherwise
void launch_bsdf_eval(const DevScene &sc, uint32_t bsdf, int type, uint32_t n, const float *in, float *out, cudaStream_t st);

} // namespace pt
