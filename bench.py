#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200 path tracer (contract: see the task
statement; metric and config: BASELINE.json).

  python bench.py --gpus N --steps K --warmup W            our arm (CUDA, C ABI)
  python bench.py --impl reference --gpus N --steps K ...  reference arm (CPU)

A *step* is one full render of the workload frame: Cornell box 512x512, 256 spp,
path integrator, max_depth 8 (BASELINE.json configs[1]); `value` is Msamples/s
with the scene resident in HBM and the developed image left on the device, `e2e`
is the same metric through the host API (`mitsuba3_b200.render`: parameters
uploaded from host memory, image copied back to the host every step).
N > 1: one process per GPU (torchrun), frame sharded by pixel tiles, ONE NCCL
all-reduce of the raw film per step. Default `--scaling strong`: the SAME frame
(512x512x256 spp) is split over the N GPUs, which is the split BASELINE.json's
north_star describes; `--scaling weak` renders spp = 256 * N (fixed work per GPU).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (width, height, spp per GPU, max_depth, rfilter)
    "cornell_box_512x512_256spp_8bounce": (512, 512, 256, 8, "gaussian"),
    "cornell_box_256x256_64spp_8bounce": (256, 256, 64, 8, "gaussian"),
    # stand-in for BASELINE.json configs[4] (`bathroom2` is not in the reference tree): Cornell box whose floor is a
    # 204 800-triangle heightfield, at the config's stated size and at a size one GPU renders in a second
    "heightfield205k_1920x1080_512spp_8bounce": (1920, 1080, 512, 8, "gaussian"),
    "heightfield205k_1024x1024_64spp_8bounce": (1024, 1024, 64, 8, "gaussian"),
    # BASELINE.json configs[3]: the reference's own asset resources/data/scenes/matpreview (meshes + envmap extracted
    # into tests/golden/matpreview_scene.npz by tests/golden/gen_matpreview.py), principled BSDF on the preview object
    "matpreview_1024x1024_128spp_8bounce": (1024, 1024, 128, 8, "gaussian"),
    # synthetic unit-test scene of the same flavour (principled spheres + procedural envmap)
    "matpreview_like_1024x1024_128spp_8bounce": (1024, 1024, 128, 8, "gaussian"),
}
DEFAULT_WORKLOAD = "cornell_box_512x512_256spp_8bounce"
METRIC = "Msamples/sec (fwd path, Cornell box)"


def build_scene(workload, textured_wall=False):
    import mitsuba3_b200 as mb
    w, h, spp, md, rf = WORKLOADS[workload]
    if workload.startswith("heightfield"):
        d = mb.cornell_box_heightfield(320)
    elif workload.startswith("matpreview_like"):
        d = mb.matpreview_like()
    elif workload.startswith("matpreview"):
        d = mb.matpreview_scene()
    else:
        d = mb.cornell_box()
    if textured_wall and "back" in d:
        # BASELINE.json configs[2] / SURVEY 8(d): the back wall's albedo is a 64x64x3 bitmap texture (initial 0.5,
        # bilinear, clamp, raw) -- the parameter the PRB gradient step differentiates
        d["wall-tex"] = {"type": "diffuse", "reflectance": {"type": "bitmap", "data": np.full((64, 64, 3), 0.5, np.float32), "raw": True,
                                                            "filter_type": "bilinear", "wrap_mode": "clamp"}}
        d["back"]["bsdf"] = {"type": "ref", "id": "wall-tex"}
    d["sensor"]["film"].update(width=w, height=h, rfilter={"type": rf})
    d["sensor"]["sampler"]["sample_count"] = spp
    d["integrator"] = {"type": "path", "max_depth": md}
    return mb.load_dict(d), (w, h, spp, md, rf)


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True); self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def effective_cores():
    """Host threads this process can really use: the affinity mask capped by the cgroup CPU quota (a 128-CPU box
    leased with a 32-CPU quota has 128 `os.cpu_count()` CPUs and 32 effective ones)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]           # cgroup v2
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:                                                                  # cgroup v1
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    eff = n if quota is None else max(1, min(n, int(quota + 0.5)))
    return eff, {"affinity": n, "cgroup_quota": quota, "os_cpu_count": os.cpu_count()}


def cpu_baseline_port(scene, spp_sample):
    """CPU oracle (port of the reference algorithm, OpenMP over pixels) on a bounded sample."""
    from oracle import oracle
    o = oracle.OracleScene(scene)
    H, W, _ = scene.film_shape
    o.render(spp=1, seed=0, mode=0)                      # warm-up (page-in, thread pool)
    t0 = time.perf_counter()
    o.render(spp=spp_sample, seed=0, mode=0)
    dt = time.perf_counter() - t0
    return W * H * spp_sample / dt / 1e6, dt


def cpu_baseline_reference(workload, spp_sample, reps=1, prb_spp=0):
    """The UNMODIFIED reference on all host threads when its runtime travels with the repo (oracle/build_ref.sh ->
    oracle/_ref): `llvm_ad_rgb` -- the variant BASELINE.json names, Dr.Jit's LLVM backend started through
    oracle/llvm_shim -- else `scalar_rgb`. None when no runtime is present or the workload has no reference scene."""
    from oracle.ref_env import reference_env
    env = reference_env(ROOT)
    if env is None or not (workload.startswith("cornell_box") or (workload.startswith("matpreview_") and not workload.startswith("matpreview_like"))):
        return None
    w, h, spp, md, rf = WORKLOADS[workload]
    for variant in ("llvm_ad_rgb", "scalar_rgb"):
        try:
            # the JIT variant renders the frame at its full sample count, three times (~10-20 s of CPU work on the
            # 16-core lease); the scalar variant gets the bounded sample
            vs, vr = (spp, max(reps, 3)) if variant == "llvm_ad_rgb" else (spp_sample, reps)
            r = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "ref_bench.py"), variant, workload, str(w), str(h), str(vs), str(md), rf,
                                str(vr), str(min(prb_spp, vs))], env=env, capture_output=True, text=True, timeout=1500)
            j = json.loads(r.stdout.strip().splitlines()[-1])
            if "error" not in j:
                j["spp_sample"] = vs
                return j
            print("reference arm:", j["error"], file=sys.stderr)
        except Exception as e:      # noqa: BLE001
            print("reference arm:", variant, e, file=sys.stderr)
    return None


def cpu_baseline(scene, workload, spp1, prb=False):
    """Reported CPU baseline on a bounded sample (same frame, fewer spp): the reference itself when
    available, else the oracle port."""
    cores, detail = effective_cores()
    spp_sample = max(1, min(spp1, int(round(32 * cores / 8))))
    w, h, _, md, _ = WORKLOADS[workload]
    ref = cpu_baseline_reference(workload, spp_sample, prb_spp=min(64, spp_sample) if prb else 0)
    if ref is not None:
        out = {"value": ref["msamples_per_s"], "unit": "Msamples/s", "cores": cores, "cores_detail": detail, "threads": ref.get("threads"),
               "kind": "reference", "seconds": ref["seconds"], "variant": ref["variant"], "accel": ref["accel"],
               "sample": f"mitsuba {ref['version']} {ref['variant']}, {ref['accel']}, {cores} effective host cores ({ref.get('threads')} Dr.Jit threads), "
                         f"same frame {w}x{h}, max_depth {md}, {ref['spp_sample']} of {spp1} spp ({ref['seconds']:.1f} s per render)"}
        if "prb_ms_per_grad_step" in ref:
            # scaled linearly in spp to the GPU arm's 64 spp gradient step when the sample used fewer
            out["prb"] = {"ms_per_grad_step": ref["prb_ms_per_grad_step"] * 64.0 / ref["prb_spp"], "measured_spp": ref["prb_spp"],
                          "what": "mi.render(scene, params, spp) with the prb integrator + dr.backward(mean(image)), wall albedo 64x64x3 bitmap; "
                                  "time at measured_spp scaled to 64 spp"}
        elif "prb_error" in ref:
            out["prb"] = {"error": ref["prb_error"]}
        return out
    spp_sample = max(1, spp_sample // 2)
    v, dt = cpu_baseline_port(scene, spp_sample)
    return {"value": v, "unit": "Msamples/s", "cores": cores, "cores_detail": detail, "kind": "port", "seconds": dt,
            "sample": f"CPU oracle (OpenMP, {cores} effective host cores), same frame {w}x{h}, max_depth {md}, {spp_sample} of {spp1} spp ({dt:.1f} s)"}


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path on the host cores -- the unmodified mitsuba
    (llvm_ad_rgb with Embree when the runtime under oracle/_ref can start it, else scalar_rgb), else the CPU oracle
    that restates it (pinned per pixel to the reference's renders, DESIGN.md section 4)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    scene, (w, h, spp, md, rf) = build_scene(args.workload)
    vals = []
    base = None
    for _ in range(max(1, args.steps)):
        base = cpu_baseline(scene, args.workload, spp, prb=not args.no_prb)
        vals.append(base["value"])
    v = float(np.mean(vals))
    base["value"] = v
    out = {
        "impl": "reference", "metric": METRIC if args.workload.startswith("cornell") else "Msamples/sec (fwd path, %s)" % args.workload,
        "value": v, "unit": "Msamples/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": base["seconds"] * 1e3, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "parallelism": "host cores", "sample": base["sample"]},
        "cpu_baseline": base,
        "e2e": {"value": v, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if "prb" in base:
        out["prb"] = base["prb"]
    print(json.dumps(out))
    return 0


def e2e_mi_render(workload, steps, device):
    """The same metric through `mi.render(scene)` of a LIVE, unmodified Mitsuba whose scene names the registered
    `b200_path` integrator (tools/bench_mi_render.py in the environment of oracle/_ref). None without the runtime."""
    from oracle.ref_env import reference_env
    env = reference_env(ROOT)
    if env is None or not workload.startswith("cornell_box"):
        return None
    w, h, spp, md, rf = WORKLOADS[workload]
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_mi_render.py"), str(w), str(h), str(spp), str(md), rf, str(steps), str(device)],
                           env=env, capture_output=True, text=True, timeout=900)
        # the JSON object sits on the last stdout line, possibly behind a log message of the host Mitsuba on the same line
        line = r.stdout.strip().splitlines()[-1]
        return json.loads(line[line.index('{"value"'):])
    except Exception as e:      # noqa: BLE001
        tail = ""
        try:
            tail = (r.stdout[-300:] + " | " + r.stderr[-500:]).replace("\n", " ")
        except Exception:
            pass
        return {"error": f"{type(e).__name__}: {str(e)[:160]}", "output_tail": tail}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write every array as <out_dir>/<name>.npy in float32. When all of them together exceed DUMP_LIMIT_BYTES, an array
    larger than its even share of the limit is replaced by a fixed sample of its rows along the first two axes (pixels
    of an image): seed 0, sorted, so two runs with the same arguments sample the same pixels."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v, np.float32) for k, v in arrays.items()}
    share = DUMP_LIMIT_BYTES // max(1, len(arrays))
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_LIMIT_BYTES and a.nbytes > share and a.ndim >= 2:
            rows = a.reshape((a.shape[0] * a.shape[1],) + a.shape[2:])
            n = max(1, share // (rows.nbytes // rows.shape[0]))
            a = rows[np.sort(np.random.default_rng(0).choice(rows.shape[0], n, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps of every timed loop (device render, e2e, PRB gradient step)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--prb", action="store_true", help="(default on) also time the PRB gradient step (ms/grad-step)")
    ap.add_argument("--no-prb", action="store_true", help="skip the PRB gradient-step timing")
    ap.add_argument("--no-mi-render", action="store_true", help="skip the e2e leg through a live mi.render")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step of each timed loop returned as DIR/<name>.npy "
                         "(float32; image, e2e_image, prb_image, prb_grad.<parameter>); inputs and seeds depend only on the arguments")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    if os.environ.get("B200PT_HANG_DUMP"):      # debugging aid: python stacks of all threads after N seconds
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ["B200PT_HANG_DUMP"]), exit=False)
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import __graft_entry__ as g
    g.build()
    import mitsuba3_b200 as mb
    from mitsuba3_b200 import dist as mbd
    from mitsuba3_b200.integrators import PathIntegrator, PRBIntegrator, device_scene, update_params

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    if args.gpus != world and rank == 0 and world > 1:
        print(f"warning: --gpus {args.gpus} but WORLD_SIZE {world}", file=sys.stderr)
    n_gpus = world
    dev = f"cuda:{local}"

    os.environ.setdefault("B200PT_PROFILE", "1")          # per-launch CUDA events around the traversal kernel
    scene, (w, h, spp1, md, rf) = build_scene(args.workload)
    spp = spp1 * n_gpus if args.scaling == "weak" else spp1
    integ = PathIntegrator(max_depth=md)
    ds = device_scene(scene, local)
    samples_per_step = w * h * spp

    def step_device(seed):
        return mbd.render_distributed(scene, integ, seed=seed, spp=spp, device=local)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for i in range(args.warmup):
        step_device(1000 + i)
    # the clock sampler (an nvidia-smi subprocess per rank) starts BEFORE the barrier: its start-up time must not sit
    # between the barrier and the first event of a rank
    clocks = ClockSampler(local); clocks.start()
    time.sleep(0.3)
    sync_all()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = bounces = shadow = trace_launches = trace_rays = 0
    trace_ms = 0.0
    t0 = time.perf_counter(); ev0.record()
    for i in range(args.steps):
        image = step_device(i)      # working set per step (wavefront state) >> L2, see DESIGN.md; nothing here waits for the device
    ev1.record()
    sync_all()
    wall = time.perf_counter() - t0
    own_ms = ev0.elapsed_time(ev1)
    outputs = {}
    if args.dump_outputs:
        outputs["image"] = image.cpu().numpy()     # the buffer is overwritten by the next render
    clk = clocks.stop()
    dev_ms = max_over_ranks(own_ms)
    ms_per_step = dev_ms / args.steps
    value = samples_per_step / (ms_per_step * 1e-3) / 1e6
    # per-rank device time of the timed region (events of every rank), gathered for the limiter analysis
    per_rank_ms = [own_ms / args.steps]
    if world > 1:
        tl = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(tl, torch.tensor([own_ms / args.steps], dtype=torch.float64, device=dev))
        per_rank_ms = [float(t.item()) for t in tl]

    # ---- per-kernel statistics: a separate, UNTIMED pass (reading them back synchronises the host with the device) -----
    stat_steps = min(3, args.steps)
    render_ms = []
    for i in range(stat_steps):
        step_device(i)
        st = ds.stats()
        launches += st["kernel_launches"]; bounces += st["bounces"]; shadow += st["shadow_rays"]
        trace_ms += st["trace_ms"]; trace_launches += st["trace_launches"]; trace_rays += st["trace_rays"]
        render_ms.append(st["device_ms"])
    launches_per_step = launches / stat_steps
    # the film all-reduce alone (NCCL, in place on the cached raw block), device-timed
    allreduce_us = None
    if world > 1:
        film = ds._dist_bufs[0]
        for _ in range(3):
            mbd.all_reduce_film(film)
        sync_all()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(20):
            mbd.all_reduce_film(film)
        a1.record(); sync_all()
        allreduce_us = max_over_ranks(a0.elapsed_time(a1) / 20 * 1e3)
    own_render_ms = float(np.mean(render_ms))          # this rank's kernels only (b200pt_render_accumulate), no collective
    render_ms_ranks = [own_render_ms]
    if world > 1:
        tl = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(tl, torch.tensor([own_render_ms], dtype=torch.float64, device=dev))
        render_ms_ranks = [float(t.item()) for t in tl]

    # ---- e2e: host API, params uploaded + image copied back every step -------------------
    names = scene.parameters()
    h2d = sum(scene.textures[i].size * 4 for i in names.values())
    img_bytes = w * h * 3 * 4
    pinned = torch.empty((h, w, 3), dtype=torch.float32).pin_memory()          # the step's result lands in pinned host memory
    pinned_np = pinned.numpy()

    def step_host(seed):
        update_params(scene, {k: scene.textures[i].array() for k, i in names.items()}, local)
        if world == 1:
            return integ.render(scene, seed=seed, spp=spp, device=local, out=pinned_np)
        pinned.copy_(mbd.render_distributed(scene, integ, seed=seed, spp=spp, device=local), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return pinned.numpy()
    for i in range(3):
        step_host(77 + i)
    sync_all()
    host_ms = []
    t1 = time.perf_counter()
    for i in range(args.steps):
        t_s = time.perf_counter()
        img = step_host(i)
        host_ms.append((time.perf_counter() - t_s) * 1e3)
    sync_all()
    e2e_s = max_over_ranks((time.perf_counter() - t1) / args.steps)
    if args.dump_outputs:
        outputs["e2e_image"] = np.array(img)
    e2e = {"value": samples_per_step / e2e_s / 1e6, "unit": "Msamples/s", "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": img_bytes, "checksum": float(np.asarray(img).mean()),
           "per_step_ms": [round(x, 3) for x in host_ms],      # rank 0: wall time of every timed host step (an outlier shows here)
           "api": "mitsuba3_b200.render -> b200pt_render (C ABI), host buffers in and out, wall clock, max over ranks"}

    # ---- PRB gradient step (BASELINE.json: "ms/grad-step (PRB)"): primal + adjoint, device-timed -------
    prb = None
    if not args.no_prb and args.workload.startswith("cornell"):
        pint = PRBIntegrator(max_depth=md)
        scene_p, _ = build_scene(args.workload, textured_wall=True)      # configs[2]: wall albedo texture is the parameter
        gi = torch.full((h, w, 3), 1.0 / (h * w * 3), device=dev)
        spp_g = 64 * n_gpus if args.scaling == "weak" else 64
        n_grad = args.steps
        for i in range(2):
            mbd.render_distributed(scene_p, pint, seed=50 + i, spp=spp_g, device=local)
            mbd.render_backward_distributed(scene_p, gi, pint, seed=150 + i, spp=spp_g, device=local)
        sync_all()
        pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        pe0.record()
        for i in range(n_grad):
            prb_image = mbd.render_distributed(scene_p, pint, seed=i, spp=spp_g, device=local)
            grads = mbd.render_backward_distributed(scene_p, gi, pint, seed=100 + i, spp=spp_g, device=local)
        pe1.record()
        sync_all()
        tp = max_over_ranks(pe0.elapsed_time(pe1))
        if args.dump_outputs:
            outputs["prb_image"] = prb_image.cpu().numpy()
            outputs.update({f"prb_grad.{k}": v for k, v in grads.items()})
        pst = device_scene(scene_p, local).stats()
        n_params = int(sum(t.size for t in scene_p.textures if t.differentiable))
        # bytes of path state the gradient step streams (DESIGN.md section 5): primal pass + adjoint's own primal pass at
        # 144 + 304 b per sample each, replay at 144 + (304 + 64) b (adj_L, adj_dL read + written per vertex)
        prb = {"ms_per_grad_step": tp / n_grad, "spp": spp_g, "grad_steps": n_grad, "differentiated_floats": n_params,
               "what": "wall albedo = 64x64x3 bitmap texture; primal render + render_backward (PRB adjoint, atomicAdd gradient scatter%s), CUDA events, "
                       "max over ranks, max_depth %d" % (" + gradient all-reduce" if world > 1 else "", md),
               "adjoint_device_ms": pst["device_ms"], "adjoint_launches": pst["kernel_launches"]}

    mi_e2e = None
    if rank == 0 and world == 1 and not args.no_mi_render:
        mi_e2e = e2e_mi_render(args.workload, args.steps, local)

    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
        lanes_rank0 = max(1, (samples_per_step // n_gpus) * stat_steps)
        b_bar = bounces / lanes_rank0   # rank 0's lanes
        # dominant kernel: k_trace. Algorithmic bytes per ray (DESIGN.md "Roofline"): closest-hit ray 28 B read +
        # 20 B hit record written; shadow ray 40 B record read + 24 B result read-modify-write.
        closest = trace_rays - shadow
        trace_bytes = closest * 48.0 + shadow * 64.0
        trace_avg_ms = trace_ms / max(1, trace_launches)
        trace_gbs = trace_bytes / max(trace_ms * 1e-3, 1e-12) / 1e9 if trace_ms > 0 else None
        # DRAM traffic of the dominant kernel per launch: NOT measured in this run -- the per-ray constant of the committed
        # `ncu --set full` capture (profiles/*_trace_traffic.json: dram__bytes_{read,write}.sum over all traversal launches
        # of a frame / rays traced) times the rays one launch of this run processed
        traffic = None; traffic_src = None
        for fn in (("r02_trace_traffic.json", "r01_trace_traffic.json") if args.workload.startswith("cornell") else ()):
            try:
                tj = json.load(open(os.path.join(ROOT, "profiles", fn)))
                traffic = tj["dram_bytes_per_ray"] * trace_rays / max(1, trace_launches)
                traffic_src = f"ncu constant {tj['dram_bytes_per_ray']:.1f} B/ray (profiles/{fn}) x rays per launch of this run; not measured in this run"
                break
            except Exception:
                continue
        step_bytes = (144.0 + 304.0 * b_bar) * (samples_per_step // n_gpus)
        rank0_ms = float(np.mean(render_ms))
        step_gbs = step_bytes / (rank0_ms * 1e-3) / 1e9
        out = {
            "metric": METRIC if args.workload.startswith("cornell") else "Msamples/sec (fwd path, %s)" % args.workload, "value": value, "unit": "Msamples/s", "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "spp_total": spp, "global_samples_per_step": samples_per_step,
                       "parallelism": f"pixel-tile x{n_gpus} (32x32 tiles, diagonal deal), 1 film all-reduce" if n_gpus > 1 else "single GPU",
                       "l2": "wavefront state per chunk (hundreds of MB to GB) > L2 (126 MB); film and scene are L2-resident by design",
                       "mean_bounces_per_sample": b_bar},
            "e2e": e2e, "gpu_launches": int(round(launches_per_step * args.steps)), "clocks": clk, "wall_ms_per_step": wall / args.steps * 1e3,
            "per_rank": {"step_ms": per_rank_ms, "render_kernels_ms": render_ms_ranks, "film_allreduce_us": allreduce_us,
                         "imbalance": (max(render_ms_ranks) / (sum(render_ms_ranks) / len(render_ms_ranks)) - 1) if render_ms_ranks else None,
                         "note": "step_ms: CUDA events around the timed region of every rank / steps; render_kernels_ms: the rank's own kernels of a frame "
                                 "(no collective), separate untimed pass; film_allreduce_us: 20 back-to-back all-reduces of the raw film, max over ranks"},
            "roofline": {"kernel": ("k_trace_flat (<= 32 leaves: every lane tests every leaf box, warp-shared exact triangle tests; NEE shadow ray + closest hit)"
                                    if args.workload.startswith("cornell") else "k_trace_dyn (BVH walk with dynamic fetch: NEE shadow ray + closest hit)"), "bound": "hbm",
                         "achieved": trace_gbs, "peak": hbm_peak, "unit": "GB/s",
                         "frac": (trace_gbs / hbm_peak) if trace_gbs else None, "traffic": traffic, "traffic_source": traffic_src,
                         "algorithmic_bytes_per_launch": trace_bytes / max(1, trace_launches), "peak_source": peak_src,
                         "avg_launch_ms": trace_avg_ms, "launches": int(trace_launches), "rays_per_launch": trace_rays / max(1, trace_launches),
                         "share_of_step": trace_ms / max(sum(render_ms), 1e-9), "measured_on": f"{stat_steps} untimed frames after the timed region (rank 0)",
                         "step": {"bytes_per_sample": 144.0 + 304.0 * b_bar, "achieved": step_gbs, "frac": step_gbs / hbm_peak}},
        }
        if mi_e2e is not None:
            out["e2e_mi_render"] = mi_e2e
        if prb:
            out["prb"] = prb
        if not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(scene, args.workload, spp1, prb=prb is not None)
            if prb and "prb" in out["cpu_baseline"]:
                prb["reference"] = out["cpu_baseline"]["prb"]
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
