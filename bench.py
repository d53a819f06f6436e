#!/usr/bin/env python3
"""bench.py -- Msamples/s (pixels x spp) of the volumetric render pass, BASELINE.json's metric.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--config C] [--dump-outputs DIR]

Default workload (the one the metric is quoted on): BASELINE.json configs[1] -- dragon.vdb, 1920x1080, 64 spp per step,
ray_depth 100, volume_depth 1, direct integrator, sun + HDRI environment: 132.7 M samples per step.  `--config 1|3|4|5`
selects the other BASELINE configurations (measurement table of BASELINE.md; see WORKLOADS below).
  * ours      : vpt_render_passes(spp) through the C ABI (libvpt_b200.so).  N > 1 shards the frame by interleaved row
                stripes over N ranks (scene replicated) and gathers the rank-local accumulators with NCCL.
  * reference : the reference's own `volume_rt_kernel` (oracle/_ref, compiled from /root/reference), launched as
                source/main.cpp:1823-1829 does: one launch + cudaDeviceSynchronize per spp, on the REFERENCE's own octree.
                The reference has no CPU path and no multi-GPU path: rank 0 runs it on one GPU.
Rank 0 prints ONE JSON line.  Timing: CUDA events on the launching stream around each step, L2 flushed between steps
(untimed), barrier + synchronize on both sides, max over ranks.  After the timed region (untimed) the frame of the timed
configuration is rendered once more from a fresh state and compared with the reference kernel's frame ("parity"); with
N > 1 rank 0 also checks that the gathered frame equals its own single-GPU frame bit for bit.  A parity failure exits non-zero.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np
import torch

METRIC = "Msamples/sec (pixels x spp) on dragon.vdb 1920x1080"
RTOL, ATOL, MAX_FLIPPED = 1e-4, 1e-5, 1e-3        # the parity tolerance of tests/test_parity_gpu.py


# ---------------------------------------------------------------------------------------------------------------------
# workloads: BASELINE.json configs, made concrete in SURVEY.md 8(d)
# ---------------------------------------------------------------------------------------------------------------------
def _kp(V, **over):
    kp = V.default_kernel_params()
    kp.environment_type = 1; kp.max_interactions = 100000
    for k, v in over.items(): setattr(kp, k, v)
    return kp


def build_workload(V, cfg, dev):
    """-> dict(name, scene, kp, width, height, spp, data, ref_ok)"""
    hdri = "Barce_Rooftop_C_3k.hdr"
    if cfg in (1, 2):
        vol = V.Volume.load_vdb(V.find_asset("dragon.vdb"))
        scene = V.Scene([vol.instance()], device=dev, env=hdri)
        if cfg == 1:
            return dict(name="dragon.vdb 512x512 1spp ray_depth=1 single scatter, sun + HDRI env (BASELINE configs[0]; the survey's environment_type 0 "
                             "needs the Bruneton tables, see --config 1 note in BASELINE.md)", scene=scene, kp=_kp(V, ray_depth=1, volume_depth=1),
                        width=512, height=512, spp=1, data="dragon.vdb (reference asset)", keep=[vol])
        return dict(name="dragon.vdb 1920x1080 64spp ray_depth=100 volume_depth=1 direct integrator, sun + HDRI env (BASELINE configs[1])",
                    scene=scene, kp=_kp(V, ray_depth=100, volume_depth=1, integrator=0), width=1920, height=1080, spp=64,
                    data="dragon.vdb (reference asset)", keep=[vol])
    if cfg == 3:
        p = V.find_asset("fireball.vdb")
        if p is None: raise SystemExit("fireball.vdb is not staged (oracle/_ref/assets)")
        vol = V.Volume.load_vdb(p)
        scene = V.Scene([vol.instance()], device=dev, env=hdri)
        return dict(name="fireball.vdb 1920x1080 256spp emission + multiple scatter (ray_depth=2, volume_depth=50), sun + HDRI env (BASELINE configs[2])",
                    scene=scene, kp=_kp(V, ray_depth=2, volume_depth=50, emission_scale=1.0, emission_pivot=1.0), width=1920, height=1080, spp=256,
                    data="fireball.vdb density + heat (reference asset)", keep=[vol])
    if cfg == 4:
        n = int(os.environ.get("VPT_BENCH_GRID", "1024"))
        vol = V.Volume.procedural((n, n, n), scale=0.1, seed=123, device=dev)
        scene = V.Scene([vol.instance()], device=dev, env=hdri)
        return dict(name=f"synthetic {n}^3 Perlin-noise density grid ({n ** 3 * 4 / 2 ** 30:.1f} GiB fp32, perlinNoise scale 0.1 seed 123, zero jitter), 1920x1080 128spp, "
                         "defaults (ray_depth 50, volume_depth 1), sun + HDRI env (BASELINE configs[3])",
                    scene=scene, kp=_kp(V), width=1920, height=1080, spp=128, data=f"procedural {n}^3 grid (vpt_procedural_fill)", keep=[vol], volume=vol)
    if cfg == 5:
        vol = V.Volume.load_vdb(V.find_asset("dragon.vdb"))
        n = int(os.environ.get("VPT_BENCH_INSTANCES", "1000"))
        # fixed LCG: positions uniform in a cube, random unit quaternions, scale 1 (SURVEY 8(d) cfg 5)
        state = 12345
        def lcg():
            nonlocal state
            state = (1103515245 * state + 12345) & 0x7fffffff
            return state / float(0x7fffffff)
        inst = []
        side = 6.0 * n ** (1.0 / 3.0)
        for _ in range(n):
            pos = tuple((lcg() - 0.5) * side for _ in range(3))
            q = np.array([lcg() - 0.5 for _ in range(4)]); q /= max(np.linalg.norm(q), 1e-6)
            inst.append(vol.instance(pos=pos, quat=tuple(q), scale=1.0))
        scene = V.Scene(inst, device=dev, env=hdri)
        return dict(name=f"{n} x dragon.vdb instances (LCG placement), 1920x1080 64spp ray_depth=50, sun + HDRI env (BASELINE configs[4])",
                    scene=scene, kp=_kp(V, ray_depth=50, volume_depth=1), width=1920, height=1080, spp=64,
                    data=f"dragon.vdb x {n} instances", keep=[vol], ref_max_instances=600)
    raise SystemExit(f"--config {cfg} is not available in this build")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md).  The sampler is started before the
    warm-up (nvidia-smi needs ~1 s to start) and samples are kept by timestamp inside the timed window."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index; self.proc = None; self.lines = []; self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.gpu)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True); self.t.start()
            time.sleep(1.5)
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def window(self, t0, t1):
        self.t0, self.t1 = t0, t1

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try: self.proc.wait(timeout=2)
        except Exception: self.proc.kill()
        def parse(lines):
            sm, smax, reasons = [], None, set()
            for _, ln in lines:
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 9: continue
                try:
                    sm.append(float(f[1])); smax = float(f[2])
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"): reasons.add(name)
            return sm, smax, reasons
        inside = [x for x in self.lines if self.t0 is not None and self.t0 - 0.02 <= x[0] <= self.t1 + 0.05]
        sm, smax, reasons = parse(inside if inside else self.lines[-10:])
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm),
                "window_s": None if self.t0 is None else round(self.t1 - self.t0, 4)}


def flush_l2(buf):
    buf.add_(1)      # 256 MiB read+write > 126 MB L2


def timed_steps(step_fn, steps, warmup, dist, flush_buf, sampler=None):
    for _ in range(warmup):
        step_fn()
    torch.cuda.synchronize()
    if dist is not None: dist.barrier()
    torch.cuda.synchronize()
    evs = []
    wall0 = time.perf_counter(); tw0 = time.time()
    for _ in range(steps):
        flush_l2(flush_buf)
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record(); step_fn(); b.record()
        evs.append((a, b))
    torch.cuda.synchronize()
    if dist is not None: dist.barrier()
    torch.cuda.synchronize()
    wall = time.perf_counter() - wall0
    if sampler is not None: sampler.window(tw0, time.time())
    ms = sum(a.elapsed_time(b) for a, b in evs)
    if dist is not None:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms, wall


def dump_outputs(out_dir, arrays):
    """--dump-outputs: what the timed path computed in its last step, one float32 .npy per array (34 MB at 1920x1080), so
    that two builds run with the same arguments (hence the same inputs) can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().cpu().numpy().astype(np.float32))


def cpu_baseline_sample(V, scene, cam, kp, width, height, seconds_target=12.0):
    """CPU restatement (oracle/vpt_oracle.c, 'port') timed on the host cores over a bounded sample of the same workload."""
    try:
        import oracle_cpu
    except Exception as e:                                     # pragma: no cover
        return {"value": None, "unit": "Msamples/s", "cores": 0, "kind": "port", "sample": f"unavailable: {e}"}
    return oracle_cpu.timed_sample(scene, cam, kp, width, height, seconds_target)


def frame_parity(got, want):
    got = np.asarray(got, dtype=np.float64); want = np.asarray(want, dtype=np.float64)
    d = np.abs(got - want)
    bad = (d > ATOL + RTOL * np.abs(want)).reshape(-1, 3).any(axis=1)
    return {"flipped_frac": float(bad.mean()), "max_abs": float(d.max()), "pixels": int(bad.size),
            "tolerance": f"|d| <= {ATOL} + {RTOL}*|ref| per channel; flipped_frac must stay <= {MAX_FLIPPED}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, help="BASELINE.json configuration (1-based); 2 is the one the metric is quoted on")
    ap.add_argument("--chunk", type=int, default=0, help="passes fused per kernel round (0 = library default)")
    ap.add_argument("--sched-min-lanes", type=int, default=0, help="trace scheduler threshold (0 = library default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the (untimed) check of the timed frame against the reference kernel")
    ap.add_argument("--generic-kernel", action="store_true", help="A/B: force the generic trace kernel instantiation")
    ap.add_argument("--ref-jit61", action="store_true", help="with --impl reference: load the reference kernel as compute_61 PTX (its shipped form) and let the driver JIT it")
    ap.add_argument("--level-a", action="store_true", help="time the level (A) module: volume_rt_kernel_b200.cubin loaded and launched through the "
                    "Driver API exactly like the reference kernel (one launch + synchronize per spp), instead of the wavefront library")
    ap.add_argument("--cells", action="store_true", help="config 4: trace from the cell table (8 corner texels per cell = one 32-byte sector per look-up, software filter) instead of the 3-D texture")
    ap.add_argument("--fast", action="store_true", help="config 4: trace from the brick pool (TMA-staged software sampler) instead of the 3-D texture")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last step's frame (accum, depth) and blue-noise "
                    "state as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        torch.cuda.set_device(local)
        dist_mod.init_process_group(backend="nccl", device_id=torch.device(f"cuda:{local}"))
        dist = dist_mod
    else:
        torch.cuda.set_device(0)
    if args.impl == "reference" and rank != 0:
        if dist is not None: dist.destroy_process_group()
        return 0

    import vpt_b200 as V
    dev = f"cuda:{local if world > 1 else 0}"
    wl = build_workload(V, args.config, dev)
    scene, kp, WIDTH, HEIGHT, SPP = wl["scene"], wl["kp"], wl["width"], wl["height"], wl["spp"]
    data = wl["data"] + " + " + ("Barce_Rooftop_C_3k.hdr" if not scene.data_notes else "; ".join(scene.data_notes))
    flush_buf = torch.zeros(64 * 1024 * 1024, dtype=torch.float32, device=dev)
    samples_per_step = WIDTH * HEIGHT * SPP
    sampler = ClockSampler(local if world > 1 else 0)
    config = {"workload": wl["name"], "baseline_config": args.config, "width": WIDTH, "height": HEIGHT, "spp_per_step": SPP,
              "l2": "flushed between steps (256 MiB rewrite, untimed)"}
    n_inst = len(scene.instances)

    if args.impl == "reference":
        import oracle_ref
        if not oracle_ref.available():
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref (the reference kernel build) is not in this snapshot"}), flush=True)
            return 0
        if n_inst > wl.get("ref_max_instances", 10 ** 9):
            # the reference overflows OCTNode::vol_indices[600] beyond 600 instances (quirk Q11): run it on the first 600
            n_inst = wl["ref_max_instances"]
            scene = V.Scene(scene.instances[:n_inst], device=dev, env="Barce_Rooftop_C_3k.hdr")
            config["reference_instances"] = n_inst
        orc = oracle_ref.RefOracle(); orc.load_kernels()
        which = orc.UNMODIFIED
        kernel_note = "source/render_kernel.cu compiled unmodified with -O3 --use_fast_math --maxrregcount=128 for sm_100a"
        if args.ref_jit61:
            # the reference as shipped: PTX for compute_61 (source/CMakeLists.txt:133), JIT-compiled by the driver at module load (untimed)
            orc.load_candidate(os.path.join(oracle_ref.REF_DIR, "render_kernel_ref_cc61.ptx")); which = orc.CANDIDATE
            kernel_note = "source/render_kernel.cu as compute_61 PTX (the reference's own build), JIT-compiled by the driver for this GPU"
        r = V.Renderer(scene, WIDTH, HEIGHT, kp=kp)
        r.params.p_oct.value = orc.build_octree(scene.h_volumes, n_inst)      # the reference's own octree builder
        def step():
            r.kp.iteration = 0
            for _ in range(SPP):                               # main.cpp:1823-1829: launch, ++iteration, cudaDeviceSynchronize
                orc.launch(r.params.array, WIDTH, HEIGHT, which, sync=True)
                r.kp.iteration += 1
        sampler.start()
        ms, wall = timed_steps(step, args.steps, args.warmup, None, flush_buf, sampler)
        clocks = sampler.stop()
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"accum": r.buffers.accum, "depth": r.buffers.depth, "blue_noise": scene.d_blue_noise})
        val = samples_per_step * args.steps / (ms * 1e-3) / 1e6
        config.update({"launch_protocol": "reference main loop: 1 launch + cudaDeviceSynchronize per spp, grid (W/16+1,H/16+1)x(16,16)",
                       "kernel": kernel_note,
                       "octree": "reference build_octree (bvh_kernels.cu:582-604)"})
        line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "Msamples/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                "data": data, "config": config, "clocks": clocks, "gpu_launches": SPP * args.steps,
                "cpu_baseline": {"value": val, "unit": "Msamples/s", "cores": 1, "kind": "reference",
                                 "sample": "the reference has no CPU path (BASELINE.json): its own CUDA kernel on 1 B200, 1 host thread driving it, full workload"},
                "e2e": {"value": val, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "wall_s": wall}
        print(json.dumps(line), flush=True)
        return 0

    # ------------------------------------------------------------------------------------------ ours
    opts = {}
    if args.chunk: opts["passes_per_chunk"] = args.chunk
    if args.sched_min_lanes: opts["sched_min_lanes"] = args.sched_min_lanes
    if args.generic_kernel: opts["generic_kernel"] = 1
    for kv in filter(None, os.environ.get("VPT_BENCH_OPTIONS", "").split(",")):     # A/B runs: e.g. VPT_BENCH_OPTIONS=trace_slots=3
        k, v = kv.split("="); opts[k.strip()] = int(v)
    stream = torch.cuda.current_stream().cuda_stream
    if world > 1:
        dr = V.DistributedRenderer(scene, WIDTH, HEIGHT, kp=kp, stripe_rows=8, options=opts, exchange=os.environ.get("VPT_EXCHANGE", "p2p"))
        r = dr.r
        def step():
            r.kp.iteration = 0
            dr.render(SPP, stream=stream)
    elif args.level_a:
        dr = None
        r = V.Renderer(scene, WIDTH, HEIGHT, kp=kp, options=opts)
        mod = V.LevelAModule()
        config["entry"] = "level (A): volume_rt_kernel_b200.cubin via cuModuleLoad / cuModuleGetFunction / cuLaunchKernel, 1 launch + synchronize per spp"
        def step():
            r.kp.iteration = 0
            for _ in range(SPP): mod.launch(r, sync=True)
        r.render = lambda n, stream=None: [mod.launch(r, sync=True) for _ in range(n)]      # parity / profile legs below go through the same entry
    else:
        dr = None
        r = V.Renderer(scene, WIDTH, HEIGHT, kp=kp, options=opts)
        def step():
            r.kp.iteration = 0
            r.render(SPP, stream=stream)

    if args.fast:
        if "volume" not in wl: raise SystemExit("--fast needs a workload with a procedural volume (--config 4)")
        r.set_brick_volume(wl["volume"])
        config["trace_mode"] = f"brick pool ({wl['volume'].brick_bytes / 2 ** 30:.2f} GiB) staged by cp.async.bulk (TMA), the texture unit's filter in software"
    elif args.cells:
        if "volume" not in wl: raise SystemExit("--cells needs a workload with a procedural volume (--config 4)")
        r.set_cell_volume(wl["volume"])
        config["trace_mode"] = f"cell table ({wl['volume'].cell_bytes / 2 ** 30:.2f} GiB: 32 B = one sector per look-up), the texture unit's filter in software"
    else:
        config["trace_mode"] = "parity: tex3D (bit-exact per seed)"
    l0, _ = r.stats()
    sampler.start()
    ms, wall = timed_steps(step, args.steps, args.warmup, dist, flush_buf, sampler)
    clocks = sampler.stop()
    if args.dump_outputs:
        if world > 1:
            full = dr.full_accum().reshape(-1, 3)          # the gathered frame; depth and blue noise stay rank-local
            if rank == 0: dump_outputs(args.dump_outputs, {"accum": full})
        else:
            dump_outputs(args.dump_outputs, {"accum": r.buffers.accum, "depth": r.buffers.depth, "blue_noise": scene.d_blue_noise})
    l1, _ = r.stats()
    launches_per_step = (l1 - l0) // (args.steps + args.warmup)
    value = samples_per_step * args.steps / (ms * 1e-3) / 1e6

    # ---- end to end through the public API with host buffers: parameter blocks from host memory in,
    #      the finished frame (accum float3 + display u32) copied back to pinned host memory, every step
    pin_accum = torch.empty(WIDTH * HEIGHT, 3, dtype=torch.float32).pin_memory()
    pin_disp = torch.empty(WIDTH * HEIGHT, dtype=torch.int32).pin_memory()
    def step_e2e():
        step()
        if world > 1:
            if rank == 0: pin_accum.copy_(dr.full_accum().view(-1, 3), non_blocking=True)
        else:
            pin_accum.copy_(r.buffers.accum, non_blocking=True)
            pin_disp.copy_(r.buffers.display, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    e2e_steps = max(3, args.steps // 2)
    ms_e2e, _ = timed_steps(step_e2e, e2e_steps, 1, dist, flush_buf)
    e2e_val = samples_per_step * e2e_steps / (ms_e2e * 1e-3) / 1e6
    h2d = 104 + 16 + 5 * 8 + 464 + 312                     # the by-value launch parameter block, per render call
    d2h = WIDTH * HEIGHT * (12 + 4) if world == 1 else (WIDTH * HEIGHT * 12 if rank == 0 else 0)

    # ---- parity of the timed configuration (untimed): fresh state, same 64-spp frame, against the reference kernel ------------
    parity = None
    parity_fail = False
    if not args.no_parity:
        scene.reset_blue_noise(); r.kp.iteration = 0; r.buffers.zero_()
        if world > 1:
            dr.render(SPP, stream=stream); full = dr.full_accum().reshape(-1, 3).clone()
        else:
            r.render(SPP, stream=stream); full = r.buffers.accum
        torch.cuda.synchronize()
        if rank == 0:
            parity = {}
            if world > 1:
                scene.reset_blue_noise()
                one = V.Renderer(scene, WIDTH, HEIGHT, kp=_copy_kp(V, kp), cam=r.cam, options=opts)
                if args.fast: one.set_brick_volume(wl["volume"])
                if args.cells: one.set_cell_volume(wl["volume"])
                one.render(SPP, stream=stream); torch.cuda.synchronize()
                parity["gathered_equals_single_gpu_bitwise"] = bool(torch.equal(full, one.buffers.accum))
                parity_fail |= not parity["gathered_equals_single_gpu_bitwise"]
                one.close()
            try:
                import oracle_ref
                have_ref = oracle_ref.available() and n_inst <= 600
            except Exception:
                have_ref = False
            if have_ref:
                orc = oracle_ref.RefOracle()
                ref = V.Renderer(scene, WIDTH, HEIGHT, kp=_copy_kp(V, kp), cam=r.cam)
                ref.params.p_oct.value = orc.build_octree(scene.h_volumes, n_inst)
                scene.reset_blue_noise(); orc.render(ref, SPP)                 # race-free protocol (SURVEY 8(c))
                parity.update(frame_parity(full.cpu().numpy(), ref.buffers.accum.cpu().numpy()))
                parity["against"] = "reference volume_rt_kernel (oracle/_ref), same parameter block, its own octree, same frame as timed"
                parity_fail |= parity["flipped_frac"] > MAX_FLIPPED
            else:
                parity["against"] = "unavailable (oracle/_ref not in this snapshot, or > 600 instances: beyond the reference's capacity)"
        if world > 1: dist.barrier()

    # ---- roofline of the dominant kernel (k_trace), measured live with CUDA events on its stream
    roofline = None
    if rank == 0 and args.level_a:
        roofline = {"bound": "hbm", "kernel": "volume_rt_kernel (level A megakernel)", "achieved": None, "peak": None, "unit": "GB/s", "frac": None, "traffic": None,
                    "note": "the level (A) entry is the strict drop-in, not the measured hot path: no per-kernel breakdown is taken for it"}
    kt = cnt = None
    per_rank_ms = None
    if not args.level_a:
        # rank-local work only, on EVERY rank (per-rank kernel times show the stripe imbalance); the library's all-gather is switched
        # off for these runs -- a collective that only some ranks enter would hang the job
        if dr is not None: dr.set_gather(False)
        def render_only():
            r.kp.iteration = 0
            r.render(SPP, stream=stream)
        r.set_option("profile", 1); r.kernel_times()         # per-kernel CUDA events, production kernels
        for _ in range(2): render_only()
        torch.cuda.synchronize()
        kt = r.kernel_times()
        r.set_option("profile", 0); r.set_option("count_stats", 1); r.counters(reset=True)   # work counters of the SAME instantiation that was timed
        for _ in range(2): render_only()
        torch.cuda.synchronize()
        cnt = r.counters()
        r.set_option("count_stats", 0)
        if dr is not None: dr.set_gather(True)
        if world > 1:
            mine = {k: round(v["ms"] / 2, 4) for k, v in kt.items()}
            gathered = [None] * world
            dist.all_gather_object(gathered, mine)
            per_rank_ms = gathered
    if rank == 0 and not args.level_a:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak = float(json.load(open(peaks_path))["hbm_gbs"]); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak = 6650.0; peak_src = "fallback (B200_PROFILING.md 6.65 TB/s)"
        n_steps_prof = 2
        samples = r.n_local * SPP * n_steps_prof
        launches = max(1, kt["trace"]["launches"])
        t_trace = kt["trace"]["ms"] / launches
        lookups_per_sample = cnt["lookups"] / max(1, samples)
        # k_trace's own algorithmic bytes: 32 B per density lookup (SURVEY 8(d)) + per traced ray a 24-B queue record
        # (+16 B start position) read and a 48-B sample record written
        bytes_trace = 32.0 * cnt["lookups"] + (24.0 + 16.0 + 48.0) * cnt["rays"]
        achieved = bytes_trace / launches / (t_trace * 1e-3) / 1e9
        simt = cnt["lane_steps"] / max(1, 32 * cnt["warp_step_iters"])
        traffic = None
        for name in ("r02_traffic.json", "r01_traffic.json"):
            tpath = os.path.join(ROOT, "profiles", name)
            if os.path.exists(tpath):
                tj = json.load(open(tpath))
                ent = tj if args.config == tj.get("baseline_config", 2) else tj.get("configs", {}).get(str(args.config))
                if ent and not args.fast and not args.cells and world == 1 and ent.get("passes_per_launch") == (opts.get("passes_per_chunk") or 32):
                    traffic = ent["k_trace_dram_bytes_per_launch"]
                break
        bytes_per_sample = 88.0 + 32.0 * lookups_per_sample          # SURVEY 8(d): framebuffer stream + 32 B per density lookup
        step_gbs = value * bytes_per_sample / 1e3
        roofline = {"bound": "hbm", "kernel": "k_trace_brick" if args.fast else "k_trace", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": bytes_trace / launches, "avg_launch_ms": t_trace, "launches_per_step": launches / n_steps_prof,
                    "density_lookups_per_sample": lookups_per_sample, "rays_traced_per_sample": cnt["rays"] / max(1, samples),
                    "bricks_staged_per_lookup": (cnt["brick_fetches"] / max(1, cnt["lookups"])) if args.fast else None,
                    "step_loop_simt_efficiency": simt, "service_round_lanes": cnt["lane_services"] / max(1, cnt["warp_service_rounds"]),
                    "kernel_ms_per_step": {k: v["ms"] / n_steps_prof for k, v in kt.items()}, "kernel_ms_per_step_by_rank": per_rank_ms,
                    "step": {"bytes_per_sample": bytes_per_sample, "achieved": step_gbs, "achieved_per_gpu": step_gbs / world, "frac": step_gbs / world / peak,
                             "note": "whole step charged with SURVEY 8(d)'s 88 B + 32 B x lookups per sample; per-GPU rate over one GPU's peak"},
                    "note": ("4 GiB grid, nothing cache-resident: every look-up is a DRAM round trip (152 B of sector traffic for 32 algorithmic bytes); "
                             "the kernel is bound by memory LATENCY (ncu: 44 % of DRAM throughput, 40 % long-scoreboard stalls); see profiles/r02_cfg4_*") if args.config == 4 else
                            ("the volume is L2-resident (dragon.vdb: 425 KB): look-ups are served by L1/TEX/L2, DRAM only sees the ray queue and the sample planes; "
                             "the path is bound by latency / instruction issue, not HBM (SURVEY 8(d)); see profiles/")}

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and args.config in (1, 2):      # N = 1 only
        cpu_base = cpu_baseline_sample(V, scene, r.cam, kp, WIDTH, HEIGHT)

    if rank == 0:
        config.update({"passes_per_chunk": opts.get("passes_per_chunk", 32), "partition": f"{world} rank(s), interleaved 8-row stripes" if world > 1 else "single GPU",
                       "collective": dr.collective_note if world > 1 else "none", "instances": n_inst})
        line = {"metric": METRIC, "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                "data": data, "config": config, "clocks": clocks,
                "e2e": {"value": e2e_val, "unit": "Msamples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
                "gpu_launches": int(SPP * args.steps) if args.level_a else int(launches_per_step * args.steps), "roofline": roofline, "cpu_baseline": cpu_base, "parity": parity, "wall_s": wall}
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier(); dist.destroy_process_group()
    return 1 if parity_fail else 0


def _copy_kp(V, kp):
    import ctypes as C
    k = V.Kernel_params(); C.memmove(C.byref(k), C.byref(kp), C.sizeof(k)); k.iteration = 0
    return k


if __name__ == "__main__":
    sys.exit(main())
