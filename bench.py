#!/usr/bin/env python
"""bench.py — frames/s of the md_script per-frame hot path on N B200s, next to the reference CPU path.

Metric / config (BASELINE.json): "frames/sec RDF+SDF eval, 100k-atom synthetic traj". Default workload = synthetic water box
n=32 (98 304 atoms, 32 768 O, L = 99.328 A, viamd_b200/csrc/synth.h), script
    r = rdf(element('O'), element('O'), 10.0);  v = sdf(residue(1:1000), element('O'), 10.0);
i.e. BASELINE configs[1] and configs[2] evaluated together on every frame, as VIAMD evaluates all properties of a script per frame.
`--config 2 | 3 | 4` select BASELINE configs[1] (rdf alone), configs[2] (sdf alone), configs[3] (1M-atom membrane: lipid-tail rdf +
density_z over all atoms) instead; the line then carries that config's own metric name.

A "step" = one pass of the hot path over one batch of `--frames-per-step` frames. Every step reads different frames (no frame is
reused inside the timed region), and one step's input is far larger than the 126 MB L2.

  value : whole-job frames/s with the frames already resident in HBM when the timed region starts (device stopwatch: CUDA events
          on the library's streams, max over ranks).
  e2e   : same metric through the public host API with HOST (pinned) buffers: every step brings its frames host->device — the library
          gathers the atoms the script reads into pinned staging (ingest threads) and copies those — and reads the step's results (RDF
          bins/weights 8 KB + SDF volume 8 MB) back to the host inside the timed region.
  roofline : the dominant kernel, timed ALONE (a second plan with one stream, CUDA events around each launch): `achieved` = algorithmic
          DRAM bytes (SURVEY.md 8(d)) / that time against the measured HBM peak, as the contract asks — and `fp32`, the bound that
          actually holds for the pair kernel: pair tests the kernel executed (device counter, padding lanes included; tests avoided by
          the cull and the symmetric mode are NOT counted) x 9 FP32 lane-operations / time, against SMs x 128 lanes x clock.
  N > 1 : frames are sharded contiguously per rank (weak scaling: every rank processes frames_per_step frames per step); one NCCL
          all-reduce of the RDF bins and SDF voxel grid at the end, inside the timed region; per-rank and all-reduce times in the line.

`--impl reference` times the reference's own CPU md_script_eval_frame_range (oracle/_ref/ref_harness_fast: the unmodified mdlib
sources compiled with their shipped -O3 -ffast-math flags) on all host cores for the same script/workload: ONE process, frames already in
memory, untimed warm-up passes inside it, every step a bounded sample of 8 frames per thread.

`--dump-outputs DIR` writes, after the timed steps, the values array of every result property of the config as DIR/<name>.npy (float32):
what a caller of the timed path receives after its last step (rdf: 1024 bin values + 1024 weights; sdf: the 128^3 volume). The frames are
generated from fixed seeds, so runs with the same arguments see the same inputs and two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the tree may be read-only: nothing is written there, byte-code caches included

UNIT = "frames/s"
WATER_N, WATER_SEED = 32, 1234
MEMB = (38, 100, 48, 4321)   # nl, nw_xy, nwz, seed -> 994 656 atoms
CONFIGS = {
    "bench": dict(metric="frames/sec RDF+SDF eval, 100k-atom synthetic traj", system="water",
                  script="r = rdf(element('O'), element('O'), 10.0); v = sdf(residue(1:1000), element('O'), 10.0);",
                  what="BASELINE configs[1]+[2] on one trajectory", fps=4736, results=("r", "v")),
    "2": dict(metric="frames/sec rdf(O,O,10) eval, 100k-atom synthetic traj", system="water",
              script="r = rdf(element('O'), element('O'), 10.0);", what="BASELINE configs[1]", fps=4736, results=("r",)),
    "3": dict(metric="frames/sec sdf(1000 structures, O, 10) eval, 100k-atom synthetic traj", system="water",
              script="v = sdf(residue(1:1000), element('O'), 10.0);", what="BASELINE configs[2]", fps=4736, results=("v",)),
    "4": dict(metric="frames/sec lipid-tail rdf + density_z eval, 1M-atom synthetic membrane", system="membrane",
              script="rt = rdf(name('C2*'), name('C2*'), 12.0); dz = density_z(all);", what="BASELINE configs[3]", fps=288, results=("rt", "dz")),
}


def workload_string(cfg):
    if cfg["system"] == "water":
        return (f"{cfg['what']}: synthetic water n={WATER_N} ({3 * WATER_N ** 3} atoms, {WATER_N ** 3} O, L={WATER_N * 3.104:.3f} A), script: {cfg['script']}")
    return f"{cfg['what']}: synthetic coarse-grained membrane (994656 atoms, 12-bead lipids + solvent beads, cell 304 x 304 x 111.6 A), script: {cfg['script']}"


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe). In-process NVML (pynvml) when available:
    spawning nvidia-smi several times a second on an 8-GPU box perturbs the driver and slowed the sampled rank; nvidia-smi is the fallback."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.rows, self.stop_ev, self.th = gpu_index, [], threading.Event(), None
        self.nv = None; self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            phys = self.idx
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                try: phys = int(vis.split(",")[self.idx])
                except Exception: phys = self.idx
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys); self.nv = pynvml
        except Exception:
            self.nv = None

    def _sample_nvml(self):
        nv = self.nv
        sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM); mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        try: r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception: r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        def bit(name_new, name_old):
            m = getattr(nv, name_new, None) or getattr(nv, name_old, 0)
            return "Active" if (r & m) else "Not Active"
        self.rows.append([str(self.idx), str(sm), str(mx), "0",
                          bit("nvmlClocksEventReasonHwSlowdown", "nvmlClocksThrottleReasonHwSlowdown"),
                          bit("nvmlClocksEventReasonHwThermalSlowdown", "nvmlClocksThrottleReasonHwThermalSlowdown"),
                          bit("nvmlClocksEventReasonSwThermalSlowdown", "nvmlClocksThrottleReasonSwThermalSlowdown"),
                          bit("nvmlClocksEventReasonSwPowerCap", "nvmlClocksThrottleReasonSwPowerCap")])

    def _run(self):
        while not self.stop_ev.is_set():
            try:
                if self.nv is not None: self._sample_nvml()
                else:
                    out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.idx)],
                                         capture_output=True, text=True, timeout=5).stdout.strip()
                    if out:
                        self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop_ev.wait(0.05 if self.nv is not None else 0.5)

    def start(self):
        self.th = threading.Thread(target=self._run, daemon=True); self.th.start()

    def stop(self):
        self.stop_ev.set()
        if self.th: self.th.join(3)
        sm = sorted(int(float(r[1])) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit())
        mx = [int(float(r[2])) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(self.rows),
                "source": "nvml" if self.nv is not None else "nvidia-smi"}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)", float(d.get("sm_max_mhz", 1965.0))
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)", 1965.0


def measured_traffic(kernel: str, frames_per_launch: float):
    """dram__bytes_read+write of `kernel` per launch, from the committed ncu --set full capture of this round (profiles/r2_traffic.json,
    scaled to this run's frames per launch); None when no capture is recorded."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))[kernel]
        return (t["dram_bytes_read"] + t["dram_bytes_write"]) * (frames_per_launch / t["frames_per_launch"])
    except Exception:
        return None


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def harness_path(kind="fast"):
    return os.path.join(ROOT, "oracle", "_ref", f"ref_harness_{kind}")


def ensure_gro(cfg, tmpdir):
    tool = os.path.join(ROOT, "oracle", "build", "synth_tool")
    if not os.path.exists(tool):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "oracle"])
    if cfg["system"] == "water":
        gro = os.path.join(tmpdir, f"water{WATER_N}_{WATER_SEED}.gro")
        if not os.path.exists(gro): subprocess.check_call([tool, "water-gro", str(WATER_N), str(WATER_SEED), gro])
        return gro, f"synthwater:{WATER_N}:{WATER_SEED}:%d"
    gro = os.path.join(tmpdir, "membrane_%d_%d_%d_%d.gro" % MEMB)
    if not os.path.exists(gro): subprocess.check_call([tool, "membrane-gro", *map(str, MEMB), gro])
    return gro, "synthmembrane:%d:%d:%d:%d:" % MEMB + "%d"


def run_reference(cfg, frames: int, threads: int, repeat: int, warmup: int):
    """The reference's CPU md_script_eval_frame_range on `frames` in-memory frames with `threads` threads: ONE process, `warmup` untimed
    and `repeat` timed full passes inside it (oracle/ref_harness.c mode `time`). Returns the harness's JSON dict or None."""
    h = harness_path("fast")
    if not os.path.exists(h):
        return None
    gro, spec = ensure_gro(cfg, os.environ.get("TMPDIR", "/tmp"))
    out = subprocess.run([h, "time", "--sys", gro, "--traj", spec % frames, "--script", cfg["script"], "--frames", f"0:{frames}", "--threads", str(threads),
                          "--repeat", str(repeat), "--warmup", str(warmup)], capture_output=True, text=True)
    for line in out.stdout.splitlines():
        if line.startswith("{"):
            return json.loads(line)
    sys.stderr.write(out.stderr[-2000:])
    return None


def oracle_port_sample(frames: int):
    """CPU baseline when the reference harness is not built: the plain-C oracle port on one core (kind 'port'), water workload."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import numpy as np
    import oracle_lib as O
    import viamd_b200 as vb
    base, L = vb.synth_water_base(WATER_N, WATER_SEED)
    fr = vb.synth_water_frames_host(WATER_N, WATER_SEED, base, 0, frames)
    s = vb.water_system(WATER_N); o = np.arange(0, s.num_atoms, 3, dtype=np.int32)
    structs = np.arange(3000, dtype=np.int32).reshape(1000, 3); oc = O.UnitCell.ortho(L, L, L)
    vol = np.zeros(128 ** 3, np.float32)
    t0 = time.perf_counter()
    for f in range(frames):
        O.rdf_frame(*fr[f], o, o, oc, 0.0, 10.0)
        O.sdf_frame(*fr[f], fr[0], s.mass, structs, o, s.conn_offset, s.conn_idx, oc, 10.0, vol=vol)
    dt = time.perf_counter() - t0
    return {"frames": frames, "threads": 1, "best_s": dt, "frames_per_s": frames / dt}


CPU_NOTE = ("unmodified mdlib sources, flags as shipped (-O3 -mavx2 -mfma -ffast-math; parity is pinned against the strict-IEEE build of the same sources), "
            "one process, frames generated into memory before the clock starts, untimed warm-up passes inside the process")


def cpu_sample_frames(cfg, threads):
    return max(8 * threads, 16) if cfg["system"] == "water" else max(threads, 8)   # a membrane frame is 12 MB and ~10x the work


def impl_reference(args, cfg):
    rank, local_rank, world = dist_env()
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    sample = cpu_sample_frames(cfg, threads)
    line = {"impl": "reference", "metric": cfg["metric"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(cfg), "frames_per_step": sample, "threads": threads, "host_cpu": cpu_model()}}
    r = run_reference(cfg, sample, threads, max(1, args.steps), max(1, args.warmup))
    if r:
        t_total = sum(r["times_s"]); frames_total = r["frames"] * len(r["times_s"])
        kind, note = "reference", CPU_NOTE
    else:
        r = oracle_port_sample(4); t_total, frames_total = r["best_s"], r["frames"]
        kind, threads, sample, note = "port", 1, 4, "oracle/md_oracle.c scalar port (reference harness not built)"
    v = frames_total / t_total
    line.update({"value": v, "ms_per_step": 1e3 * t_total / max(1, args.steps),
                 "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": kind, "host_cpu": cpu_model(),
                                  "sample": f"{sample} frames ({sample // max(threads, 1)} per thread) per step x {args.steps} steps of the same workload; {note}"},
                 "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    emit(line)
    return 0


_REAL_STDOUT = None


def emit(line):
    """the ONE JSON line goes to the process's real stdout; everything else written to fd 1 meanwhile (NCCL's version banner, library
    chatter) was redirected to stderr in main()"""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None: sys.stdout.write(data.decode()); sys.stdout.flush()
    else: os.write(_REAL_STDOUT, data)


class Workload:
    """system + device-resident synthetic frames of one config"""

    def __init__(self, vb, cfg, dev, rank, frames_local):
        import numpy as np
        self.vb, self.cfg, self.dev = vb, cfg, dev
        if cfg["system"] == "water":
            self.base, L = vb.synth_water_base(WATER_N, WATER_SEED); self.na = self.base.shape[1]
            self.sysm = vb.water_system(WATER_N); self.cell = vb.UnitCell.from_basis(L, L, L); self.mol = None
            self.f0 = vb.synth_water_frames_host(WATER_N, WATER_SEED, self.base, 0, 1)
        else:
            self.base, whole, self.mol, L3 = vb.synth_membrane_base(*MEMB); self.na = self.base.shape[1]
            self.sysm = vb.membrane_system(*MEMB[:3]); self.cell = vb.UnitCell.from_basis(*L3)
            self.f0 = vb.synth_membrane_frames_host(*MEMB, self.base, self.mol, 0, 1)
        self.props = vb.compile_script(cfg["script"], self.sysm)
        self.fstride = 3 * self.na
        self.d_base = vb.device_alloc(dev, self.base.nbytes); vb.memcpy_h2d(dev, self.d_base, self.base.ctypes.data, self.base.nbytes)
        self.d_mol = None
        if self.mol is not None:
            self.d_mol = vb.device_alloc(dev, self.mol.nbytes); vb.memcpy_h2d(dev, self.d_mol, self.mol.ctypes.data, self.mol.nbytes)
        self.d_frames = vb.device_alloc(dev, frames_local * self.fstride * 4)
        if cfg["system"] == "water":
            vb.synth_water_frames_device(dev, WATER_N, WATER_SEED, self.d_base, rank * frames_local, frames_local, self.d_frames, self.fstride, self.na)
        else:
            vb.synth_membrane_frames_device(dev, *MEMB, self.d_base, self.d_mol, rank * frames_local, frames_local, self.d_frames, self.fstride, self.na)

    def plan(self, num_frames, **kw):
        p = self.vb.Plan(self.sysm, self.props, num_frames, device=self.dev, **kw)
        p.set_initial_frame(*self.f0[0], self.cell)   # frame 0 of the trajectory is the initial configuration on every rank
        return p

    def free(self):
        for p in (self.d_base, self.d_mol, self.d_frames):
            if p: self.vb.device_free(self.dev, p)


def main():
    global _REAL_STDOUT
    sys.stdout.flush(); _REAL_STDOUT = os.dup(1); os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--config", default="bench", choices=list(CONFIGS))
    ap.add_argument("--frames-per-step", type=int, default=0)   # 0 = the config's default (32 x 148 frames for the water box)
    ap.add_argument("--batch-frames", type=int, default=0)
    ap.add_argument("--streams", type=int, default=0)
    ap.add_argument("--rdf-variant", type=int, default=0)
    ap.add_argument("--ingest-mode", type=int, default=0)       # 1 = whole frames cross PCIe (the round-1 behaviour)
    ap.add_argument("--ingest-threads", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-iso", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None)
    # rehearsal switches for the N>1 flow on a ONE-GPU machine (never set by the driver): every rank on cuda:0 and gloo instead of NCCL, which refuses
    # two ranks on one device. Everything else — torchrun environment, sharding, barriers, the exchange step, max over ranks, rank-0 line — is the real flow.
    ap.add_argument("--dist-backend", default="nccl", choices=["nccl", "gloo"])
    ap.add_argument("--one-device", action="store_true")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = CONFIGS[args.config]
    if args.impl == "reference":
        return impl_reference(args, cfg)

    import numpy as np
    import torch
    import viamd_b200 as vb
    from viamd_b200 import dist as vdist

    rank, local_rank, world = dist_env()
    dev = 0 if args.one_device else local_rank
    if world > 1:
        import torch.distributed as tdist
        torch.cuda.set_device(dev)
        if args.dist_backend == "nccl": tdist.init_process_group("nccl", device_id=torch.device("cuda", dev))
        else: tdist.init_process_group("gloo")
    small = f"cuda:{dev}" if args.dist_backend == "nccl" else "cpu"   # where the few scalars exchanged between ranks live (gloo gathers CPU tensors only)
    if vb.device_count() == 0:
        raise SystemExit("bench.py: no CUDA device (the product has no CPU path)")
    # this rank's host side (pinned staging, ingest threads, this thread) next to its GPU: GPU0-3 / GPU4-7 hang off different NUMA nodes
    numa_cpus = vb.bind_host_to_device(dev)

    K, W = args.steps, max(args.warmup, 3)
    FPS = args.frames_per_step or cfg["fps"]
    B = args.batch_frames or (148 if cfg["system"] == "water" else 24)
    total_steps = W + K
    na_est = 3 * WATER_N ** 3 if cfg["system"] == "water" else 994656
    # all (warm-up + timed) steps read distinct device-resident frames; keep that shard under ~60 GB of the 180 GB HBM
    max_fps = int(60e9 // (total_steps * 3 * na_est * 4)) // B * B
    FPS = max(B, min(FPS, max_fps))
    frames_local = total_steps * FPS
    wl = Workload(vb, cfg, dev, rank, frames_local)
    na, fstride, cell = wl.na, wl.fstride, wl.cell
    plan = wl.plan(frames_local, batch_frames=B, num_streams=args.streams, rdf_variant=args.rdf_variant, ingest_mode=args.ingest_mode, ingest_threads=args.ingest_threads)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            tdist.barrier()
        torch.cuda.synchronize(dev)

    def step_device(i):
        plan.eval_device_frames(wl.d_frames + i * FPS * fstride * 4, fstride, na, cell, i * FPS, FPS)

    # ---- warm-up (untimed)
    for i in range(W):
        step_device(i)
    plan.sync()
    vb.launch_count(reset=True)
    sampler = ClockSampler(dev); sampler.start()
    barrier()
    plan.timer_begin()
    t_wall0 = time.perf_counter()
    for i in range(W, W + K):
        step_device(i)
    ms_allreduce = 0.0
    if world > 1:
        plan.sync()
        ta = time.perf_counter()
        vdist.allreduce_plan(plan, total_frames=world * (W + K) * FPS)   # the one exchange step: bins + voxels over NCCL
        ms_allreduce = (time.perf_counter() - ta) * 1e3
    ms_dev = plan.timer_end()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop()
    launches = vb.launch_count()
    ms_rank = ms_dev; per_rank_ms = [ms_dev]; per_rank_ar = [ms_allreduce]
    if world > 1:
        t = torch.tensor([ms_dev, ms_allreduce], dtype=torch.float64, device=small)
        g = [torch.zeros_like(t) for _ in range(world)]; tdist.all_gather(g, t)
        per_rank_ms = [float(x[0]) for x in g]; per_rank_ar = [float(x[1]) for x in g]; ms_dev = max(per_rank_ms)
        t = torch.tensor([float(launches)], dtype=torch.float64, device=small)
        tdist.all_reduce(t, op=tdist.ReduceOp.SUM); launches = int(t.item())
    value = world * K * FPS / (ms_dev * 1e-3)
    checks = {}
    for name in cfg["results"]:
        d = plan.property_data(name)
        checks[name + "_sum_per_frame"] = float(np.float64(d.values[:1024] if d.weights is not None else d.values).sum())
        if args.dump_outputs and rank == 0:
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), d.values.astype(np.float32))

    # ---- end-to-end through the host API: pinned host frames -> (gather of the atoms the script reads) -> H2D -> kernels -> D2H of the step's results
    e2e = None
    if not args.no_e2e:
        plan.clear(); plan.set_initial_frame(*wl.f0[0], cell)
        nbuf = 2
        h_ptrs = [vb.host_alloc_pinned(FPS * fstride * 4) for _ in range(nbuf)]
        for b, hp in enumerate(h_ptrs):   # fill the pinned buffers from the device-generated frames (exactly the frames of the device run)
            vb.memcpy_d2h(dev, hp, wl.d_frames + b * FPS * fstride * 4, FPS * fstride * 4)
        Ke = max(2, min(K, 4))
        atoms_copied, ingest_threads = plan.ingest_info()

        def step_host(i):
            plan.eval_host_ptr(h_ptrs[i % nbuf], fstride, na, cell, i * FPS, FPS)
            s = 0.0
            for name in cfg["results"]:   # sync + D2H of the step's results
                s += float(plan.property_data(name).values[0])
            return s

        for i in range(2):
            step_host(i)
        barrier()
        t0 = time.perf_counter()
        for i in range(2, 2 + Ke):
            step_host(i)
        barrier()
        dt = time.perf_counter() - t0
        per_rank_e2e = [dt]
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device=small)
            g = [torch.zeros_like(t) for _ in range(world)]; tdist.all_gather(g, t); per_rank_e2e = [float(x[0]) for x in g]; dt = max(per_rank_e2e)
        d2h = sum((2 * 1024 * 4) if plan.property_data(n).weights is not None else plan.property_data(n).values.size * 4 for n in cfg["results"])
        e2e = {"value": world * Ke * FPS / dt, "unit": UNIT, "h2d_bytes_per_step": FPS * 3 * atoms_copied * 4, "d2h_bytes_per_step": d2h, "steps": Ke,
               "host_frame_bytes_per_step": FPS * fstride * 4,
               "ingest": {"atoms_copied_per_frame": atoms_copied, "atoms_per_frame": na, "gather_threads": ingest_threads,
                          "note": "the library gathers the atoms the script reads out of the caller's whole frames into pinned staging and copies only those"
                                  if atoms_copied < na else "whole frames are copied"},
               "numa_bound_cpus": numa_cpus, "per_rank_s": per_rank_e2e}
        for hp in h_ptrs:
            vb.host_free_pinned(hp)

    # ---- the kernels alone: a second plan with ONE stream, CUDA events around every launch, device counter of executed pair tests
    iso = {}
    if rank == 0 and not args.no_iso:
        nb_iso = 6
        p1 = wl.plan(frames_local, batch_frames=B, num_streams=1, rdf_variant=args.rdf_variant)
        p1.eval_device_frames(wl.d_frames, fstride, na, cell, 0, 2 * B); p1.sync(); p1.clear(); p1.set_initial_frame(*wl.f0[0], cell)
        p1.enable_kernel_timing(True)
        p1.eval_device_frames(wl.d_frames + 2 * B * fstride * 4, fstride, na, cell, 2 * B, nb_iso * B); p1.sync()
        for k in ("k_rdf_pairs", "k_rdf_cull", "k_sdf", "k_density"):
            t, n = p1.kernel_time_ms(k)
            if n: iso[k] = {"ms_per_launch": t / n, "launches": n, "frames_per_launch": B}
        if "k_rdf_pairs" in iso:
            iso["k_rdf_pairs"]["pair_tests_executed_per_launch"] = p1.kernel_counter(0) / iso["k_rdf_pairs"]["launches"]
            iso["k_rdf_pairs"]["pair_tests_useful_per_launch"] = p1.kernel_counter(1) / iso["k_rdf_pairs"]["launches"]
        p1.close()

    if rank == 0:
        peak, peak_src, sm_mhz_max = measured_peaks()
        sm_count = 148
        roof = {"bound": "hbm", "peak": peak, "unit": "GB/s", "peak_source": peak_src}
        rdf_props = [p for p in wl.props if p.op == vb.OP_RDF]; sdf_props = [p for p in wl.props if p.op == vb.OP_SDF]
        dens_props = [p for p in wl.props if vb.OP_DENSITY_X <= p.op <= vb.OP_DENSITY_Z]
        cand = {}
        if "k_rdf_pairs" in iso: cand["k_rdf_pairs"] = iso["k_rdf_pairs"]["ms_per_launch"] + iso.get("k_rdf_cull", {}).get("ms_per_launch", 0.0)
        if "k_sdf" in iso: cand["k_sdf"] = iso["k_sdf"]["ms_per_launch"]
        if "k_density" in iso: cand["k_density"] = iso["k_density"]["ms_per_launch"]
        if cand:
            dom = max(cand, key=cand.get); ms = cand[dom]
            if dom == "k_rdf_pairs":
                sel = set(rdf_props[0].idx[0].tolist()) | set(rdf_props[0].idx[1].tolist())
                algo = 12 * len(sel); kname = "k_rdf_cull + k_rdf_pairs_v2"
                what = "12 B x |reference U target atoms|: their coordinates read once, bins stay on chip (SURVEY.md 8(d))"
            elif dom == "k_sdf":
                algo = 12 * (len(sdf_props[0].idx[0]) + len(sdf_props[0].idx[1])); kname = "k_sdf_ref0 + k_sdf_fit + k_sdf_scatter"
                what = "12 B x (atoms of the reference structures + target atoms) (SURVEY.md 8(d)); the 8 MB voxel grid stays in L2"
            else:
                algo = 4 * len(dens_props[0].idx[0]); kname = "k_density"
                what = "4 B x atoms: density_z reads one coordinate per atom (SURVEY.md 8(d) quotes 12 B/atom for xyz; masses and indices are static and L2-resident)"
            achieved = algo * B / (ms * 1e-3) / 1e9
            roof.update({"kernel": kname, "achieved": achieved, "frac": achieved / peak, "algorithmic_bytes_per_launch": algo * B, "algorithmic_bytes_per_frame": algo,
                         "algorithmic_bytes_definition": what, "ms_per_launch_alone": ms, "frames_per_launch": B,
                         "traffic": measured_traffic(dom, B),
                         "timing": "CUDA events on the launching stream around each launch of a one-stream plan (no other kernel in flight), %d launches" % iso[dom]["launches"],
                         "kernel_share_of_step": ms / (sum(cand.values()) or 1.0)})
            if "k_rdf_pairs" in iso and iso["k_rdf_pairs"].get("pair_tests_executed_per_launch"):
                tests = iso["k_rdf_pairs"]["pair_tests_executed_per_launch"]; t_pair = iso["k_rdf_pairs"]["ms_per_launch"] * 1e-3
                lane_peak = sm_count * 128 * sm_mhz_max * 1e6
                roof["fp32"] = {"kernel": "k_rdf_pairs_v2", "pair_tests_executed_per_launch": tests, "pair_tests_useful_per_launch": iso["k_rdf_pairs"]["pair_tests_useful_per_launch"],
                                "lane_ops_per_test": 9, "ms_per_launch_alone": iso["k_rdf_pairs"]["ms_per_launch"],
                                "achieved_lane_ops_per_s": tests * 9 / t_pair, "peak_lane_ops_per_s": lane_peak, "frac": tests * 9 / t_pair / lane_peak,
                                "pair_tests_per_s": tests / t_pair,
                                "definition": "tests the kernel executed (device counter; the cull's and the symmetric mode's avoided tests are not counted, padding lanes are) x 9 FP32 "
                                              "operations (3 sub, 4 mul, 2 fma, each one lane-cycle; packed FFMA2-class instructions occupy the pipe two cycles) / the kernel's own time; "
                                              "peak = %d SMs x 128 FP32 lanes x %.0f MHz" % (sm_count, sm_mhz_max),
                                "cull_ms_per_launch_alone": iso.get("k_rdf_cull", {}).get("ms_per_launch")}
            roof["kernels_alone_ms_per_launch"] = {k: v["ms_per_launch"] for k, v in iso.items()}
        line = {
            "metric": cfg["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(cfg),
                       "frames_per_step": FPS, "batch_frames": B, "parallelism": f"frame-sharded x{world}",
                       "l2_policy": "every step reads fresh frames; one step's input (%.2f GB) exceeds the 126 MB L2" % (FPS * fstride * 4 / 1e9)},
            "gpu_launches": launches,
            "clocks": clocks,
            "wall_s": t_wall,
            "checks": checks,
            "roofline": roof,
        }
        if args.one_device or args.dist_backend != "nccl":
            line["config"]["rehearsal"] = "NOT a multi-GPU measurement: every rank on cuda:0, ranks exchange through %s" % args.dist_backend
        if world > 1:
            line["per_rank"] = {"device_ms": per_rank_ms, "allreduce_ms": per_rank_ar, "note": "device_ms: CUDA-event time of the timed region on each rank (the value uses the max); allreduce_ms: host time of the one exchange step"}
        if e2e:
            line["e2e"] = e2e
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            sample = cpu_sample_frames(cfg, cores)
            r = run_reference(cfg, sample, cores, 1, 1)
            if r:
                line["cpu_baseline"] = {"value": r["frames"] / r["times_s"][0], "unit": UNIT, "cores": cores, "kind": "reference", "host_cpu": cpu_model(),
                                        "sample": f"{sample} frames ({sample // cores} per thread) of the same workload through md_script_eval_frame_range on {cores} threads; {CPU_NOTE}"}
            else:
                r = oracle_port_sample(4)
                line["cpu_baseline"] = {"value": r["frames_per_s"], "unit": UNIT, "cores": 1, "kind": "port", "host_cpu": cpu_model(), "sample": "4 frames, oracle/md_oracle.c scalar port"}
        emit(line)
    wl.free()
    plan.close()
    if world > 1:
        tdist.barrier()   # rank 0 times the kernels alone after the timed region; the others wait for it here
        tdist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
