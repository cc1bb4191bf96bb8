#!/usr/bin/env python
"""bench.py -- ESKF frames/s and residuals/s of the FAST-LIVO measurement + iterated-ESKF hot
path on B200 (BASELINE.json metric), with the reference-equivalent CPU path timed beside it.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C2] [--impl reference] [--dump-outputs DIR]

A *step* is one frame: one full LIO update (all passes, kNN on the rematch passes) followed by
one full VIO update (ComputeJ: 3 pyramid levels) whose prior is the LIO posterior, on one
synthetic Avia-shaped frame (fast-livo_b200/synth.py).  Pass counts are fixed (early stop
disabled, SURVEY.md §8d) so that the GPU and CPU arms do identical work.

  value : frames/s with all inputs resident in HBM (state reset on the device each step)
  e2e   : frames/s through the C ABI with HOST buffers: per step the scan, image, patch list
          and both states go host->device and the updated state + reports come back
  roofline / cpu_baseline : see DESIGN.md §5.
  other_workloads : BASELINE.json configs[2], configs[3] (C3, C4) measured in the same run (N = 1)
  batched : B independent frames per launch (SURVEY.md §7 H2(iv)): the roofline where it is physically meaningful

N > 1 (torchrun, one rank per GPU): the scan points and patches are block-sharded, map / image /
state replicated, the packed normal equations exchanged every pass (BASELINE.json config 5) --
total work is fixed, so scaling is "strong".  Every N > 1 line carries `parity` (state vs the
unsharded CPU path, rank-to-rank bit equality) and the NCCL-collective number as a secondary key.
"""
from __future__ import annotations

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
import fastlivo_loader  # noqa: E402

METRIC = "eskf_frames_per_sec"
UNIT = "frames/s"

# Algorithmic bytes per unit (SURVEY.md §8d / DESIGN.md §4)
B_LIO_KNN, B_LIO_PLAIN, B_VIO = 132, 33, 405


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock + throttle reasons DURING the run, sampled by a thread through NVML (nvidia_ml_py); falls back to
    an `nvidia-smi -lms` child whose stdout is read line by line (a block-buffered child killed by SIGTERM loses
    its output: that is why round 1 reported 0 samples)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, device):
        self.sm, self.smax, self.reasons, self.power = [], [], set(), []
        self.stop_flag = False
        self.mode = None
        self.t_mark = None
        self.marks = []
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(int(device))
            self.mode = "nvml"
            self.th = threading.Thread(target=self._run_nvml, daemon=True)
            self.th.start()
        except Exception:
            try:
                q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                     "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
                self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20",
                                           "-i", str(device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, bufsize=1)
                self.mode = "nvidia-smi"
                self.th = threading.Thread(target=self._run_smi, daemon=True)
                self.th.start()
            except OSError:
                self.mode = None

    def _run_nvml(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.smax.append(float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
                try:
                    self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                except Exception:
                    pass
            except Exception:
                pass
            time.sleep(0.002)

    def _run_smi(self):
        for line in self.p.stdout:
            c = [x.strip() for x in line.split(",")]
            if len(c) < 7:
                continue
            try:
                self.sm.append(float(c[0]))
                self.smax.append(float(c[1]))
                self.power.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[3:7]):
                if v.lower().startswith("active"):
                    self.reasons.add(name)
            if self.stop_flag:
                break

    def mark(self):
        """Start of the timed region: the median is taken over the samples from here on (if any)."""
        self.t_mark = len(self.sm)

    def stop(self):
        if self.mode is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["clock sampling unavailable"]}
        self.stop_flag = True
        if self.mode == "nvidia-smi":
            try:
                self.p.terminate()
                self.p.wait(timeout=5)
            except Exception:
                pass
        self.th.join(timeout=5)
        sm = self.sm[self.t_mark:] if (self.t_mark is not None and len(self.sm) > self.t_mark + 2) else self.sm
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(self.smax) if self.smax else None,
                "samples": len(sm), "samples_total": len(self.sm), "power_w_max": max(self.power) if self.power else None,
                "reasons": sorted(self.reasons), "source": self.mode}


def pass_counts(cfg):
    """Fixed pass schedule with early stop disabled (SURVEY.md §8d / Appendix A): K LIO passes with
    kNN on the first and the last, K VIO passes on each of 3 levels."""
    k = cfg.lio_passes
    knn = min(k, 2) if k >= 2 else 1
    return dict(lio_T=k - 1, lio_knn=knn, lio_plain=k - knn, vio_T=cfg.vio_passes, vio_passes=3 * cfg.vio_passes)


def cpu_tree(po, frame):
    """The reference's own ikd-Tree over the frame's map (oracle/_ref), or None where it was not built.  ONE per process:
    every KD_TREE starts a background thread that is never joined, and processes holding several have crashed."""
    return po.IkdTreeRef(frame["map_xyz"]) if po.ref_lib() is not None else None


def cpu_frame_runner(po, frame, nthreads, tree="build"):
    """The CPU arm: oracle restatement + the reference's own ikd-Tree (oracle/_ref) when present."""
    cfg = frame["cfg"]
    pc = pass_counts(cfg)
    if tree == "build":
        tree = cpu_tree(po, frame)
    lio = po.Lio(frame["map_xyz"], frame["scan_body"], tree)
    vio = po.Vio(frame["image"], frame["patch_pos"], frame["patch_ref"], frame["patch_level"], frame["cam"]) if cfg.n_patch else None
    lprm = po.lio_params(frame, pc["lio_T"], nthreads=nthreads, early_stop=False)
    vprm = po.vio_params(frame, pc["vio_T"], early_stop=False, force_all_passes=True) if vio else None

    def run(reports=None):
        x = po.state_from_frame(frame)
        lrep = lio.update(lprm, x, x.copy())
        vrep = None
        rows = lrep.rows_total
        if vio:
            vrep = vio.update(vprm, x, x.copy())
            rows += vrep.rows_total
        if reports is not None:
            reports[:] = [lrep, vrep]
        return x, rows
    kind = "reference kNN (ikd_Tree.cpp via oracle/_ref) + line-cited C++ port of the rest" if tree else "port (brute-force kNN)"
    return run, kind


def dump_outputs(out_dir, x, lrep, vrep):
    """--dump-outputs: what the last timed step returned to its caller, one float64 .npy per array: the state (rotation,
    position, velocity, gyro / accelerometer biases, gravity), its 18x18 covariance and the two update reports."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"state": x.vector(), "cov": x.P,
              "lio_report": [lrep.passes, lrep.knn_passes, lrep.n_eff_last, lrep.res_mean_last, lrep.rows_total, lrep.converged_last]}
    if vrep is not None:
        arrays["vio_report"] = [*vrep.passes, *vrep.last_error, vrep.rows_total, vrep.skipped_last, vrep.cov_updated]
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, np.float64))


def cpu_one_frame_child(name):
    """`bench.py --cpu-one-frame NAME`: one frame of workload NAME on the CPU path, result as one JSON line.  A process of its
    own because the reference's KD_TREE (oracle/_ref: a background rebuild thread per tree, never joined) has crashed when
    a third tree was built in one process; the parent only loses this secondary figure if that happens."""
    synth = fastlivo_loader.load().synth
    po = fastlivo_loader.oracle()
    cfg = synth.CONFIGS[name]
    frame = synth.make_frame(cfg)
    cores = os.cpu_count() or 1
    run4, kind = cpu_frame_runner(po, frame, min(4, cores))
    t0 = time.perf_counter()
    xo, _ = run4()
    dt = time.perf_counter() - t0
    print(json.dumps({"dt": dt, "x": [float(v) for v in xo.vector()], "kind": kind, "cores": min(4, cores)}), flush=True)
    os._exit(0)          # do not run the trees' destructors / thread teardown


def cpu_baseline_child_main(name, frames):
    """`bench.py --cpu-baseline-child NAME --cpu-frames K`: the cpu_baseline sample (4 threads and all cores), one JSON line."""
    synth = fastlivo_loader.load().synth
    po = fastlivo_loader.oracle()
    frame = synth.make_frame(synth.CONFIGS[name])
    cores = os.cpu_count() or 1
    tree = cpu_tree(po, frame)
    run4, kind = cpu_frame_runner(po, frame, min(4, cores), tree)
    runall, _ = cpu_frame_runner(po, frame, cores, tree)
    xo, _ = run4()
    runall()
    t0 = time.perf_counter()
    for _ in range(frames):
        run4()
    dt4 = (time.perf_counter() - t0) / frames
    t0 = time.perf_counter()
    for _ in range(frames):
        runall()
    dtall = (time.perf_counter() - t0) / frames
    print(json.dumps({"dt4": dt4, "dtall": dtall, "x": [float(v) for v in xo.vector()], "kind": kind}), flush=True)
    os._exit(0)


def cpu_baseline_child(name, frames, timeout=600):
    import subprocess
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-baseline-child", name, "--cpu-frames", str(frames)],
                           capture_output=True, text=True, timeout=timeout)
        lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
        if r.returncode != 0 or not lines:
            return {"error": f"CPU-path child exited with {r.returncode}"}
        return json.loads(lines[-1])
    except Exception as e:
        return {"error": repr(e)}


def cpu_one_frame(name, timeout=300):
    import subprocess
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-one-frame", name], capture_output=True, text=True, timeout=timeout)
        lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
        if r.returncode != 0 or not lines:
            return {"error": f"CPU-path child exited with {r.returncode}"}
        return json.loads(lines[-1])
    except Exception as e:
        return {"error": repr(e)}


def workload_config(cfg, gpus):
    """Identical in both arms (GPU and --impl reference): names the workload only."""
    pc = pass_counts(cfg)
    return {"workload": f"{cfg.name}: {cfg.n_scan} scan pts vs {cfg.n_map}-pt map, {cfg.img_w}x{cfg.img_h} image, "
                        f"{cfg.n_patch} 8x8 patches; {cfg.lio_passes} LIO passes ({pc['lio_knn']} with kNN) + "
                        f"3x{cfg.vio_passes} VIO passes per frame, early stop disabled",
            "parallelism": "single GPU" if gpus == 1 else f"scan/patch block-sharded over {gpus} GPUs, normal equations exchanged every pass",
            "seed": cfg.seed}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    flb = fastlivo_loader.load()
    po = fastlivo_loader.oracle()
    cfg = flb.synth.CONFIGS[args.workload]
    frame = flb.synth.make_frame(cfg)
    cores = os.cpu_count() or 1
    # the reference compiles its OpenMP team size in (MP_PROC_NUM = 4, CMakeLists.txt:19-37); more threads
    # can be SLOWER (per-query heap allocation inside ikd-Tree), so pick the fastest team size <= cores from the
    # median of 3 timed frames per setting (after one untimed frame each).
    trials = {}
    runners = {}
    tree = cpu_tree(po, frame)            # one tree for every team size (queries only)
    for nt in sorted({t for t in (4, 8, 16, 32, cores) if t <= cores}):
        r, kind = cpu_frame_runner(po, frame, nt, tree)
        r()
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            r()
            ts.append(time.perf_counter() - t0)
        trials[nt] = float(np.median(ts))
        runners[nt] = r
    nthreads = min(trials, key=trials.get)
    run = runners[nthreads]
    for _ in range(args.warmup):
        run()
    t0 = time.perf_counter()
    rows = 0
    reports = []
    for _ in range(args.steps):
        x, r = run(reports)
        rows += r
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, x, *reports)
    fps = args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
        "config": workload_config(cfg, args.gpus),
        "residuals_per_sec": rows / dt,
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": nthreads, "kind": "port", "host_cores": cores,
                         "fps_4_threads": (1.0 / trials[4]) if 4 in trials else None,
                         "team_size_trials_fps": {str(k): 1.0 / v for k, v in trials.items()},
                         "sample": f"{args.steps} frames of {cfg.name}; {kind}; OpenMP over scan points "
                                   f"({nthreads} threads = fastest of 4/8/16/32/all on this host by the median of 3 frames each; "
                                   f"the reference compiles 4 in), VIO serial as in the reference"},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def shard(n, rank, world):
    per = (n + world - 1) // world
    lo = min(rank * per, n)
    return lo, min(lo + per, n)


class Rig:
    """One workload set up on one handle: uploads, the per-frame enqueue, timing helpers."""

    def __init__(self, flb, torch, cfg, frame, h, dev, stream, rank=0, world=1, dist=None, flush=None):
        self.flb, self.torch, self.cfg, self.frame, self.h = flb, torch, cfg, frame, h
        self.dev, self.stream, self.rank, self.world, self.dist, self.flush = dev, stream, rank, world, dist, flush
        self.pc = pass_counts(cfg)
        s0, s1 = shard(cfg.n_scan, rank, world)
        p0, p1 = shard(cfg.n_patch, rank, world)
        self.scan = frame["scan_body"][s0:s1]
        self.ppos, self.pref, self.plev = frame["patch_pos"][p0:p1], frame["patch_ref"][p0:p1], frame["patch_level"][p0:p1]
        self.has_vio = cfg.n_patch > 0
        self.lprm = flb.capi.lio_params(frame, self.pc["lio_T"], early_stop=False)
        self.vprm = flb.capi.vio_params(frame, self.pc["vio_T"], early_stop=False, force_all_passes=True)
        self.x0 = flb.capi.State18.from_frame(frame)

    def upload(self, with_map=True):
        h = self.h
        if with_map:
            h.map_upload(self.frame["map_xyz"])
        h.scan_upload(self.scan)
        if self.has_vio:
            h.camera_set(self.frame["cam"])
            h.image_upload(self.frame["image"])
            h.patches_upload(self.ppos, self.pref, self.plev)
        h.state_upload(self.x0, self.x0.copy())

    def enqueue_frame(self):
        # x := x_prop := prior ; LIO update ; x_prop := x (zero-motion propagation) ; VIO update
        h = self.h
        h.state_reset_enqueue()
        h.lio_update_enqueue(self.lprm)
        if self.has_vio:
            h.state_set_prior_enqueue()
            h.vio_update_enqueue(self.vprm)

    def barrier(self):
        self.torch.cuda.synchronize(self.dev)
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def time_resident(self, steps):
        """`steps` frames with inputs resident, one CUDA-event pair per frame on the launching stream, L2 flushed
        between frames; returns (total_ms as max over ranks, launches, wall_s)."""
        torch = self.torch
        starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        l0 = self.h.launch_count()
        self.barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            if self.flush is not None:
                self.flush.zero_()
            starts[i].record(self.stream)
            self.enqueue_frame()
            ends[i].record(self.stream)
        self.barrier()
        wall = time.perf_counter() - t0
        total_ms = float(sum(s.elapsed_time(e) for s, e in zip(starts, ends)))
        if self.dist is not None:
            t = torch.tensor([total_ms], device=self.dev, dtype=torch.float64)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            total_ms = float(t.item())
        return total_ms, self.h.launch_count() - l0, wall

    def pass_trace(self):
        """Device-side per-pass trace of the persistent kernels (one extra frame, outside any timed region)."""
        h = self.h
        h.trace_enable(True)
        if self.flush is not None:
            self.flush.zero_()
        self.enqueue_frame()
        self.barrier()
        tl, tv = h.trace_download(0), h.trace_download(1)
        h.trace_enable(False)

        def split(t):
            t = t[:63]
            t = t[:int(np.argmax(t == 0))] if (t == 0).any() else t     # entries 64.. are the fine leader stamps
            t = np.concatenate([[0.0], t])
            return {"pass_us": [round(float(t[i + 1] - t[i]), 2) for i in range(0, len(t) - 1, 2)],
                    "solve_us": [round(float(t[i + 2] - t[i + 1]), 2) for i in range(0, len(t) - 2, 2)]}
        return {"lio": split(tl), "vio": split(tv),
                "note": "per pass: time until every block reached the barrier / leader reduce+solve+publish (globaltimer)"}

    def families(self, prof_steps, persistent, hbm):
        """Per-kernel-family device time (separate profiled run: one event pair per launch) + algorithmic GB/s."""
        h, pc = self.h, self.pc
        h.profile_start()
        for _ in range(prof_steps):
            if self.flush is not None:
                self.flush.zero_()
            self.enqueue_frame()
        fam_ms, fam_n = h.profile_stop()
        self.barrier()
        n_loc, pn_loc = len(self.scan), len(self.ppos)
        if persistent:
            # one cooperative kernel per update: its algorithmic bytes are the sum over its passes
            fam_bytes = [(B_LIO_KNN * pc["lio_knn"] + B_LIO_PLAIN * pc["lio_plain"]) * n_loc, 0, B_VIO * pc["vio_passes"] * pn_loc, 0]
            fam_names = [f"k_lio_update_persistent ({pc['lio_knn']} kNN + {pc['lio_plain']} plain passes + solves)", "-",
                         f"k_vio_update_persistent ({pc['vio_passes']} passes + solves)", "-"]
        else:
            fam_bytes = [B_LIO_KNN * n_loc, B_LIO_PLAIN * n_loc, B_VIO * pn_loc, 0]
            fam_names = ["k_lio_pass(kNN+plane+residual)", "k_lio_pass(cached plane)", "k_vio_pass", "k_*_finalize/begin(solve)"]
        fams = []
        for i in range(4):
            if fam_n[i] == 0:
                continue
            avg_us = 1e3 * fam_ms[i] / fam_n[i]
            gbs = fam_bytes[i] / (avg_us * 1e-6) / 1e9 if fam_bytes[i] else 0.0
            fams.append({"kernel": fam_names[i], "launches_per_frame": float(fam_n[i]) / prof_steps, "avg_us": avg_us,
                         "share_of_frame": float(fam_ms[i] / max(fam_ms.sum(), 1e-12)), "algorithmic_bytes": int(fam_bytes[i]),
                         "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / hbm})
        return fams


def traffic_table():
    """dram__bytes_read+write per launch of the persistent kernels from this round's ncu --set full captures
    (profiles/r02_traffic.json, regenerated by profiles/make_traffic.py whenever a kernel changes)."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            with open(p) as f:
                return json.load(f), name
    return {}, None


def roofline_of(fams, hbm, peak_src, workload, note):
    dom = max((f for f in fams if f["algorithmic_bytes"] > 0), key=lambda f: f["share_of_frame"], default=None)
    if dom is None:
        return None
    tj, tname = traffic_table()
    key = dom["kernel"].split(" ")[0]
    traffic = (tj.get(workload) or {}).get(key) if isinstance(tj.get(workload), dict) else (tj.get(key) if workload == "C2" else None)
    return {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["achieved_gbs"], "peak": hbm, "unit": "GB/s",
            "frac": dom["achieved_gbs"] / hbm, "traffic": traffic,
            "traffic_source": f"ncu --set full capture of this code, profiles/{tname}" if traffic else None,
            "peak_source": peak_src, "avg_launch_us": dom["avg_us"], "algorithmic_bytes_per_launch": dom["algorithmic_bytes"],
            "note": note}


def measure_other_workload(flb, torch, name, local, dev, stream, flush, hbm, peak_src, po, steps=10):
    """BASELINE.json configs[2] / configs[3] on one GPU: value, per-kernel roofline, pass trace, parity vs the CPU path."""
    cfg = flb.synth.CONFIGS[name]
    frame = flb.synth.make_frame(cfg)
    h = flb.Handle(device=local, cell_size=cfg.cell_size)
    h.set_stream(stream.cuda_stream)
    rig = Rig(flb, torch, cfg, frame, h, dev, stream, flush=flush)
    rig.upload()
    for _ in range(3):
        rig.enqueue_frame()
    rig.barrier()
    xw, lrep, vrep = h.state_download()
    rows = lrep.rows_total + (vrep.rows_total if rig.has_vio else 0)
    total_ms, launches, _ = rig.time_resident(steps)
    fps = steps / (total_ms * 1e-3)
    trace = rig.pass_trace()
    fams = rig.families(min(steps, 5), True, hbm)
    out = {"config": workload_config(cfg, 1), "value": fps, "unit": UNIT, "steps": steps, "warmup": 3, "ms_per_step": total_ms / steps,
           "rows_per_frame": int(rows), "residuals_per_sec": rows * fps, "gpu_launches": int(launches), "kernels": fams,
           "roofline": roofline_of(fams, hbm, peak_src, name, "see DESIGN.md section 4: which pipe bounds each kernel at this size"),
           "pass_trace": trace}
    if po is not None:
        c = cpu_one_frame(name)              # in a child process (see cpu_one_frame_child)
        if "error" in c:
            out["cpu_baseline"] = c
        else:
            vo = np.array(c["x"])
            out["cpu_baseline"] = {"value": 1.0 / c["dt"], "unit": UNIT, "cores": c["cores"], "kind": "port",
                                   "sample": f"1 frame of {cfg.name} (first call, includes the ikd-Tree build); {c['kind']}"}
            out["parity"] = {"state_rel_err_vs_cpu": float(np.abs(xw.vector() - vo).max() / np.abs(vo).max())}
    h.close()
    return out


def measure_batched(flb, torch, name, B, local, dev, stream, flush, hbm, peak_src, steps=5):
    """SURVEY.md section 7 H2(iv): B independent frames per launch (flb_batch_*): every pass of the iterated update is ONE
    kernel over all B frames, so the pass kernels run at their throughput.  Frames: B different sub-scans of the
    workload's scan (97 %, permuted) with jittered priors, against its map / image / patch list."""
    cfg = flb.synth.CONFIGS[name]
    frame = flb.synth.make_frame(cfg)
    pc = pass_counts(cfg)
    h = flb.Handle(device=local, cell_size=cfg.cell_size)
    h.set_stream(stream.cuda_stream)
    h.load_frame(frame)
    rng = np.random.default_rng(5)
    n_sub = int(0.97 * cfg.n_scan)
    h.batch_begin(B, n_sub)
    for b in range(B):
        idx = rng.permutation(cfg.n_scan)[:n_sub]
        R = frame["R_prop"] @ flb.synth.exp_so3(rng.normal(0, 0.002, 3))
        p = frame["p_prop"] + rng.normal(0, 0.01, 3)
        x = flb.capi.State18.make(R, p, frame["vel"], frame["bg"], frame["ba"], frame["grav"], frame["cov"])
        h.batch_set_frame(b, frame["scan_body"][idx], x, x.copy())
    lprm = flb.capi.lio_params(frame, pc["lio_T"], early_stop=False)
    vprm = flb.capi.vio_params(frame, pc["vio_T"], early_stop=False, force_all_passes=True) if cfg.n_patch else None

    def step():
        h.batch_state_reset_enqueue()
        h.batch_update_enqueue(lprm, vprm)
    for _ in range(3):
        step()
    torch.cuda.synchronize(dev)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    l0 = h.launch_count()
    for a, b_ in ev:
        if flush is not None:
            flush.zero_()
        a.record(stream)
        step()
        b_.record(stream)
    torch.cuda.synchronize(dev)
    launches = h.launch_count() - l0
    ms = float(sum(a.elapsed_time(b_) for a, b_ in ev)) / steps
    _, lrep, vrep = h.batch_state_download(0)
    rows = lrep.rows_total + (vrep.rows_total if vprm is not None else 0)
    h.profile_start()
    for _ in range(2):
        if flush is not None:
            flush.zero_()
        step()
    fam_ms, fam_n = h.profile_stop()
    torch.cuda.synchronize(dev)
    names = ["k_lio_pass_batched (kNN + plane + residual + reduce)", "k_lio_pass_batched (cached plane)", "k_vio_pass_batched",
             "k_*_finalize_batched (B leader blocks)"]
    per_launch_bytes = [B_LIO_KNN * n_sub * B, B_LIO_PLAIN * n_sub * B, B_VIO * cfg.n_patch * B, 0]
    fams = []
    for i in range(4):
        if fam_n[i] == 0:
            continue
        avg_us = 1e3 * fam_ms[i] / fam_n[i]
        gbs = per_launch_bytes[i] / (avg_us * 1e-6) / 1e9 if per_launch_bytes[i] else 0.0
        fams.append({"kernel": names[i], "launches_per_batch": float(fam_n[i]) / 2, "avg_us": avg_us,
                     "share_of_batch": float(fam_ms[i] / max(fam_ms.sum(), 1e-12)), "algorithmic_bytes_per_launch": int(per_launch_bytes[i]),
                     "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / hbm})
    h.close()
    return {"workload": f"{B} frames of {cfg.name} per launch ({n_sub} scan pts each, shared {cfg.n_map}-pt map, {cfg.n_patch} patches)",
            "frames_per_batch": B, "value": B / (ms * 1e-3), "unit": UNIT, "ms_per_batch": ms, "steps": steps,
            "residuals_per_sec": rows * B / (ms * 1e-3), "gpu_launches": int(launches), "kernels": fams, "peak": hbm, "peak_source": peak_src,
            "note": "kernel-per-pass path with blockIdx.y = frame; every frame bit-identical to the frame run alone (tests/test_gpu_batch.py)"}


def measure_full_frame(flb, torch, name, local, dev, stream, flush, steps=20, raw=None):
    """One frame through EVERY stage that is on the device, host buffers in, state out (SURVEY.md section 8 rows a + f1-f4):
    IMU propagation + undistortion -> LIO update -> map maintenance (Add_Points) -> visible-patch selection + warp ->
    VIO update -> map growth -> new observations.  The patch list never crosses PCIe (it is built on the device)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from imu_util import product_inputs
    cfg = flb.synth.CONFIGS[name]
    seq = flb.synth.make_visual_sequence(cfg, 2, with_map=True)
    f0, f1 = seq["frames"]
    grid = 12 if cfg.img_w <= 640 else 16
    h = flb.Handle(device=local, cell_size=cfg.cell_size)
    h.set_stream(stream.cuda_stream)
    fdict = dict(R_LI=seq["R_LI"], t_LI=seq["t_LI"], Rcl=seq["Rcl"], Pcl=seq["Pcl"], cfg=cfg)
    pc = pass_counts(cfg)
    lprm = flb.capi.lio_params(fdict, pc["lio_T"], early_stop=False)
    vprm = flb.capi.vio_params(fdict, pc["vio_T"], early_stop=False, force_all_passes=True)
    h.map_upload(seq["map_xyz"])
    h.camera_set(seq["cam"])
    h.image_upload(f0["image"])
    h.vmap_reset(seq, grid_size=grid, outlier_threshold=300.0)
    h.vmap_select(f0["Rcw"], f0["Pcw"], f0["pg_down"])
    h.vmap_grow(f0["Rcw"], f0["Pcw"], f0["pg"], 0)          # the visual map now holds frame 0's points
    base = h.vmap_counts()
    fi = flb.synth.make_imu_frame(seed=41, n_points=cfg.n_scan)
    packed = np.concatenate([f1["scan_body"], fi["offset_ms"][:len(f1["scan_body"]), None]], 1).astype(np.float32)
    x0 = flb.capi.State18.make(f1["R_prop"], f1["p_prop"], cov=seq["cov"], grav=seq["grav"])
    stage = {k: 0.0 for k in ("imu_undistort", "scan+lio_enqueue", "map_add_points", "image+select_enqueue", "vio+grow+observe_enqueue", "state_download")}
    n_sel = 0

    def frame(k, timed):
        nonlocal n_sel
        t = [time.perf_counter()]
        Pg, Cg, xg = product_inputs(flb, fi)
        h.state_upload(x0, x0.copy())
        h.imu_undistort(Pg, Cg, fi["v_imu"], fi["pcl_beg_time"], fi["pcl_end_time"], packed, offset_index=3)
        t.append(time.perf_counter())
        h.state_upload(x0, x0.copy())                       # the synthetic IMU stream is not this trajectory's: restore the prior
        h.scan_upload(f1["scan_body"])
        h.lio_update_enqueue(lprm)
        t.append(time.perf_counter())
        h.map_add_points(f1["pg"], cfg.pitch)
        t.append(time.perf_counter())
        h.image_upload(f1["image"])
        h.vmap_select(None, None, f1["pg_down"], blocking=False)
        t.append(time.perf_counter())
        h.vmap_grow(None, None, f1["pg"], k + 1)
        h.state_set_prior_enqueue()
        h.vio_update_enqueue(vprm)
        h.vmap_add_observations(None, None, k + 1)
        t.append(time.perf_counter())
        x, lrep, vrep = h.state_download()
        t.append(time.perf_counter())
        if timed:
            for key, a, b in zip(stage, t[:-1], t[1:]):
                stage[key] += b - a
            if raw is not None:
                raw.append([round(1e3 * (b - a), 3) for a, b in zip(t[:-1], t[1:])])
        return x, lrep, vrep
    for k in range(3):
        x, lrep, vrep = frame(k, False)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for k in range(steps):
        if flush is not None:
            flush.zero_()
        x, lrep, vrep = frame(3 + k, True)
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    if flush is not None:
        torch.cuda.synchronize(dev)
        tf = time.perf_counter()
        for _ in range(steps):
            flush.zero_()
        torch.cuda.synchronize(dev)
        dt -= time.perf_counter() - tf
    c = h.vmap_counts()
    h.close()
    h2d = packed.nbytes + len(fi["v_imu"]) * 56 + f1["scan_body"].nbytes + f1["pg"].nbytes * 2 + f1["image"].size + f1["pg_down"].nbytes + 3 * 2 * 2736
    return {"workload": f"{cfg.name}-shaped 2-frame sequence: {cfg.n_scan} scan pts, {cfg.n_map}-pt map, {cfg.img_w}x{cfg.img_h} image, "
                        f"{grid} px grid ({(cfg.img_w // grid) * (cfg.img_h // grid)} cells), {c['selected']} patches selected on the device",
            "value": steps / dt, "unit": UNIT, "ms_per_frame": 1e3 * dt / steps, "steps": steps,
            "host_ms_per_stage": {k: 1e3 * v / steps for k, v in stage.items()},
            "h2d_bytes_per_frame": int(h2d), "d2h_bytes_per_frame": int(len(packed) * 16 + 2736 + 128),
            "patches": int(c["selected"]), "vio_rows_per_frame": int(vrep.rows_total), "lio_rows_per_frame": int(lrep.rows_total),
            "visual_map": {"points_before": base["points"], "points_after": c["points"], "features_after": c["features"], "keyframe_images": c["images"]},
            "note": "stages: flb_imu_undistort (blocking: the undistorted points go back to the caller's voxel filter), flb_scan_upload + "
                    "flb_lio_update_enqueue, flb_map_add_points (incremental merge; one small sync), flb_image_upload + flb_vmap_select "
                    "(enqueue-only, pose from the device state), flb_vmap_grow + flb_vio_update_enqueue + flb_vmap_add_observations, "
                    "flb_state_download; L2 flushed between frames"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 1000; 30 with --impl reference, whose CPU "
                                                                "frames take 0.1-1 s each)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--workload", default="C2", choices=["C1", "C2", "C3", "C4", "T0", "T1"])
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-flush", action="store_true", help="do not flush L2 between timed steps")
    ap.add_argument("--cpu-frames", type=int, default=8, help="frames in the bounded cpu_baseline sample")
    ap.add_argument("--collective", default="p2p", choices=["p2p", "nccl"],
                    help="N > 1: fused NVLink exchange inside the persistent kernels (default) or NCCL between per-pass kernels")
    ap.add_argument("--quick", action="store_true", help="profiling aid: skip the e2e / profile / cpu_baseline legs")
    ap.add_argument("--no-others", action="store_true", help="skip the other_workloads (C3, C4) and batched legs")
    ap.add_argument("--cell-size", type=float, default=0.0, help="experiment: kNN grid cell size (default 2 x the map pitch)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the state, covariance and reports of the last timed step to DIR/<name>.npy (float64), so "
                         "that two builds can be compared output for output (the inputs are seeded)")
    ap.add_argument("--cpu-one-frame", default=None, help=argparse.SUPPRESS)      # child process of measure_other_workload
    ap.add_argument("--cpu-baseline-child", default=None, help=argparse.SUPPRESS)  # child process of the cpu_baseline leg
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 30 if args.impl == "reference" else 1000
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)

    if args.cpu_one_frame:
        return cpu_one_frame_child(args.cpu_one_frame)
    if args.cpu_baseline_child:
        return cpu_baseline_child_main(args.cpu_baseline_child, args.cpu_frames)

    import torch
    flb = fastlivo_loader.load()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    cfg = flb.synth.CONFIGS[args.workload]
    frame = flb.synth.make_frame(cfg)
    pc = pass_counts(cfg)
    h = flb.Handle(device=local, cell_size=args.cell_size if args.cell_size > 0 else cfg.cell_size)
    # a dedicated (non-default) torch stream: the library's kernels, the L2 flush and the timing events
    # must all be on the SAME stream, and flb_set_stream(NULL) would mean "the handle's own stream"
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    h.set_stream(stream.cuda_stream)
    if world > 1 and args.collective == "nccl":
        uid = [flb.Handle.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        h.comm_init(uid[0], rank, world)
    elif world > 1:
        handles = [None] * world
        dist.all_gather_object(handles, h.p2p_export())
        h.p2p_attach(rank, world, handles)
    flush = None if args.no_flush else torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    rig = Rig(flb, torch, cfg, frame, h, dev, stream, rank, world, dist, flush)
    rig.upload()
    scan, ppos, pref, plev, has_vio, x0, lprm, vprm = rig.scan, rig.ppos, rig.pref, rig.plev, rig.has_vio, rig.x0, rig.lprm, rig.vprm
    barrier = rig.barrier

    # ---- warm-up (the clock sampler starts here: the timed region may be shorter than one sampling period)
    sampler = ClockSampler(local) if rank == 0 else None
    for _ in range(args.warmup):
        rig.enqueue_frame()
    barrier()
    xw, lrep, vrep = h.state_download()
    rows_per_frame = lrep.rows_total + (vrep.rows_total if has_vio else 0)   # N > 1: already global (reduced n_eff / n_meas)

    # ---- timed region: value (inputs resident)
    if sampler:
        sampler.mark()
    total_ms, launches, t_wall = rig.time_resident(args.steps)
    clocks = sampler.stop() if sampler else None
    fps = args.steps / (total_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        xd, ld, vd = h.state_download()          # every rank holds the same state (bit-identical, see parity)
        dump_outputs(args.dump_outputs, xd, ld, vd if has_vio else None)

    trace = rig.pass_trace() if world == 1 else None
    if args.quick:
        if rank == 0:
            print(json.dumps({"metric": METRIC, "value": fps, "unit": UNIT, "ms_per_step": total_ms / args.steps,
                              "gpu_launches": int(launches), "quick": True, "trace": trace}), flush=True)
        h.close()
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- N > 1: parity of the sharded result (driver-visible): every rank's state bit-identical, and equal to the
    # unsharded CPU path within the bar
    parity = None
    if world > 1:
        vecs = [None] * world
        dist.all_gather_object(vecs, (xw.vector().tolist(), list(xw.cov[:])))
        if rank == 0:
            po = fastlivo_loader.oracle()
            run4, kind = cpu_frame_runner(po, frame, min(4, os.cpu_count() or 1))
            xo, _ = run4()
            vo = xo.vector()
            v0 = np.array(vecs[0][0])
            identical = all(vecs[r][0] == vecs[0][0] and vecs[r][1] == vecs[0][1] for r in range(world))
            parity = {"state_rel_err_vs_cpu": float(np.abs(v0 - vo).max() / np.abs(vo).max()),
                      "cov_rel_err_vs_cpu": float(np.abs(np.array(vecs[0][1]) - np.array(xo.cov[:])).max() / np.abs(np.array(xo.cov[:])).max()),
                      "ranks_bit_identical": bool(identical), "ranks": world,
                      "cpu_path": f"unsharded; {kind}", "bar": 1e-5}

    # ---- e2e: host buffers through the C ABI, H2D + D2H inside the timed region
    e2e_steps = max(min(args.steps, 50), 3)
    img = frame["image"]
    # e2e_pinned: the same calls with the caller's image / patch buffers page-locked (flb_host_alloc):
    # the library then skips its staging copy
    pin_img, pin_pos, pin_ref, pin_lev = (h.pinned_like(a) for a in (img, ppos, pref.reshape(len(ppos), 192), plev)) if has_vio else (None,) * 4

    def e2e_frame(pinned=False, blocking=False, slot=None):
        # One frame through the C ABI with HOST buffers; the map stays resident.
        #   default : the device-resident loop of the public header -- uploads and both updates are enqueued
        #             (the library packs host inputs into pinned staging and returns), the image / patch list
        #             are staged while the LIO update runs, ONE blocking call (flb_state_download) ends the frame.
        #   blocking: the reference's call shape -- flb_lio_update / flb_vio_update each upload the state, run,
        #             download and synchronise.
        h.scan_upload(scan)
        if blocking:
            if has_vio:
                h.image_upload(pin_img if pinned else img)
                if pinned:
                    h.patches_upload(pin_pos, pin_ref, pin_lev)
                else:
                    h.patches_upload(ppos, pref, plev)
            x = x0.copy()
            h.lio_update(lprm, x, x0)
            if has_vio:
                xp = x.copy()
                h.vio_update(vprm, x, xp)
            return x
        h.state_upload(x0, x0)
        h.lio_update_enqueue(lprm)
        if has_vio:
            h.image_upload(pin_img if pinned else img)
            if pinned:
                h.patches_upload(pin_pos, pin_ref, pin_lev)
            else:
                h.patches_upload(ppos, pref, plev)
            h.state_set_prior_enqueue()          # state_propagat of the VIO step = the LIO result, on the device
            h.vio_update_enqueue(vprm)
        if slot is not None:                     # pipelined: the result of THIS frame is collected one frame later
            h.state_download_enqueue(slot)
            return None
        x, _, _ = h.state_download()
        return x
    for _ in range(3):
        xe = e2e_frame()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        if flush is not None:
            flush.zero_()
        xe = e2e_frame()
    barrier()
    e2e_dt = time.perf_counter() - t0
    if flush is not None:   # subtract the flush cost measured separately (it is not part of the step)
        barrier()
        tf = time.perf_counter()
        for _ in range(e2e_steps):
            flush.zero_()
        barrier()
        e2e_dt -= time.perf_counter() - tf
    if dist is not None:
        t = torch.tensor([e2e_dt], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_dt = float(t.item())
    e2e_fps = e2e_steps / e2e_dt
    # pipelined: frame k+1's uploads / sort are enqueued before frame k's result is collected (two result slots)
    e2e_pipe_fps = None
    if world == 1:
        for k in range(4):
            e2e_frame(slot=k & 1)
            if k:
                xq, _, _ = h.state_download_wait((k - 1) & 1)
        xq, _, _ = h.state_download_wait(3 & 1)
        barrier()
        t0 = time.perf_counter()
        for k in range(e2e_steps):
            if flush is not None:
                flush.zero_()
            e2e_frame(slot=k & 1)
            if k:
                xq, _, _ = h.state_download_wait((k - 1) & 1)
        xq, _, _ = h.state_download_wait((e2e_steps - 1) & 1)
        barrier()
        dtp = time.perf_counter() - t0
        if flush is not None:
            barrier()
            tf = time.perf_counter()
            for _ in range(e2e_steps):
                flush.zero_()
            barrier()
            dtp -= time.perf_counter() - tf
        e2e_pipe_fps = e2e_steps / dtp
        assert np.array_equal(np.array(xq.rot[:]), np.array(xe.rot[:])), "pipelined and serial e2e must give the same state"
    # the one-call frame API with page-locked caller buffers, pipelined: the contract's e2e (inputs from PINNED host
    # memory, the call a user makes), and what the line reports as e2e.value at N = 1
    e2e_frame_api_fps = None
    e2e_frame_api_serial_fps = None
    e2e_live_fps = None
    if world == 1 and has_vio:
        pin_scan = h.pinned_like(np.ascontiguousarray(scan, np.float32))
        fi = h.frame_inputs(pin_scan, x0, x0.copy(), pin_img, pin_pos, pin_ref, pin_lev)
        for k in range(4):
            h.frame_enqueue(fi, lprm, vprm, k & 1)
            if k:
                xf, _, _ = h.state_download_wait((k - 1) & 1)
        xf, _, _ = h.state_download_wait(3 & 1)
        barrier()
        t0 = time.perf_counter()
        for k in range(e2e_steps):
            if flush is not None:
                flush.zero_()
            h.frame_enqueue(fi, lprm, vprm, k & 1)
            if k:
                xf, _, _ = h.state_download_wait((k - 1) & 1)
        xf, _, _ = h.state_download_wait((e2e_steps - 1) & 1)
        barrier()
        dtf = time.perf_counter() - t0
        if flush is not None:
            barrier()
            tf = time.perf_counter()
            for _ in range(e2e_steps):
                flush.zero_()
            barrier()
            dtf -= time.perf_counter() - tf
        e2e_frame_api_fps = e2e_steps / dtf
        # the same call, but every frame's result is collected before the next frame is enqueued: the call pattern of a live
        # odometry loop, whose next prior depends on this posterior
        for k in range(3):
            h.frame_enqueue(fi, lprm, vprm, 0)
            xf, _, _ = h.state_download_wait(0)
        barrier()
        t0 = time.perf_counter()
        for k in range(e2e_steps):
            if flush is not None:
                flush.zero_()
            h.frame_enqueue(fi, lprm, vprm, 0)
            xf, _, _ = h.state_download_wait(0)
        barrier()
        dts = time.perf_counter() - t0
        if flush is not None:
            barrier()
            tf = time.perf_counter()
            for _ in range(e2e_steps):
                flush.zero_()
            barrier()
            dts -= time.perf_counter() - tf
        e2e_frame_api_serial_fps = e2e_steps / dts
        # live loop with look-ahead on the SENSOR data only: frame k+1's scan / image / patch list do not depend on frame k's
        # posterior, so they are uploaded (own streams, idle device sets) while frame k runs; the prior of frame k+1 is set
        # only after frame k's posterior has been read back
        def sensor_uploads():
            h.scan_upload(pin_scan)
            h.image_upload(pin_img)
            h.patches_upload(pin_pos, pin_ref, pin_lev)

        def live_frame():
            h.state_upload(x0, x0)              # (a real loop: the IMU-propagated posterior of the previous frame)
            h.lio_update_enqueue(lprm)
            h.state_set_prior_enqueue()
            h.vio_update_enqueue(vprm)
            h.state_download_enqueue(0)
            sensor_uploads()                    # next frame's sensor data, under this frame's updates
            return h.state_download_wait(0)
        sensor_uploads()
        for k in range(3):
            xl, _, _ = live_frame()
        barrier()
        t0 = time.perf_counter()
        for k in range(e2e_steps):
            if flush is not None:
                flush.zero_()
            xl, _, _ = live_frame()
        barrier()
        dtl = time.perf_counter() - t0
        if flush is not None:
            barrier()
            tf = time.perf_counter()
            for _ in range(e2e_steps):
                flush.zero_()
            barrier()
            dtl -= time.perf_counter() - tf
        e2e_live_fps = e2e_steps / dtl
        assert np.array_equal(np.array(xl.rot[:]), np.array(xe.rot[:])), "the live-loop e2e must give the same state"
        assert np.array_equal(np.array(xf.rot[:]), np.array(xe.rot[:])) and np.array_equal(np.array(xf.cov[:]), np.array(xe.cov[:])), \
            "flb_frame_enqueue must give the same state as the separate calls"
    e2e_blocking_fps = None
    if world == 1:
        for _ in range(3):
            xb = e2e_frame(blocking=True)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            xb = e2e_frame(blocking=True)
        barrier()
        e2e_blocking_fps = e2e_steps / (time.perf_counter() - t0)
        assert np.array_equal(np.array(xb.rot[:]), np.array(xe.rot[:])) and np.array_equal(np.array(xb.cov[:]), np.array(xe.cov[:])), \
            "enqueue and blocking call shapes must give the same state"
    e2e_pinned_fps = None
    if has_vio and world == 1:
        for _ in range(3):
            e2e_frame(True)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_frame(True)
        barrier()
        e2e_pinned_fps = e2e_steps / (time.perf_counter() - t0)
    state_b = 2736
    # device-resident loop: scan + x, x_prop (+ image + patch list); one state + two reports come back
    h2d = len(scan) * 12 + 2 * state_b + ((img.size + len(ppos) * (24 + 768 + 4)) if has_vio else 0)
    d2h = state_b + 2 * 64

    # ---- per-kernel-family device time + roofline of the dominant kernel
    hbm, peak_src = peaks()
    persistent = world == 1 or args.collective == "p2p"   # the NCCL path runs kernel-per-pass
    fams = rig.families(max(min(args.steps, 20), 3), persistent, hbm)
    roofline = roofline_of(fams, hbm, peak_src, args.workload,
                           "the whole working set (~8 MB) is L2-resident and every pass is a dependent step: the kernel is "
                           "latency-bound, not bandwidth-bound, at this size (SURVEY.md section 7 H2; DESIGN.md section 4); "
                           "see `batched` and `other_workloads` for the sizes where the bandwidth roofline is meaningful")

    # ---- N > 1, fused exchange: the NCCL-collective number beside it (kernel-per-pass + ncclAllReduce / AllGather)
    nccl_alt = None
    if world > 1 and args.collective == "p2p":
        barrier()
        h.p2p_detach()
        uid = [flb.Handle.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        h.comm_init(uid[0], rank, world)
        if has_vio:
            h.patches_upload(ppos, pref, plev)       # agrees on the all-gather shard size
        h.state_upload(x0, x0.copy())
        for _ in range(3):
            rig.enqueue_frame()
        barrier()
        xn, _, _ = h.state_download()
        n_steps = max(min(args.steps, 50), 3)
        ms_n, _, _ = rig.time_resident(n_steps)
        nccl_alt = {"value": n_steps / (ms_n * 1e-3), "unit": UNIT, "ms_per_step": ms_n / n_steps, "steps": n_steps,
                    "state_rel_diff_vs_fused": float(np.abs(xn.vector() - xw.vector()).max() / np.abs(xw.vector()).max()),
                    "note": "kernel-per-pass path with ncclAllReduce(29 doubles) + ncclAllGather(per-patch errors) between the "
                            "pass and finalize kernels: the baseline collective BASELINE.json names"}

    # ---- N > 1: independent frames, one whole (unsharded) frame stream per GPU, no exchange: the throughput mode next to
    # the sharded single-frame mode above (DESIGN.md section 6: a frame's passes are narrower than one GPU, so sharding
    # cannot shorten them; frames are independent, so replicas scale)
    replicas = None
    if world > 1:
        barrier()
        h2 = flb.Handle(device=local, cell_size=args.cell_size if args.cell_size > 0 else cfg.cell_size)
        h2.set_stream(stream.cuda_stream)
        rig2 = Rig(flb, torch, cfg, frame, h2, dev, stream, 0, 1, dist, flush)     # rank 0 of 1: the whole frame; dist only for the barrier
        rig2.upload()
        for _ in range(3):
            rig2.enqueue_frame()
        barrier()
        n_steps = max(min(args.steps, 200), 3)
        ms_r, _, _ = rig2.time_resident(n_steps)       # max over ranks
        h2.close()
        replicas = {"value": world * n_steps / (ms_r * 1e-3), "unit": UNIT, "per_gpu": n_steps / (ms_r * 1e-3), "steps": n_steps,
                    "scaling": "weak", "note": "every GPU runs its own whole frames (same kernels, no exchange); aggregate = "
                                               "N x the slowest rank's rate"}

    # ---- cpu_baseline (rank 0, N == 1 only): bounded sample on the host cores
    cpu = None
    po = None
    if rank == 0 and world == 1:
        po = fastlivo_loader.oracle()
        cores = os.cpu_count() or 1
        # in a child process: the reference's KD_TREE has crashed hosts of several trees (cpu_one_frame_child); a second child
        # is tried before giving up, and the line is printed either way
        c = cpu_baseline_child(args.workload, args.cpu_frames)
        if "error" in c:
            c = cpu_baseline_child(args.workload, args.cpu_frames)
        if "error" in c:
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "unavailable: " + c["error"]}
            parity = {"state_rel_err_vs_cpu": None, "bar": 1e-5, "note": "CPU path unavailable in this run"}
        else:
            dt4, dtall, kind = c["dt4"], c["dtall"], c["kind"]
            best = min(dt4, dtall)
            cpu = {"value": 1.0 / best, "unit": UNIT, "cores": cores if dtall <= dt4 else min(4, cores), "kind": "port",
                   "sample": f"{args.cpu_frames} frames of {cfg.name} per thread setting; {kind}",
                   "fps_4_threads": 1.0 / dt4, "fps_all_cores": 1.0 / dtall, "host_cores": cores}
            ve, vo = xe.vector(), np.array(c["x"])
            parity = {"state_rel_err_vs_cpu": float(np.abs(ve - vo).max() / np.abs(vo).max()),
                      "state_rel_err_resident_vs_cpu": float(np.abs(xw.vector() - vo).max() / np.abs(vo).max()), "bar": 1e-5}

    # ---- map maintenance (SURVEY section 8 row f1), informational: one Add_Points(downsample) of the scan, host buffer
    # in, device map + kNN grid refreshed, vs a full re-upload of the map
    map_maint = None
    if rank == 0 and world == 1:
        Rw, pw = frame["R_true"], frame["p_true"]
        world_pts = ((Rw @ (frame["R_LI"] @ frame["scan_body"].T.astype(np.float64) + frame["t_LI"][:, None])).T + pw).astype(np.float32)
        h.map_add_points(world_pts, cfg.pitch)       # first call allocates the scratch buffers
        h.map_upload(frame["map_xyz"])
        barrier()
        t_adds = []
        m_after = 0
        for _ in range(5):
            t0 = time.perf_counter()
            h.map_add_points(world_pts, cfg.pitch)
            barrier()
            t_adds.append(time.perf_counter() - t0)
            m_after = h.M
            h.map_upload(frame["map_xyz"])
            barrier()
        t0 = time.perf_counter()
        h.map_upload(frame["map_xyz"])
        barrier()
        t_up = time.perf_counter() - t0
        map_maint = {"add_points_ms": 1e3 * float(np.median(t_adds)), "points_added": int(len(world_pts)), "map_size_after": int(m_after),
                     "full_map_upload_ms": 1e3 * t_up, "note": "ikdtree.Add_Points(scan, downsample) on the device vs re-uploading the whole map"}

    # row f3: ImuProcess::UndistortPcl through the C ABI (host buffers in, host buffers out) next to the CPU port
    imu_f3 = None
    if rank == 0 and world == 1:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from imu_util import oracle_inputs, product_inputs
        fi = flb.synth.make_imu_frame(seed=41, n_points=cfg.n_scan if hasattr(cfg, "n_scan") else 24000)
        Pg, Cg, xg = product_inputs(flb, fi)
        packed = np.concatenate([fi["pts"], fi["offset_ms"][:, None]], 1).astype(np.float32)
        reps = 20
        t_gpu = []
        for it in range(reps + 3):
            Pg, Cg, xg = product_inputs(flb, fi)         # the call updates the carry in place: fresh inputs every time
            h.state_upload(xg, xg.copy())
            barrier()
            t0 = time.perf_counter()
            got, _ = h.imu_undistort(Pg, Cg, fi["v_imu"], fi["pcl_beg_time"], fi["pcl_end_time"], packed, offset_index=3)
            t_gpu.append(time.perf_counter() - t0)
        t_cpu = []
        for it in range(5):
            Po, Co, xo_i = oracle_inputs(po, fi)
            t0 = time.perf_counter()
            ref, _ = po.imu_undistort(Po, Co, fi["v_imu"], fi["pcl_beg_time"], fi["pcl_end_time"], xo_i, fi["pts"], fi["offset_ms"])
            t_cpu.append(time.perf_counter() - t0)
        imu_f3 = {"abi_call_ms": 1e3 * float(np.median(t_gpu[3:])), "cpu_port_ms": 1e3 * float(np.median(t_cpu)),
                  "points": int(len(packed)), "imu_samples": int(len(fi["v_imu"])),
                  "points_identical_frac": float((got == ref).mean()), "points_max_abs_diff": float(np.abs(got - ref).max()),
                  "note": "flb_imu_undistort (H2D + propagate + undistort + D2H, blocking) vs the single-thread oracle port of UndistortPcl"}
    h.close()

    # ---- BASELINE.json configs[2], configs[3] in the same run (N = 1): the sizes where a bandwidth roofline can be met
    others = None
    if rank == 0 and world == 1 and not args.no_others and args.workload == "C2":
        others = {}
        for name in ("C3", "C4"):
            try:
                others[name] = measure_other_workload(flb, torch, name, local, dev, stream, flush, hbm, peak_src, po)
            except Exception as e:      # never lose the headline line to a secondary leg
                others[name] = {"error": repr(e)}

    # ---- batched frames (SURVEY.md section 7 H2(iv)): the pass kernels at their throughput
    batched = None
    if rank == 0 and world == 1 and not args.no_others and args.workload == "C2":
        batched = {}
        for name, B in (("C2", 64), ("C4", 16)):
            try:
                batched[f"{name}x{B}"] = measure_batched(flb, torch, name, B, local, dev, stream, flush, hbm, peak_src)
            except Exception as e:
                batched[f"{name}x{B}"] = {"error": repr(e)}

    full_frame = None
    if rank == 0 and world == 1 and not args.no_others and args.workload == "C2":
        try:
            full_frame = measure_full_frame(flb, torch, "C2", local, dev, stream, flush)
        except Exception as e:
            full_frame = {"error": repr(e)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32+f64", "data": "synthetic",
            "config": workload_config(cfg, world),
            "l2": "inputs resident; L2 flushed (256 MiB write) between timed steps" if flush is not None
                  else "inputs resident; L2 NOT flushed (working set < L2)",
            "collective": None if world == 1 else ("NCCL all-reduce between per-pass kernels" if args.collective == "nccl"
                                                   else "fused NVLink peer-memory exchange inside the persistent kernels (LL units)"),
            "residuals_per_sec": rows_per_frame * fps, "rows_per_frame": int(rows_per_frame),
            "wall_ms_per_step_incl_flush": 1e3 * t_wall / args.steps,
            "gpu_launches": int(launches), "clocks": clocks,
            "e2e": {"value": e2e_frame_api_fps if e2e_frame_api_fps else e2e_fps, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "steps": e2e_steps,
                    "residuals_per_sec": rows_per_frame * (e2e_frame_api_fps if e2e_frame_api_fps else e2e_fps),
                    "api": "flb_frame_enqueue + flb_state_download_wait (one call per frame, page-locked caller buffers, result read back one "
                           "frame behind)" if e2e_frame_api_fps else "separate upload / update calls, one blocking flb_state_download per frame",
                    "frame_api_serial_value": e2e_frame_api_serial_fps, "live_loop_value": e2e_live_fps,
                    "separate_calls_serial_value": e2e_fps, "pipelined_value": e2e_pipe_fps,
                    "pinned_caller_buffers_value": e2e_pinned_fps, "blocking_calls_value": e2e_blocking_fps,
                    "note": "value (N = 1): every frame moves scan + image + patch list + two states H2D from page-locked host memory and its "
                            "state + reports D2H inside the timed region, through ONE C-ABI call per frame, with the read-back pipelined by one "
                            "frame (the frames are independent: each prior is given up front).  frame_api_serial_value: the same call with "
                            "every result collected before the next frame is enqueued -- the pattern of a live odometry loop whose next "
                            "prior depends on this posterior.  live_loop_value: that dependency kept (the state of frame k+1 is uploaded only "
                            "after frame k's posterior has been read back) but frame k+1's scan / image / patch list -- which do not depend "
                            "on it -- uploaded while frame k runs (separate calls, page-locked buffers).  "
                            "pipelined_value: the same calls with the result read-back one frame behind (flb_state_download_enqueue / "
                            "_wait, two slots): frame k+1 uploads and sorts while frame k runs; every frame still moves its inputs "
                            "H2D and its state + reports D2H inside the timed region.  "
                            "separate_calls_serial_value: device-resident loop of the C ABI (uploads + both updates enqueued, one blocking "
                            "flb_state_download per frame), pageable caller buffers staged by the library, L2 flushed between "
                            "frames; pinned_caller_buffers_value: image/patch buffers from flb_host_alloc, no L2 flush; "
                            "blocking_calls_value: flb_lio_update + flb_vio_update (two synchronisations and state round "
                            "trips per frame, the reference's call shape), no L2 flush"},
            "roofline": roofline, "kernels": fams, "pass_trace": trace, "map_maintenance": map_maint, "imu_undistort": imu_f3,
            "cpu_baseline": cpu, "parity": parity, "nccl_collective": nccl_alt, "replicas": replicas, "other_workloads": others, "batched": batched, "e2e_full_frame": full_frame,
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
