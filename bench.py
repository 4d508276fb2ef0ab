#!/usr/bin/env python
"""bench.py -- headline benchmark of the batched time-stepping contact hot path.

A "step" is one TimeSteppingSimulator::step(dt = 1 ms) of every env of the workload (BASELINE.json configs[1]:
65,536 randomized sitting-box / bouncing-ball envs per GPU, SURVEY.md 8(d) case 2).  Envs are independent, so
N GPUs each own their own 65,536 envs (weak scaling, no collective on the step path); one NCCL all-reduce (max of
the elapsed time, sum of the counters) closes the run.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...   # the CPU restatement of the reference on the host cores

Prints ONE JSON line (rank 0).  Timing: CUDA events on the launching stream around each step kernel, L2 flushed
between steps (a 256 MiB write, outside the events), max over ranks.

  --dump-outputs DIR   rank 0 writes what the timed path returned after its last timed step as DIR/<name>.npy (float64):
                       <part>_q, <part>_v (+ <part>_jq, <part>_jqd) of the stepped paths, z / status / pivots of --workload lcp.
                       Inputs come from fixed seeds, so two builds run with the same arguments can be compared file by file.
                       Compare dumps of the same arm: --impl reference steps its own, smaller seeded batch (the workload's
                       ref_sample envs), so its files have other shapes and other envs than those of the CUDA arm.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

# one hardware queue per stream of a step (main, hard queue, one per LCP class; twice that for the mix): set before CUDA starts
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [ROOT]
sys.dont_write_bytecode = True       # modules that building does not import (tests/oracle_api.py, moby_b200/lcp.py, ...) leave no
                                     # __pycache__ in the source tree: the benchmark writes nothing there
DUMP_BYTES = 60_000_000              # --dump-outputs: above this the dump is a seeded sample of the envs (under 64 MB in all)

# Workloads = BASELINE.json configs.  "small" (configs[1]) is the one the metric is quoted on and the default; the
# others are the larger single-GPU configurations, selectable with --workload.
#   bytes: algorithmic HBM bytes per env-step, 2 * 8 B * (nq + nv) per moving body (SURVEY.md 8d)
WORKLOADS = {
    "small": dict(name="sitting-box/bouncing-ball batch: 65,536 randomized envs per GPU (BASELINE configs[1]; SURVEY 8d case 2)",
                  envs=65536, dt=1e-3, preroll=300, bytes=208.0, cpu_sample=(512, 40), ref_sample=4096,
                  make=lambda sc, ne, seed: sc.small_lcp_batch(ne, seed=seed)),
    "stacks": dict(name="example/stacks: 10-box stack, 4,096 envs per GPU, LCP n = 320 (BASELINE configs[2]; SURVEY 8d case 3)",
                   envs=4096, dt=1e-3, preroll=2, bytes=2080.0, cpu_sample=(2, 1), ref_sample=16, cpu_limit_s=60,
                   make=lambda sc, ne, seed: sc.box_stack(ne, 10, seed=seed)),
    "ur10": dict(name="example/ur10 arm (9-DoF RCArticulatedBody, CRB forward dynamics) + block + table, mu = 100 as ur10.xml:20 (no-slip impact model), "
                      "16,384 envs per GPU (BASELINE configs[3]; SURVEY 8d case 4)",
                 envs=16384, dt=5e-4, preroll=300, bytes=2.0 * 8.0 * (9 + 9) + 208.0, cpu_sample=(256, 40), ref_sample=2048,   # 300 like configs[1]; the step time follows the arm's motion: 3.1-4.3 ms over windows of 20 steps (tools/ur10_phases.py)
                 make=lambda sc, ne, seed: sc.ur10(ne, seed=seed, mu=100.0)),
    "feeder": dict(name="parts-feeder-like (SURVEY 8d case 5 variant): prismatic shaker tray (RCArticulatedBody) + free box part, mu = 0.01, "
                        "16,384 envs per GPU (part of BASELINE configs[4])",
                   envs=16384, dt=1e-3, preroll=50, bytes=2.0 * 8.0 * (1 + 1) + 208.0, cpu_sample=(256, 40), ref_sample=2048,
                   make=lambda sc, ne, seed: sc.parts_feeder(ne, seed=seed)),
    "wheel": dict(name="example/rimless-wheel (wheel.xml + init.cpp): 6-spoke wheel rolling downhill, spoke-tip contacts of coldet-plugin.cpp, mu = 100 "
                       "(no-slip impact model), theta_dot in [0.5, 1.5] rad/s, 16,384 envs per GPU (part of BASELINE configs[4])",
                  envs=16384, dt=1e-3, preroll=50, bytes=208.0, cpu_sample=(512, 40), ref_sample=4096,
                  make=lambda sc, ne, seed: sc.rimless_wheel(ne, theta_dot=1.0, seed=seed)),
}
# BASELINE configs[4]: both scene types on EVERY GPU in equal shares (SURVEY 8e: interleave scene types across GPUs rather
# than giving each GPU one scene), two batches stepped concurrently on two streams of the rank's GPU.
MIX = dict(name="parts-feeder / rimless-wheel mix (BASELINE configs[4]; SURVEY 8d case 5): per GPU 8,192 parts-feeder-like envs (prismatic shaker tray + "
                "free box part, mu = 0.01) and 8,192 rimless wheels (mu = 100), two batches stepped concurrently",
           envs=16384, dt=1e-3, preroll=50, parts=("feeder", "wheel"))


class SimGroup:
    """Several batches (one TimeSteppingSimulator handle each) of one GPU stepped together: each batch on its own stream,
    forked from and joined to the caller's stream, so events on the caller's stream bracket all of them."""

    def __init__(self, sims, names):
        import torch
        self.sims, self.names = sims, names
        self.streams = [torch.cuda.Stream() for _ in sims]

    def step(self, dt, n_steps=1):
        import torch
        cur = torch.cuda.current_stream()
        for sim, st in zip(self.sims, self.streams):
            st.wait_stream(cur)
            sim.step(dt, n_steps, stream=st.cuda_stream)
        for st in self.streams:
            cur.wait_stream(st)
        return dt

    def reset_counters(self):
        for sim in self.sims:
            sim.reset_counters()

    def launch_count(self):
        return sum(sim.launch_count() for sim in self.sims)

    def counters(self):
        out = {}
        for sim in self.sims:
            for k, v in sim.counters().items():
                out[k] = max(out.get(k, 0), v) if k == "max_lcp_n" else out.get(k, 0) + v
        return out

    def kernel_profile(self, enable=True, reset=True):
        out = []
        for sim, name in zip(self.sims, self.names):
            for k in sim.kernel_profile(enable=enable, reset=reset) or []:
                k = dict(k)
                k["name"] = name + ":" + k["name"]
                out.append(k)
        return out



def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    hbm, src = 6650.0, "fallback (B200_PROFILING.md)"
    if os.path.exists(p):
        try:
            hbm, src = float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    fp64, fsrc = 36.07, "measured r01 (profiles/r01_fp64_peak.json)"
    q = os.path.join(ROOT, "profiles", "r01_fp64_peak.json")
    if os.path.exists(q):
        try:
            fp64 = float(json.load(open(q))["fp64_dfma_tflops"])
        except Exception:
            pass
    return hbm, src, fp64, fsrc


class StdoutGuard:
    """Rank 0 prints ONE JSON line: while the benchmark runs, file descriptor 1 points at stderr so that library banners
    (NCCL prints its version to stdout at communicator creation) cannot precede it; emit() restores it for the line."""

    def __init__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def emit(self, obj):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        print(json.dumps(obj), flush=True)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.lines, self.p = gpu_index, [], None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: [self.lines.append(l) for l in self.p.stdout], daemon=True).start()
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        sm, mx, reasons = [], None, set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def _dump_outputs(out_dir, parts):
    """--dump-outputs: parts = [(prefix, axis, {name: array})], `axis` the env (or problem) index of every array of the part.
    Writes out_dir/<prefix><name>.npy in float64.  When everything would exceed DUMP_BYTES, each part keeps the same fixed,
    seeded sample of its envs in every array, and the sampled indices go to out_dir/<prefix>sample.npy."""
    os.makedirs(out_dir, exist_ok=True)
    n_of = lambda axis, arrs: next(iter(arrs.values())).shape[axis]      # noqa: E731
    total = 8 * sum(sum(a.size for a in arrs.values()) + n_of(axis, arrs) for _, axis, arrs in parts)   # arrays + sample indices
    frac = min(1.0, DUMP_BYTES / total)
    for prefix, axis, arrs in parts:
        if frac < 1.0:
            n = n_of(axis, arrs)
            idx = np.sort(np.random.default_rng(0).choice(n, int(n * frac), replace=False))
            np.save(os.path.join(out_dir, prefix + "sample.npy"), idx.astype(np.float64))
            arrs = {k: np.take(a, idx, axis=axis) for k, a in arrs.items()}
        for k, a in arrs.items():
            np.save(os.path.join(out_dir, prefix + k + ".npy"), np.asarray(a, np.float64))


def _state_arrays(state, joints):
    """{q, v[, jq, jqd]} of one batch: state = (q, v) [body][7|6][env], joints = (jq, jqd) [dof][env] or None."""
    out = dict(zip(("q", "v"), state))
    if joints is not None:
        out.update(zip(("jq", "jqd"), joints))
    return out


def _cpu_baseline(scene, q, v, joints, dt, n_envs, n_steps, threads):
    """The oracle (CPU restatement of the reference; the reference itself cannot be built here) on the host cores."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_api as O
    import copy
    sc = copy.copy(scene)
    sc.q, sc.v = q, v
    batch = O.OracleBatch(sc, 0, n_envs)
    if joints is not None:
        batch.set_joint_state(*joints)
    t0 = time.perf_counter()
    c = batch.run(dt, n_steps, threads=threads)
    el = time.perf_counter() - t0
    return c["env_steps"] / el, c["lcp_solves"] / el, el, c


def _cpu_baseline_bounded(limit_s, *a):
    """_cpu_baseline in a forked child with a wall-clock limit (the oracle is CPU-only code: the child never touches CUDA).
    Degenerate n = 320 stack LCPs can cost the LU-per-pivot CPU solver minutes per env-step; past the limit the child is killed
    (by its own PID) and the sample's rate is reported as an upper bound: (env-steps asked for) / limit."""
    if not limit_s:
        return _cpu_baseline(*a) + (False,)
    import multiprocessing as mp
    ctx = mp.get_context("fork")
    qd = ctx.Queue()

    def work():
        qd.put(_cpu_baseline(*a))
    pr = ctx.Process(target=work)
    pr.start()
    pr.join(limit_s)
    if pr.is_alive():
        pr.kill()
        pr.join()
        n_envs, n_steps = a[5], a[6]
        return n_envs * n_steps / limit_s, float("nan"), float(limit_s), {}, True
    return qd.get() + (False,)


def _stab_iters(args):
    """constraint-stabilization-max-iterations of the measured scene: ur10.xml sets 0 itself (example/ur10/ur10.xml:12)."""
    return 0 if (args.stabilization == "off" or args.workload == "ur10") else -1


def _stab_text(args):
    return ("on (reference default: until no pair is closer than sqrt(eps), ConstraintStabilization.cpp:53-59)" if _stab_iters(args)
            else "off (constraint-stabilization-max-iterations=0" + (", as example/ur10/ur10.xml:12)" if args.workload == "ur10" else ")"))


def _device_timed(sim, dt, steps, warmup, flush, stream):
    """steps x step(dt) timed with CUDA events on the launching stream, L2 flushed between steps; returns seconds."""
    import torch
    for _ in range(warmup):
        flush.fill_(1)
        sim.step(dt, 1)
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in ev:
        flush.fill_(0)
        a.record(stream)
        sim.step(dt, 1)
        b.record(stream)
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in ev) * 1e-3


def _secondary(args, W, scenes, rank_seed, local_rank, flush, stream):
    """Rank 0, after the headline measurement: (1) the same workload with constraint stabilization off -- round 1's
    configuration, kept beside the headline; (2) drift against the oracle: a fresh 512-env batch of the workload stepped
    300 steps on the GPU and by the oracle from the same initial state, share of envs above 1e-9 (relative)."""
    import copy
    from moby_b200 import TimeSteppingSimulator, sharding
    out = {}
    DT = W["dt"]
    ne = args.envs_per_gpu or W["envs"]
    if _stab_iters(args) != 0:
        sc = W["make"](scenes, ne, rank_seed)
        if args.min_step == "default" and args.workload == "small":
            sc.min_step_size_env = None
        sc.stabilization_max_iterations = 0
        sim = TimeSteppingSimulator(sc, device=local_rank)
        sim.step(DT, args.preroll)
        steps = max(5, args.steps // 2)
        t = _device_timed(sim, DT, steps, 3, flush, stream)
        out["stabilization_off"] = {"value": ne * steps / t, "unit": "env-steps/s", "ms_per_step": 1e3 * t / steps, "steps": steps, "n_gpus": 1,
                                    "note": "same workload and seed on rank 0's GPU with constraint-stabilization-max-iterations=0 (the configuration of round 1's numbers)"}
        sim.close()
    if not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_api as O
        n_d, s_d = min(512, ne), 300
        full = W["make"](scenes, max(n_d, 512), rank_seed)
        if args.min_step == "default" and args.workload == "small":
            full.min_step_size_env = None
        full.stabilization_max_iterations = _stab_iters(args)
        sc = sharding.select_envs(full, np.arange(n_d))
        sim = TimeSteppingSimulator(sc, device=local_rank)
        sim.step(DT, s_d)
        q, v = sim.get_state()
        sim.close()
        ob = O.OracleBatch(sc)
        ob.run(DT, s_d, threads=os.cpu_count() or 1)
        qo, vo = ob.get_state_soa()
        scale = np.maximum(1.0, np.maximum(np.abs(qo).max(axis=(0, 1)), np.abs(vo).max(axis=(0, 1))))
        err = np.maximum(np.abs(q - qo).max(axis=(0, 1)), np.abs(v - vo).max(axis=(0, 1))) / scale
        out["drift"] = {"envs": n_d, "steps": s_d, "envs_above_1e-9": int((err > 1e-9).sum()), "share_above_1e-9": float((err > 1e-9).mean()),
                        "max_rel_err": float(err.max()), "median_rel_err": float(np.median(err)),
                        "note": "GPU vs oracle/ from the same initial state; envs above 1e-9 ran Lemke on a singular LCP whose pivot path "
                                "differs between the tableau and the LU-per-pivot form (tests/parity_util.py, profiles/r02_lemke_path_sensitivity.json)"}
    return out


def _other_workloads(local_rank, flush, stream):
    """Rank 0, after the headline: short device-timed runs of the other BASELINE configs on rank 0's GPU, so that the one JSON
    line the driver records also carries them (each is a full bench line of its own under --workload)."""
    import torch
    from moby_b200 import TimeSteppingSimulator, scenes
    out = {}
    steps = 10
    try:
        W = WORKLOADS["ur10"]
        sc = W["make"](scenes, W["envs"], 0xB200)
        sc.stabilization_max_iterations = 0
        sim = TimeSteppingSimulator(sc, device=local_rank)
        sim.step(W["dt"], W["preroll"])
        t = _device_timed(sim, W["dt"], steps, 3, flush, stream)
        c = sim.counters()
        out["ur10"] = {"value": W["envs"] * steps / t, "unit": "env-steps/s", "ms_per_step": 1e3 * t / steps, "envs_per_gpu": W["envs"], "steps": steps, "n_gpus": 1,
                       "lcp_failures": c["lcp_failures"], "workload": W["name"]}
        sim.close()
        names = MIX["parts"]
        sims = []
        for nm in names:
            sc = WORKLOADS[nm]["make"](scenes, MIX["envs"] // len(names), 0xB200)
            sc.stabilization_max_iterations = -1
            sims.append(TimeSteppingSimulator(sc, device=local_rank))
        grp = SimGroup(sims, names)
        grp.step(MIX["dt"], MIX["preroll"])
        t = _device_timed(grp, MIX["dt"], steps, 3, flush, stream)
        out["mix"] = {"value": MIX["envs"] * steps / t, "unit": "env-steps/s", "ms_per_step": 1e3 * t / steps, "envs_per_gpu": MIX["envs"], "steps": steps, "n_gpus": 1,
                      "lcp_failures": grp.counters()["lcp_failures"], "workload": MIX["name"]}
        for sm in sims:
            sm.close()
        # batched Lemke solver, n = 32, operands in HBM (bench.py --workload lcp)
        from moby_b200 import capi, lcp as L
        n, batch = 32, 131072
        dev = torch.device("cuda", local_rank)
        gen = torch.Generator(device=dev); gen.manual_seed(0xB200)
        A = torch.randn(batch, n, n, dtype=torch.float64, device=dev, generator=gen)
        Mc = (torch.bmm(A, A.transpose(1, 2)) / n + 1e-3 * torch.eye(n, dtype=torch.float64, device=dev)).transpose(-1, -2).contiguous()
        del A
        q = torch.randn(batch, n, dtype=torch.float64, device=dev, generator=gen)
        z = torch.zeros_like(q); status = torch.zeros(batch, dtype=torch.int32, device=dev); pivots = torch.zeros_like(status)
        solve = lambda: capi.check(capi.lib().b200moby_lcp_lemke_batched(batch, n, Mc.data_ptr(), q.data_ptr(), z.data_ptr(), -1.0, -1.0, status.data_ptr(),  # noqa: E731
                                                                          pivots.data_ptr(), None, 0, L._stream_ptr(None)))
        for _ in range(3):
            solve()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(steps):
            solve()
        b.record(stream)
        torch.cuda.synchronize()
        t = a.elapsed_time(b) * 1e-3
        out["lcp_n32"] = {"value": batch * steps / t, "unit": "LCP solves/s", "ms_per_launch": 1e3 * t / steps, "batch": batch, "n": n,
                          "algorithmic_GBps": 8.0 * (n * n + 2 * n) * batch * steps / t / 1e9, "solved": int(((status == 0) | (status == 1)).sum().item())}
    except Exception as ex:                       # the headline must not be lost to a side measurement
        out["error"] = repr(ex)
    return out


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path, restated (oracle/, kind "port"),
    all host threads, each step = one step of a bounded 4,096-env sample of the same seeded workload."""
    if rank != 0:
        return
    from moby_b200 import scenes
    W = MIX if args.workload == "mix" else WORKLOADS[args.workload]
    DT, WORKLOAD = W["dt"], W["name"]
    names = W.get("parts", (args.workload,))
    cores = os.cpu_count() or 1
    if args.preroll < 0:
        args.preroll = W["preroll"]
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_api as O
    O.build()
    batches, sample = [], 0
    for nm in names:
        n_i = WORKLOADS[nm]["ref_sample"] // len(names)
        scene = WORKLOADS[nm]["make"](scenes, n_i, 0xB200)
        if args.min_step == "default" and nm == "small":
            scene.min_step_size_env = None
        scene.stabilization_max_iterations = _stab_iters(args)
        batch = O.OracleBatch(scene, 0, n_i)
        batch.run(DT, args.preroll, threads=cores)
        for _ in range(args.warmup):
            batch.run(DT, 1, threads=cores)
        batches.append(batch)
        sample += n_i
    c0 = [b.run(DT, 0, threads=1) for b in batches]
    t0 = time.perf_counter()
    for _ in range(args.steps):
        c1 = [b.run(DT, 1, threads=cores) for b in batches]
    el = time.perf_counter() - t0
    if args.dump_outputs:
        parts = []
        for nm, b in zip(names, batches):
            joints = None if b.rc is None else [np.stack(x, axis=1) for x in zip(*(b.get_joint_state(i) for i in range(b.e1 - b.e0)))]
            parts.append((nm + "_", -1, _state_arrays(b.get_state_soa(), joints)))
        _dump_outputs(args.dump_outputs, parts)
    val = sample * args.steps / el
    c0 = {"lcp_solves": sum(c["lcp_solves"] for c in c0)}
    c1 = {"lcp_solves": sum(c["lcp_solves"] for c in c1)}
    out = {
        "impl": "reference", "metric": "env_steps_per_s", "value": val, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "dt": DT, "preroll_steps": args.preroll, "seed": "0xB200", "min_step_size": args.min_step,
                   "stabilization": _stab_text(args)},
        "lcp_solves_per_s": (c1["lcp_solves"] - c0["lcp_solves"]) / el,
        "cpu_baseline": {"value": val, "unit": "env-steps/s", "cores": cores, "kind": "port",
                         "sample": f"first {sample} envs of the seeded batch, one step per timed step, {cores} host threads; "
                                   "the reference cannot be compiled here (Ravelin/Boost/qhull/libxml2 absent), so this is the "
                                   "oracle/ restatement"},
        "e2e": {"value": val, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def run_lcp(args, rank, world, local_rank):
    """--workload lcp: SURVEY.md 8(d) case 6, the batched solver microbenchmark.  A step = one call of
    b200moby_lcp_lemke_batched over a batch of random LCPs (M = A A^T / n + 1e-3 I, q ~ N(0,1)) resident in HBM;
    metric = LCP solves/s.  Roofline: algorithmic bytes 8 (n^2 + 2n) per solve (read M, q; write z) against HBM."""
    import torch
    import torch.distributed as dist
    from moby_b200 import lcp as L
    assert torch.cuda.is_available(), "bench.py needs a CUDA device: the hot path has no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    guard = StdoutGuard()
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n = args.lcp_n
    batch = args.envs_per_gpu or max(4096, min(262144, (2 << 30) // (8 * n * n)))      # ~2 GiB of matrices: larger than L2
    gen = torch.Generator(device=dev); gen.manual_seed(0xB200 + rank)
    A = torch.randn(batch, n, n, dtype=torch.float64, device=dev, generator=gen)
    M = torch.bmm(A, A.transpose(1, 2)) / n + 1e-3 * torch.eye(n, dtype=torch.float64, device=dev)
    del A
    q = torch.randn(batch, n, dtype=torch.float64, device=dev, generator=gen)
    Mc = M.transpose(-1, -2).contiguous()          # column-major blocks, as the C ABI takes them
    z = torch.zeros_like(q); status = torch.zeros(batch, dtype=torch.int32, device=dev); pivots = torch.zeros_like(status)
    from moby_b200 import capi
    lib = capi.lib()
    stream = torch.cuda.current_stream()

    def solve():
        capi.check(lib.b200moby_lcp_lemke_batched(batch, n, Mc.data_ptr(), q.data_ptr(), z.data_ptr(), -1.0, -1.0, status.data_ptr(),
                                                  pivots.data_ptr(), None, 0, L._stream_ptr(None)))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        solve()
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    sampler = ClockSampler(local_rank); sampler.start()
    barrier()
    for a, b in ev:
        a.record(stream); solve(); b.record(stream)
    barrier()
    clocks = sampler.stop()
    t_dev = sum(a.elapsed_time(b) for a, b in ev) * 1e-3
    ok = int(((status == 0) | (status == 1)).sum().item())
    piv_mean = float(pivots.double().mean().item())
    if args.dump_outputs and rank == 0:
        _dump_outputs(args.dump_outputs, [("", 0, {"z": z.cpu().numpy(), "status": status.cpu().numpy(), "pivots": pivots.cpu().numpy()})])
    # end to end with host buffers through the host-form entry point (H2D M, q; solve; D2H z inside the call)
    Mh, qh = M.cpu().numpy(), q.cpu().numpy()
    nb_e2e = min(batch, 32768)
    L.lcp_lemke_host(Mh[:nb_e2e], qh[:nb_e2e], device=local_rank)
    e0 = time.perf_counter()
    for _ in range(3):
        zh, sh, ph = L.lcp_lemke_host(Mh[:nb_e2e], qh[:nb_e2e], device=local_rank)
    t_e2e = (time.perf_counter() - e0) / 3
    tt = torch.tensor([t_dev, t_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_dev, t_e2e = tt.tolist()
    if rank == 0:
        hbm_peak, hbm_src, fp64_peak, fp64_src = _peaks()
        alg_bytes = 8.0 * (n * n + 2 * n) * batch
        ms = 1e3 * t_dev / args.steps
        gbs = alg_bytes / (ms * 1e-3) / 1e9
        flops = piv_mean * 2.0 * n * (n + 1) * batch
        out = {"metric": "lcp_solves_per_s", "value": batch * world * args.steps / t_dev, "unit": "LCP solves/s", "n_gpus": world, "steps": args.steps,
               "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
               "data": "synthetic",
               "config": {"workload": f"batched Lemke solver microbenchmark (SURVEY 8d case 6): {batch} random LCPs per GPU, n = {n}, M = A A^T / n + 1e-3 I, operands in HBM",
                          "batch_per_gpu": batch, "n": n, "l2": f"inputs {alg_bytes / 2**20:.0f} MiB per launch, larger than L2", "parallelism": f"problems sharded x{world}"},
               "solved": ok, "pivots_per_solve": piv_mean,
               "e2e": {"value": nb_e2e * world / t_e2e, "unit": "LCP solves/s", "h2d_bytes_per_step": int(8 * (n * n + n) * nb_e2e), "d2h_bytes_per_step": int(8 * n * nb_e2e + 8 * nb_e2e),
                       "how": f"b200moby_lcp_lemke_host on {nb_e2e} problems: pageable host M, q -> device, solve, z/status/pivots -> host inside the call"},
               "gpu_launches": args.steps * world, "clocks": clocks,
               "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak, "traffic": None,
                            "kernel": "lcp_warp_kernel" if n <= 160 else "lcp_block_kernel", "kernel_ms": ms, "peak_source": hbm_src,
                            "fp64": {"achieved": flops / (ms * 1e-3) / 1e12, "peak": fp64_peak, "unit": "TFLOP/s", "frac": flops / (ms * 1e-3) / 1e12 / fp64_peak,
                                     "flops": "pivots * 2 n (n + 1) (tableau rank-one update, SURVEY 8d)"}}}
        if not args.no_cpu_baseline:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import oracle_api as O
            O.build()
            ns = max(8, min(2000, int(4e8 / (n ** 4 + 1))))
            t0 = time.perf_counter()
            for b in range(ns):
                O.lcp_lemke(Mh[b], qh[b])
            el = time.perf_counter() - t0
            out["cpu_baseline"] = {"value": ns / el, "unit": "LCP solves/s", "cores": 1, "kind": "port",
                                   "sample": f"first {ns} problems of rank 0's batch, 1 thread ({el:.1f} s); oracle/ restatement of LCP::lcp_lemke (LU per pivot, as the reference)"}
        guard.emit(out)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--lcp-n", type=int, default=32, help="--workload lcp: LCP dimension")
    ap.add_argument("--workload", default="small", choices=sorted(WORKLOADS) + ["lcp", "mix"], help="BASELINE.json config (default: configs[1], the one the metric is quoted on)")
    ap.add_argument("--envs-per-gpu", type=int, default=0, help="default: the workload's own batch size")
    ap.add_argument("--preroll", type=int, default=-1, help="untimed steps before warm-up so contacts are active (default: per workload)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--stabilization", default="on", choices=["on", "off"],
                    help="on: ConstraintStabilization after every step, the reference's default (ConstraintStabilization.cpp:53-59); "
                         "off: constraint-stabilization-max-iterations=0 (round 1's configuration, as example/ur10/ur10.xml:12)")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary measurements (stabilization off, drift against the oracle)")
    ap.add_argument("--min-step", default="scene", choices=["scene", "default"],
                    help="scene: min-step-size of the source scenes (test/box.xml: 1e-3, bouncing-ball.xml: sqrt(eps)); "
                         "default: sqrt(eps) everywhere (TimeSteppingSimulator.cpp:48)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path computed in its last timed step as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
    if args.workload == "lcp":
        if args.impl == "reference":
            if rank == 0:
                print(json.dumps({"impl": "reference", "unavailable": "--workload lcp carries its CPU arm as cpu_baseline; the reference arm times the stepped path"}))
            return
        run_lcp(args, rank, world, local_rank)
        return
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from moby_b200 import TimeSteppingSimulator, scenes
    assert torch.cuda.is_available(), "bench.py needs a CUDA device: the hot path has no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    guard = StdoutGuard()
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W = MIX if args.workload == "mix" else WORKLOADS[args.workload]
    DT, WORKLOAD = W["dt"], W["name"]
    ne = args.envs_per_gpu or W["envs"]
    if args.preroll < 0:
        args.preroll = W["preroll"]
    # parts: (name, workload entry, envs); one batch normally, one per scene type for the mix
    names = W.get("parts", (args.workload,))
    sizes = [ne // len(names) + (1 if i < ne % len(names) else 0) for i in range(len(names))]
    part_scenes = []
    for nm, n_i in zip(names, sizes):
        sc = WORKLOADS[nm]["make"](scenes, n_i, 0xB200 + rank)  # every rank owns its own envs (contiguous shard of the job)
        if args.min_step == "default" and nm == "small":
            sc.min_step_size_env = None
        sc.stabilization_max_iterations = _stab_iters(args)
        part_scenes.append(sc)
    part_sims = [TimeSteppingSimulator(sc, device=local_rank) for sc in part_scenes]
    scene = part_scenes[0]
    sim = part_sims[0] if len(part_sims) == 1 else SimGroup(part_sims, names)
    bytes_env = sum(WORKLOADS[nm]["bytes"] * n_i for nm, n_i in zip(names, sizes)) / ne
    stream = torch.cuda.current_stream()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)     # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sim.step(DT, args.preroll)
    for _ in range(max(args.warmup, 3)):
        flush.fill_(1)
        sim.step(DT, 1)
    barrier()
    sim.reset_counters()
    launches0 = sim.launch_count()
    # the state the timed region starts from (also feeds the CPU baseline): per part q, v and the articulated body's joint state
    state0 = [(ps.get_state(), ps.get_joint_state() if sc.rc is not None else None) for ps, sc in zip(part_sims, part_scenes)]
    # timed region: every step is ONE cudaGraphLaunch (sim_kernels.cu: b200moby_step captures the step's launches, memsets and
    # stream fork / join once).  Per-kernel CUDA events cannot sit inside that graph, so the roofline block's kernel durations
    # come from a second pass below: the same number of steps with plain launches and an event pair around every kernel.
    sim.kernel_profile(enable=False, reset=True)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    wall0 = time.perf_counter()
    for a, b in ev:
        flush.fill_(0)                   # L2 flush, outside the timed events
        a.record(stream)
        sim.step(DT, 1)                  # the hot path: advance / impact-class / finish kernels of one step
        b.record(stream)
    barrier()
    wall = time.perf_counter() - wall0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:           # before the profile pass below steps the same batches further
        _dump_outputs(args.dump_outputs, [(nm + "_", -1, _state_arrays(ps.get_state(), ps.get_joint_state() if sc.rc is not None else None))
                                          for nm, ps, sc in zip(names, part_sims, part_scenes)])
    kernel_ms = [a.elapsed_time(b) for a, b in ev]
    t_dev = sum(kernel_ms) * 1e-3
    cnt = sim.counters()
    r_cnt = dict(cnt)
    launches = sim.launch_count() - launches0
    # profile pass: the next `steps` steps of the same batch, plain launches, CUDA events around every kernel on its own stream
    sim.kernel_profile(enable=True, reset=True)
    evp = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for a, b in evp:
        flush.fill_(0)
        a.record(stream)
        sim.step(DT, 1)
        b.record(stream)
    torch.cuda.synchronize()
    kprof = sim.kernel_profile(enable=False, reset=True)
    profile_ms = sum(a.elapsed_time(b) for a, b in evp) / args.steps
    # ---- end to end through the public API with HOST buffers: H2D state, step, D2H state, every step ----
    class HostLoop:
        """One batch's host-resident state: pinned q, v (and joint state) in, pinned out, swapped after every step."""

        def __init__(self, ps, st0, st):
            (q0, v0), j0 = st0
            self.sim, self.stream = ps, st
            self.inp = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in (q0, v0) + (tuple(j0) if j0 is not None else ())]
            self.dev = [torch.empty_like(a, device=dev) for a in self.inp]
            self.out = [torch.empty_like(a).pin_memory() for a in self.inp]
            self.bytes = sum(a.numel() * 8 for a in self.inp)

        def issue(self):
            with torch.cuda.stream(self.stream):
                for d, h in zip(self.dev, self.inp):
                    d.copy_(h, non_blocking=True)
                self.sim.set_state_dev(self.dev[0], self.dev[1])
                if len(self.dev) > 2:
                    self.sim.set_joint_state_dev(self.dev[2], self.dev[3])
                self.sim.step(DT, 1)
                self.sim.get_state_dev(self.dev[0], self.dev[1])
                if len(self.dev) > 2:
                    self.sim.get_joint_state_dev(self.dev[2], self.dev[3])
                for h, d in zip(self.out, self.dev):
                    h.copy_(d, non_blocking=True)

        def swap(self):
            self.inp, self.out = self.out, self.inp          # next step starts from this step's result

    loops = [HostLoop(ps, st0, stream if len(part_sims) == 1 else torch.cuda.Stream()) for ps, st0 in zip(part_sims, state0)]
    h2d = sum(l.bytes for l in loops)

    def e2e_step():
        for l in loops:
            l.issue()
        torch.cuda.synchronize()
        for l in loops:
            l.swap()

    for _ in range(2):
        e2e_step()
    barrier()
    e0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    barrier()
    t_e2e = time.perf_counter() - e0
    # ---- max over ranks, sums of counters ----
    tt = torch.tensor([t_dev, t_e2e, wall], dtype=torch.float64, device=dev)
    cc = torch.tensor([cnt[k] for k in ("env_steps", "mini_steps", "lcp_solves", "pivots", "pivot_flops", "lcp_failures",
                                        "lcp_fast_calls", "lemke_calls", "contacts")], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(cc, op=dist.ReduceOp.SUM)
    t_dev, t_e2e, wall = tt.tolist()
    env_steps, mini_steps, lcp_solves, pivots, pivot_flops, failures, fast_calls, lemke_calls, contacts = cc.tolist()
    if rank == 0:
        total_envs = ne * world
        hbm_peak, hbm_src, fp64_peak, fp64_src = _peaks()
        k_ms = float(np.mean(kernel_ms))
        # roofline of the dominant kernel (largest summed duration over the timed steps), per launch on this rank:
        # algorithmic bytes = state in + state out of the envs the launch processed (+ warm start in/out for an impact
        # kernel), algorithmic flops = the kernel's own recorded pivot and assembly flops (SURVEY.md 8d formulas)
        dom = max(kprof, key=lambda k: k["ms"])
        dom_launch_ms = dom["ms"] / max(dom["launches"], 1)
        dom_bytes_env = (WORKLOADS[dom["name"].split(":")[0]]["bytes"] if ":" in dom["name"] else bytes_env) + (2.0 * 8.0 * dom["lcp_nmax"] if dom["lcp_nmax"] else 0.0)
        alg_bytes = dom_bytes_env * dom["envs"] / max(dom["launches"], 1)
        alg_flops = dom["flops"] / max(dom["launches"], 1)
        achieved_gbs = alg_bytes / (dom_launch_ms * 1e-3) / 1e9
        achieved_tf = alg_flops / (dom_launch_ms * 1e-3) / 1e12
        step_ms_sum = sum(k["ms"] for k in kprof) or 1.0
        # DRAM bytes per launch of the dominant kernel: read from the round's ncu capture summary under profiles/ (written by
        # hand from `ncu --set full` raw pages, see its "source" key) when it covers this workload, batch size and kernel; null otherwise
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                if tj.get("workload") == args.workload and tj.get("envs_per_gpu") == ne:
                    traffic = tj["kernels"].get(dom["name"])
                    traffic_src = "profiles/r02_ncu_traffic.json" if traffic is not None else None
            except Exception:
                pass
        out = {
            "metric": "env_steps_per_s", "value": total_envs * args.steps / t_dev, "unit": "env-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": 1e3 * t_dev / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "envs_per_gpu": ne, "dt": DT, "preroll_steps": args.preroll, "seed": "0xB200+rank",
                       "min_step_size": ("boxes 1e-3 (test/box.xml), balls sqrt(eps) (bouncing-ball.xml)" if args.min_step == "scene" else "sqrt(eps) everywhere") if args.workload == "small" else scene.min_step_size,
                       "impact_model": "QP-as-LCP (default build); no-slip model for islands with mu >= 100", "stabilization": _stab_text(args),
                       "l2": "flushed between timed steps (256 MiB write outside the events)", "launch": "one CUDA graph per step (cudaGraphLaunch) for two-round plans such as configs[1]; plain stream launches for the four-round plans of scenes with large LCPs (UR10, stacks)", "parallelism": f"envs sharded x{world}"},
            "lcp_solves_per_s": lcp_solves / t_dev,
            "mini_steps_per_step": mini_steps / max(env_steps, 1.0), "lcp_solves_per_env_step": lcp_solves / max(env_steps, 1.0),
            "pivots_per_solve": pivots / max(lcp_solves, 1.0), "lemke_calls": lemke_calls, "lcp_fast_calls": fast_calls,
            "lcp_failures": failures, "contacts_per_env_step": contacts / max(env_steps, 1.0), "ca_iterations_per_env_step": r_cnt["ca_iterations"] / max(r_cnt["env_steps"], 1),
            "wall_s_timed_region": wall,
            "e2e": {"value": total_envs * args.steps / t_e2e, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": h2d,
                    "how": "pinned host q,v (+ joint state) -> device -> b200moby_set_state_dev -> step -> get_state_dev -> pinned host, every step; wall clock around "
                           "the loop, no L2 flush between steps (the device-timed `value` flushes L2 before every step, so e2e can come out above it); the host-pointer "
                           "entry points b200moby_set_state / get_state do the same copies synchronously from pageable memory"},
            "gpu_launches": launches * world,
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": achieved_gbs / hbm_peak,
                         "traffic": traffic, "traffic_source": traffic_src, "kernel": dom["name"],
                         "kernel_timing": "second pass of the same number of steps right after the timed region, plain launches with a CUDA event pair around every "
                                          "kernel on its own stream (the timed region itself is one CUDA graph launch per step)", "profile_pass_ms_per_step": profile_ms, "kernel_ms": dom_launch_ms, "launches": dom["launches"],
                         "envs_per_launch": dom["envs"] / max(dom["launches"], 1), "share_of_kernel_time": dom["ms"] / step_ms_sum,
                         "peak_source": hbm_src,
                         "note": "pivoting is a dependent-latency chain per env: neither HBM nor the FP64 pipe is the limiter (see DESIGN.md 3-4); "
                                 "fp64 is the same launch against the measured DFMA peak",
                         "kernels": [{"name": k["name"], "ms_per_step": k["ms"] / args.steps, "envs_per_step": k["envs"] / args.steps,
                                      "gflop_per_step": k["flops"] / args.steps / 1e9} for k in kprof if k["launches"]],
                         "fp64": {"achieved": achieved_tf, "peak": fp64_peak, "unit": "TFLOP/s", "frac": achieved_tf / fp64_peak,
                                  "peak_source": fp64_src,
                                  "flops": "SURVEY 8(d): sum pivots*2n(n+1) + F_delassus + F_apply per solve + F_fd + F_narrow per mini-step, all from recorded counts"}},
        }
        if not args.no_secondary and len(names) == 1:
            torch.cuda.synchronize()
            for ps in part_sims:
                ps.close()                   # one live simulator per GPU at a time: the secondary runs get the same schedule as the headline
            out["secondary"] = _secondary(args, W, scenes, 0xB200 + rank, local_rank, flush, stream)
            if args.workload == "small":
                out["secondary"]["other_workloads"] = _other_workloads(local_rank, flush, stream)
        out["stabilization"] = {"iterations_per_env_step": r_cnt["stab_iterations"] / max(r_cnt["env_steps"], 1),
                                "lcp_solves_per_env_step": r_cnt["stab_lcp_solves"] / max(r_cnt["env_steps"], 1),
                                "line_search_failures": r_cnt["stab_line_search_failures"]}
        if not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            tot = {1: [0.0, 0.0, 0.0], cores: [0.0, 0.0, 0.0]}        # env-steps, LCP solves, seconds
            desc = []
            bounded = False
            for nm, sc, n_i, ((q0, v0), j0) in zip(names, part_scenes, sizes, state0):
                n_cpu, s_cpu = WORKLOADS[nm]["cpu_sample"]
                n_cpu = min(n_cpu, n_i)
                for thr, n_s in ((1, n_cpu), (cores, min(n_cpu * 4, n_i))):
                    val, lps, el, _, capped = _cpu_baseline_bounded(WORKLOADS[nm].get("cpu_limit_s"), sc, q0, v0, j0, DT, n_s, s_cpu, thr)
                    bounded = bounded or capped
                    tot[thr][0] += val * el; tot[thr][1] += (0.0 if capped else lps * el); tot[thr][2] += el
                desc.append(f"first {n_cpu} {nm} envs" if len(names) > 1 else f"first {n_cpu} envs")
            out["cpu_baseline"] = {"value": tot[1][0] / tot[1][2], "unit": "env-steps/s", "cores": 1, "kind": "port",
                                   "sample": f"{' + '.join(desc)} of rank 0's batch from the same pre-rolled state, {s_cpu} steps, "
                                             f"1 thread ({tot[1][2]:.1f} s); oracle/ restatement (the reference cannot be built here)",
                                   "lcp_solves_per_s": tot[1][1] / tot[1][2],
                                   "all_cores": {"value": tot[cores][0] / tot[cores][2], "cores": cores,
                                                 "sample": f"4x the envs, {s_cpu} steps ({tot[cores][2]:.1f} s)"}}
            if bounded:
                out["cpu_baseline"]["upper_bound"] = "a sample hit its wall-clock limit and was stopped: its rate enters as (env-steps asked for) / limit, so the values are upper bounds"
        guard.emit(out)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
