#!/usr/bin/env python3
"""bench.py -- the BASELINE.json headline metric: Panda 7-DOF fkine+jacob0 evaluations/s at
batch 1M (configs[1]: Panda ETS, fp64, seed 0, q ~ U(-pi, pi), 1M rows per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]   # this repo's CUDA path
    python bench.py --impl reference [--gpus N] [--steps K] [--warmup W]   # the reference's CPU path

--dump-outputs DIR writes what the last timed step returned (T and J) for a fixed, seeded sample of
DUMP_ROWS rows as DIR/T.npy and DIR/J.npy (float64, rank 0's shard), so that two builds run with the
same arguments can be compared output for output.

A "step" is one pass of the hot path over one 1M-row batch: ONE launch of the fused
fkine+jacob0 kernel (b2k_fkine_jacob0 through the C ABI).  Rows are sharded over ranks with no
data-path collective (weak scaling: every rank evaluates its own 1M rows per step).

Timing: W warm-up steps, then exactly K steps bracketed by barrier + synchronize, CUDA events on
the launching stream, MAX over ranks.  Inputs are resident in HBM; four distinct q batches
(4 x 56 MB) are rotated and every step writes 464 MB, so nothing is served from the 126 MB L2.

Extra objects in the JSON line (see DESIGN.md "Measurement"):
  roofline      algorithmic bytes (520 B/eval, SURVEY 8d) / average kernel time vs MEASURED_PEAKS hbm_gbs
  step_ms       median / min / max of K individually timed steps (a second pass, outside `value`)
  cpu_baseline  the reference's own fknm (oracle/_ref, built from /root/reference) on the host cores,
                bounded sample, rank 0 at N=1 only; `effective_cores` = all-core / single-core throughput
  e2e           same metric through the public API with pinned HOST buffers (H2D + kernel + D2H);
                e2e.pageable = the same with the caller's q in ordinary (pageable) numpy memory
  configs       the other BASELINE.json configs, each device-timed with roofline, cpu_baseline and a parity
                record against the reference on a sampled subset: rne_puma_f64_1M (configs[2]),
                ik_lm_panda_f32_100k_* (configs[3], both protocols of SURVEY 8d), fkj_ur10_f32_1M (configs[4]
                per-GPU shard; at N > 1 it runs on every rank with seed 3 + rank: fkj_ur10_f32_sharded)
  gather        (N > 1) NCCL reassembly of the UR10 result shards, outside the metric: one all-gather of the
                packed (T|J) buffer and a gather to rank 0, achieved GB/s into a rank against 900 GB/s
  clocks        SM clocks / throttle reasons sampled through NVML during the timed region
  gpu_launches  kernels this library launched inside the timed region
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

ROWS_PER_GPU = 1_000_000
IK_ROWS = 100_000
N_JOINTS = 7
BYTES_PER_EVAL = (7 + 16 + 42) * 8  # SURVEY 8d: q + T + J0, fp64
METRIC = "Panda 7-DOF fkine+jacob0 evals/sec @ batch 1M"
WORKLOAD = "panda_ets_fkine_jacob0_f64_batch1M"
NVLINK_GBS = 900.0  # nominal NVLink 5 bandwidth per direction per GPU (B200_PROFILING.md)
PARITY_ROWS = 4096
IK_PARITY_ROWS = 1024
DUMP_ROWS = 65536  # --dump-outputs sample: 65536 x (16 + 42) x 8 B = 30 MB
IK_PROTOCOLS = {  # SURVEY 8d config 4: the notebook protocol and the API default
    "ik_lm_panda_f32_100k_chan0.1": dict(k=0.1, jl=False),
    "ik_lm_panda_f32_100k_chan1.0_jl": dict(k=1.0, jl=True),
}


def make_q(seed, rows=ROWS_PER_GPU, n=N_JOINTS):
    return np.random.default_rng(seed).uniform(-np.pi, np.pi, (rows, n))


def make_config(world):
    """The workload description, identical for both arms (the driver compares them)."""
    return {"workload": WORKLOAD, "rows_per_gpu": ROWS_PER_GPU, "global_batch": ROWS_PER_GPU * world,
            "parallelism": f"rows sharded over {world} rank(s), no data-path collective",
            "l2": "4 distinct 56 MB q batches rotated + 464 MB written per step (> 126 MB L2)"}


# ------------------------------------------------------------------ parity-sample inputs (shared by both legs)
PUMA_QLIM = np.deg2rad(np.array([[-160, 160], [-110, 110], [-135, 135], [-266, 266], [-100, 100], [-266, 266]], float)).T


def rne_inputs(seed, rows):
    """SURVEY 8d config 3: q ~ U(qlim) (reference Puma560.py:112-177), qd, qdd ~ N(0,1), exact zeros in a tail
    block of qd so the Coulomb `qd == 0` branch (ne.c:487-490) is exercised."""
    rng = np.random.default_rng(seed)
    q = rng.uniform(PUMA_QLIM[0], PUMA_QLIM[1], (rows, 6))
    qd = rng.normal(size=(rows, 6))
    qdd = rng.normal(size=(rows, 6))
    qd[-max(1, rows // 64):] = 0.0
    return q, qd, qdd


def ik_parity_inputs():
    rng = np.random.default_rng(22)
    qt = rng.uniform(-np.pi, np.pi, (IK_PARITY_ROWS, 7))
    q0 = rng.uniform(-np.pi, np.pi, (IK_PARITY_ROWS, 7))
    return qt, q0


# ------------------------------------------------------------------ CPU leg (reference implementation on the host cores)
def cpu_leg(secondary=True):
    """Runs BEFORE CUDA is initialised in this process (the worker pools fork).  Returns the cpu_baseline
    objects and the reference's outputs on the parity samples.  This is the one place bench.py touches oracle/."""
    from oracle import cpu_arm as ca

    out = {"headline": ca.baseline("panda_fkj", seconds=0.12, reps=3), "configs": {}, "refs": {}}
    if not secondary:
        return out
    out["configs"]["rne_puma_f64_1M"] = ca.baseline("puma_rne", seconds=0.3, reps=2)
    out["configs"]["fkj_ur10_f32_1M"] = ca.baseline("ur10_fkj", seconds=0.12, reps=2)
    for name, o in IK_PROTOCOLS.items():
        out["configs"][name] = ca.baseline("panda_ik", opts=o, seconds=0.5, reps=2)
    # reference outputs on the parity samples (same seeded inputs the GPU leg will evaluate)
    Q = make_q(4242, PARITY_ROWS, 7)
    out["refs"]["panda_fkj"] = ca.evaluate("panda_fkj", (Q,))
    Qu = make_q(4243, PARITY_ROWS, 6).astype(np.float32).astype(np.float64)  # the fp32-rounded inputs the GPU sees
    out["refs"]["ur10_fkj"] = ca.evaluate("ur10_fkj", (Qu,))
    out["refs"]["puma_rne"] = ca.evaluate("puma_rne", rne_inputs(4244, PARITY_ROWS))
    qt, q0 = ik_parity_inputs()
    Tep = ca.evaluate("panda_fkj", (qt,))[0]
    for name, o in IK_PROTOCOLS.items():
        out["refs"][name] = (Tep,) + tuple(ca.evaluate("panda_ik", (Tep, q0), dict(o, slimit=1)))
    out["modules_loaded"] = ca.loaded_reference_modules()
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return 0
    from oracle import cpu_arm as ca

    v1 = ca.time_inline("panda_fkj", 100_000, reps=2)  # single core, in this process (maps oracle/_ref/fknm*.so here)
    arm = ca.CpuArm("panda_fkj")
    rows_per_core = 100_000  # ~0.12 s of work per process per step
    for _ in range(args.warmup):
        arm.step(rows_per_core)
    t = 0.0
    for k in range(args.steps):
        t += arm.step(rows_per_core, seed0=1000 + k)
    arm.close()
    total = rows_per_core * arm.cores
    ms = 1e3 * t / args.steps
    value = total / (t / args.steps)
    n_sched, quota = ca.effective_cores()
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "evals/s", "n_gpus": max(args.gpus, world),
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": make_config(max(args.gpus, world)),
        "cpu_baseline": {"value": value, "unit": "evals/s", "cores": arm.cores, "kind": arm.kind,
                         "sample": f"{total} rows per step ({rows_per_core}/process x {arm.cores} processes): "
                                   + ca.DESCRIBE["panda_fkj"],
                         "single_core_value": v1, "effective_cores": round(value / v1, 2),
                         "cgroup_cpu_quota_cores": quota, "modules_loaded": ca.loaded_reference_modules()},
        "e2e": {"value": value, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "reference CPU implementation (fknm built from /root/reference) on the host cores; a step is a "
                "bounded sample of the 1M-row workload",
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------ clocks sampler (NVML)
class ClockSampler(threading.Thread):
    def __init__(self, torch_dev, period=0.002):
        super().__init__(daemon=True)
        self.period = period
        self.samples = []  # (t, sm_mhz, reasons_bitmask)
        self._stop = threading.Event()
        self.h = None
        self.max_mhz = None
        try:
            import pynvml
            import torch

            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(torch_dev).uuid)
            if not uuid.startswith("GPU-"):
                uuid = "GPU-" + uuid
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(torch_dev)
            self.nv = pynvml
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def run(self):
        if self.h is None:
            return
        nv = self.nv
        while not self._stop.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((time.perf_counter(), int(mhz), int(rs)))
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop.set()

    def summary(self, windows):
        """windows: list of (t0, t1) perf_counter intervals during which the GPU ran timed work."""
        names = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
                 0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
                 0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}
        inwin = [s for s in self.samples if any(a <= s[0] <= b for a, b in windows)]
        note = None
        if not inwin and windows:  # timed regions shorter than one sampling period: use the closest samples
            mid = 0.5 * (windows[0][0] + windows[0][1])
            inwin = sorted(self.samples, key=lambda s: abs(s[0] - mid))[:3]
            note = "timed region shorter than the sampling period; nearest samples used"
        if not inwin:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "NVML unavailable"}
        mask = 0
        for s in inwin:
            mask |= s[2]
        reasons = [n for b, n in names.items() if mask & b and n != "gpu_idle"]
        out = {"sm_mhz": float(np.median([s[1] for s in inwin])), "sm_max_mhz": self.max_mhz, "reasons": reasons,
               "samples": len(inwin)}
        if note:
            out["note"] = note
        return out


# ------------------------------------------------------------------ the B200 arm
def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def load_traffic(key=WORKLOAD):
    """dram bytes per launch from the committed ncu --set full capture of that kernel, if any."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(key)
        except Exception:
            return None
    return None


def err_stats(got, ref, atol):
    """max |got - ref| over a sample, and max |got - ref| / |ref| over its entries that are not (analytically)
    zero (|ref| >= 1e-6: entries like cos(pi/2) products come out as +-1e-17 on both sides)."""
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    d = np.abs(got - ref)
    big = np.abs(ref) >= 1e-6
    return float(d.max()), float((d[big] / np.abs(ref[big])).max()) if big.any() else 0.0


def dump_outputs(out_dir, dev, **arrays):
    """Write the same DUMP_ROWS rows (seeded, sorted) of each (ROWS_PER_GPU, ...) device array as out_dir/<name>.npy."""
    import torch

    os.makedirs(out_dir, exist_ok=True)
    rows = np.sort(np.random.default_rng(5).choice(ROWS_PER_GPU, DUMP_ROWS, replace=False))
    idx = torch.from_numpy(rows).to(dev)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.index_select(0, idx).cpu().numpy())


def run_b200(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_leg(secondary=not args.headline_only)  # before CUDA is initialised in this process (the pools fork)

    import torch

    import b2kin as rtb

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = rtb.dist.bind_to_gpu_numa(local)  # CPU affinity + first-touch placement of pinned buffers next to this GPU
    dist = None
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    peak, peak_src = load_peaks()
    L = rtb._lib.lib()
    F32, F64 = rtb._lib.F32, rtb._lib.F64
    stream = torch.cuda.current_stream(dev)
    sp = stream.cuda_stream
    windows = []

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def rank_max(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def time_steps(step, steps, warmup, per_step=False):
        """W warm-up steps, then K steps between CUDA events on the launching stream, barrier + synchronize on
        both sides, max over ranks -> ms per step.  per_step=True: every step individually (a distribution)."""
        for i in range(warmup):
            step(i)
        barrier()
        w0 = time.perf_counter()
        if per_step:
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
            ev[0].record(stream)
            for i in range(steps):
                step(i)
                ev[i + 1].record(stream)
            barrier()
            windows.append((w0, time.perf_counter()))
            return [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(steps):
            step(i)
        e1.record(stream)
        barrier()
        windows.append((w0, time.perf_counter()))
        return rank_max(e0.elapsed_time(e1)) / steps

    sampler = ClockSampler(local)
    sampler.start()
    W = max(args.warmup, 3)

    # ================================================================ headline: Panda ETS fkine+jacob0 fp64
    panda = rtb.models.Panda()
    ets = panda.ets()
    NBUF = 4
    lo, hi = rtb.dist.shard_bounds(ROWS_PER_GPU * world, world, rank)  # this rank's rows of the global batch
    assert hi - lo == ROWS_PER_GPU
    qs = [torch.from_numpy(make_q(1000 * b + rank)).to(dev) for b in range(NBUF)]
    T = torch.empty((ROWS_PER_GPU, 4, 4), dtype=torch.float64, device=dev)
    J = torch.empty((ROWS_PER_GPU, 6, N_JOINTS), dtype=torch.float64, device=dev)
    chain = ets._chain

    def step(i):
        q = qs[i % NBUF]
        rtb._lib.check(L.b2k_fkine_jacob0(chain, F64, q.data_ptr(), ROWS_PER_GPU, N_JOINTS, None, None,
                                          T.data_ptr(), J.data_ptr(), sp))

    n0 = rtb.launch_count()
    ms_step = time_steps(step, args.steps, W)
    launches = rtb.launch_count() - n0 - W
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dev, T=T, J=J)  # before the per-step pass below overwrites T and J
    value = ROWS_PER_GPU * world / (ms_step * 1e-3)
    clocks = sampler.summary(windows[-1:])
    per = time_steps(step, min(args.steps, 200), 0, per_step=True)  # distribution, outside `value`
    step_ms = {"median": float(np.median(per)), "min": float(np.min(per)), "max": float(np.max(per)), "n": len(per),
               "note": "each step between its own pair of events (second pass; the event records add ~1 us per step)"}
    del qs

    configs = {}

    def parity_fkj(e, key, Q, dt, rtol, atol):
        if cpu is None or key not in cpu["refs"]:
            return None
        Tr, Jr = cpu["refs"][key]
        Tg, Jg = e.fkine_jacob0(torch.from_numpy(Q.astype(dt)).to(dev))
        eT, rT = err_stats(Tg.cpu().numpy(), Tr, atol)
        eJ, rJ = err_stats(Jg.cpu().numpy(), Jr, atol)
        ok = bool(np.allclose(Tg.cpu().numpy(), Tr, rtol=rtol, atol=atol) and np.allclose(Jg.cpu().numpy(), Jr, rtol=rtol, atol=atol))
        return {"rows": int(Q.shape[0]), "vs": "reference fknm (ETS_fkine, ETS_jacob0) on the same seeded rows",
                "max_abs_err": max(eT, eJ), "max_rel_err_nonzero_entries": max(rT, rJ), "rtol": rtol, "atol": atol, "pass": ok}

    headline_parity = parity_fkj(ets, "panda_fkj", make_q(4242, PARITY_ROWS, 7), np.float64, 1e-10, 1e-12)

    # ================================================================ the other BASELINE configs
    def roof(bytes_per_row, rows, ms, bound="hbm", note=None, traffic_key=None):
        a = bytes_per_row * rows / (ms * 1e-3) / 1e9
        r = {"bound": bound, "achieved": a, "peak": peak, "unit": "GB/s", "frac": a / peak,
             "traffic": load_traffic(traffic_key) if traffic_key else None,
             "algorithmic_bytes_per_launch": bytes_per_row * rows}
        if note:
            r["note"] = note
        return r

    KS = max(5, min(args.steps, 30))
    if not args.headline_only:
        # ---- config 5 / configs[4]: UR10 DH fkine+jacob0 fp32, 1M rows per GPU, seed 3 + rank
        ur10 = rtb.models.UR10().ets()
        uq = [torch.from_numpy(make_q(3 + rank + 100 * b, ROWS_PER_GPU, 6).astype(np.float32)).to(dev) for b in range(8)]
        # packed result buffer [T | J] so the reassembly is ONE collective (see `gather` below)
        TJ = torch.empty(ROWS_PER_GPU * 52, dtype=torch.float32, device=dev)
        Tu, Ju = TJ[:ROWS_PER_GPU * 16].view(ROWS_PER_GPU, 4, 4), TJ[ROWS_PER_GPU * 16:].view(ROWS_PER_GPU, 6, 6)
        uch = ur10._chain

        def ustep(i):
            rtb._lib.check(L.b2k_fkine_jacob0(uch, F32, uq[i % 8].data_ptr(), ROWS_PER_GPU, 6, None, None, Tu.data_ptr(),
                                              Ju.data_ptr(), sp))

        ms = time_steps(ustep, KS, 3)
        name = "fkj_ur10_f32_1M" if world == 1 else "fkj_ur10_f32_sharded"
        configs[name] = {
            "baseline_config": "configs[4]: UR10 fkine+jacob0 fp32, 1M rows per GPU (8M over 8 GPUs), seed 3 + rank",
            "ms": ms, "value": ROWS_PER_GPU * world / (ms * 1e-3), "unit": "evals/s", "rows": ROWS_PER_GPU * world,
            "dtype": "f32", "steps": KS, "kernel": "k_fkj_fast<float,6,T,J0>",
            "roofline": roof((6 + 16 + 36) * 4, ROWS_PER_GPU, ms),
            "cpu_baseline": cpu["configs"].get("fkj_ur10_f32_1M") if cpu else None,
            "parity": parity_fkj(ur10, "ur10_fkj", make_q(4243, PARITY_ROWS, 6), np.float32, 1e-4, 1e-5),
        }
        if configs[name]["parity"]:
            configs[name]["parity"]["note"] = "fp32 results against the reference's fp64 on the fp32-rounded inputs"

        # ---- reassembly of the shards (outside the metric)
        gather = None
        if dist is not None:
            full = torch.empty(world * TJ.numel(), dtype=torch.float32, device=dev)
            recv = (world - 1) * TJ.numel() * 4

            def ag(i):
                dist.all_gather_into_tensor(full, TJ)

            ag_ms = time_steps(ag, 5, 2)
            del full
            parts = [torch.empty_like(TJ) for _ in range(world)] if rank == 0 else None

            def g0(i):
                dist.gather(TJ, parts, dst=0)

            g_ms = time_steps(g0, 5, 2)
            del parts
            # the same reassembly WITHOUT a collective: every rank's kernel writes its shard straight into rank 0's memory
            # (peer pointer from torch symmetric memory; the pose rows go out as 256-bit stores, the Jacobian tiles as TMA
            # bulk copies -- over NVLink instead of to local HBM).  Root ingress is the bound: (world - 1) shards.
            fused = None
            try:
                if args.no_fused_gather:
                    raise RuntimeError("disabled by --no-fused-gather")
                import torch.distributed._symmetric_memory as symm

                sbuf = symm.empty(world * TJ.numel(), dtype=torch.float32, device=dev)
                hdl = symm.rendezvous(sbuf, dist.group.WORLD)
                slot = int(hdl.buffer_ptrs[0]) + rank * TJ.numel() * 4
                Tp, Jp = slot, slot + ROWS_PER_GPU * 16 * 4

                def fstep(i):
                    rtb._lib.check(L.b2k_fkine_jacob0(uch, F32, uq[i % 8].data_ptr(), ROWS_PER_GPU, 6, None, None, Tp, Jp, sp))

                f_ms = time_steps(fstep, 5, 2)
                # check: rank 0's buffer now holds what an NCCL gather of the local results delivers
                ustep(6)
                fstep(6)
                barrier()
                ref = [torch.empty_like(TJ) for _ in range(world)] if rank == 0 else None
                dist.gather(TJ, ref, dst=0)
                same = bool(torch.equal(sbuf.view(world, -1), torch.stack(ref))) if rank == 0 else None
                fused = {"ms": f_ms, "GBps_into_root": recv / (f_ms * 1e-3) / 1e9, "frac_of_900GBps": recv / (f_ms * 1e-3) / 1e9 / NVLINK_GBS,
                         "identical_to_nccl_gather": same,
                         "how": "k_fkj_fast<float,6> launched with T / J pointing into rank 0's symmetric-memory buffer"}
                del sbuf
            except Exception as e:  # symmetric memory unavailable on this box / build
                fused = {"unavailable": repr(e)[:300]}
            gather = {
                "what": "UR10 fp32 result shards, packed [T | J] per rank: one NCCL all-gather; a gather to rank 0; and the kernel "
                        "writing its shard directly into rank 0's memory over NVLink (no collective)",
                "bytes_per_rank_shard": TJ.numel() * 4, "bytes_received_per_rank": recv,
                "all_gather_ms": ag_ms, "gather_to_root_ms": g_ms,
                "GBps": recv / (ag_ms * 1e-3) / 1e9, "frac_of_900GBps": recv / (ag_ms * 1e-3) / 1e9 / NVLINK_GBS,
                "gather_to_root_GBps": recv / (g_ms * 1e-3) / 1e9,
                "gather_to_root_frac_of_900GBps": recv / (g_ms * 1e-3) / 1e9 / NVLINK_GBS,
                "fused_store_to_root": fused,
                "kernel_ms": ms, "note": "GB/s = bytes received by one rank / time; the kernel that produced the shard "
                                         "takes kernel_ms, so the reassembly cannot be hidden behind it (SURVEY 8e)",
            }
        del uq, TJ, Tu, Ju

    if not args.headline_only and world == 1:
        # ---- configs[2]: Puma560 DH rne fp64, 1M rows
        puma = rtb.models.Puma560()
        rb = [tuple(torch.from_numpy(a).to(dev) for a in rne_inputs(1 + 10 * b, ROWS_PER_GPU)) for b in range(3)]
        tau = torch.empty((ROWS_PER_GPU, 6), dtype=torch.float64, device=dev)
        puma.rne(rb[0][0][:8], rb[0][1][:8], rb[0][2][:8])  # builds the handle
        g = np.ascontiguousarray(-puma.gravity)
        h = puma._rne_ob

        def rstep(i):
            a, b, c = rb[i % 3]
            rtb._lib.check(L.b2k_rne(h, F64, a.data_ptr(), b.data_ptr(), c.data_ptr(), ROWS_PER_GPU, rtb._lib.dptr(g), None,
                                     tau.data_ptr(), sp))

        ms = time_steps(rstep, KS, 3)
        par = None
        if cpu is not None:
            a, b, c = rne_inputs(4244, PARITY_ROWS)
            tg = puma.rne(torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev), torch.from_numpy(c).to(dev)).cpu().numpy()
            e_abs, e_rel = err_stats(tg, cpu["refs"]["puma_rne"], 1e-10)
            par = {"rows": PARITY_ROWS, "vs": "reference frne.frne on the same seeded rows", "max_abs_err": e_abs,
                   "max_rel_err_nonzero_entries": e_rel, "rtol": 1e-10, "atol": 1e-10,
                   "pass": bool(np.allclose(tg, cpu["refs"]["puma_rne"], rtol=1e-10, atol=1e-10))}
        configs["rne_puma_f64_1M"] = {
            "baseline_config": "configs[2]: Puma560 DHRobot rne (q, qd, qdd) batch 1M fp64",
            "ms": ms, "value": ROWS_PER_GPU / (ms * 1e-3), "unit": "rows/s", "rows": ROWS_PER_GPU, "dtype": "f64",
            "steps": KS, "kernel": rtb.rne_kernel_name(puma) if hasattr(rtb, "rne_kernel_name") else "k_rne<double,6,DH,allrev>",
            "roofline": roof(24 * 8, ROWS_PER_GPU, ms, note="issue-bound (2-cycle FP64 issue + integer / control): DESIGN 3.4", traffic_key="rne_puma_f64_1M"),
            "cpu_baseline": cpu["configs"].get("rne_puma_f64_1M") if cpu else None, "parity": par,
        }
        del rb, tau

        # ---- configs[3]: Panda ikine_LM, 100k reachable targets, fp32, both protocols of SURVEY 8d
        qstar = torch.from_numpy(make_q(2, IK_ROWS, 7)).to(dev)
        Tep64 = ets.eval(qstar)  # reachable by construction: Tep = FK(q*)
        Tep32 = Tep64.float().contiguous()
        qo = torch.empty((IK_ROWS, 7), dtype=torch.float32, device=dev)
        so, io, ro = (torch.empty(IK_ROWS, dtype=torch.int32, device=dev) for _ in range(3))
        Eo = torch.empty(IK_ROWS, dtype=torch.float32, device=dev)
        for name, o in IK_PROTOCOLS.items():
            def istep(i, o=o):
                rtb._lib.check(L.b2k_ik_lm(chain, F32, Tep32.data_ptr(), IK_ROWS, None, 30, 100, 1e-6, int(o["jl"]), None,
                                           float(o["k"]), 0, 5 + i, 0, 1, qo.data_ptr(), so.data_ptr(), io.data_ptr(),
                                           ro.data_ptr(), Eo.data_ptr(), sp))

            n_before = rtb.launch_count()
            ms = time_steps(istep, 5, 2)
            ik_launches = (rtb.launch_count() - n_before) / 7.0
            ok = so.bool()
            Tg = ets.eval(qo.double())
            pose_err = float((Tg - Tep64).abs().amax(dim=(1, 2))[ok].max()) if bool(ok.any()) else None
            par = {"targets": IK_ROWS, "success_rate": float(ok.float().mean()), "mean_iterations": float(io.float().mean()),
                   "max_iterations": int(io.max()), "mean_searches": float(ro.float().mean()), "max_searches": int(ro.max()),
                   "max_residual_E_of_successes": float(Eo[ok].max()) if bool(ok.any()) else None, "tol": 1e-6,
                   "max_pose_err_of_successes": pose_err,
                   "pose_err_note": "max |FK(q) - Tep| (fp64 FK of the fp32 solution) over the successful targets"}
            if cpu is not None:
                Tp, qr, sr_, itr, srr, Er = cpu["refs"][name]
                _, q0 = ik_parity_inputs()
                qg, sg, itg, srg, Eg = ets.ik_LM(torch.from_numpy(Tp).to(dev), q0=torch.from_numpy(q0).to(dev), ilimit=30,
                                                 slimit=1, tol=1e-6, joint_limits=o["jl"], k=o["k"], method="chan")
                sg, itg, qg = sg.cpu().numpy(), itg.cpu().numpy(), qg.cpu().numpy()
                same = (sg == sr_) & (itg == itr)
                both = same & (sr_ == 1)
                par["counters_vs_reference"] = {
                    "targets": IK_PARITY_ROWS, "protocol": "fp64, explicit q0, slimit 1 (deterministic in the reference)",
                    "vs": "reference fknm.IK_LM_c", "identical_success_and_iterations": float(same.mean()),
                    "max_abs_q_diff_where_identical": float(np.abs(qg[both] - qr[both]).max()) if both.any() else None}
            configs[name] = {
                "baseline_config": "configs[3]: Panda ikine_LM fused kernel, 100k random reachable SE(3) targets, fp32",
                "protocol": f"ilimit 30, slimit 100, tol 1e-6, chan lambda={o['k']}, joint-limit check {o['jl']}, random restarts",
                "ms": ms, "value": IK_ROWS / (ms * 1e-3), "unit": "solves/s", "rows": IK_ROWS, "dtype": "f32", "steps": 5,
                "kernel": "k_ik_lm + k_ik_restarts", "launches_per_step": ik_launches,
                "roofline": roof((16 + 7 + 4) * 4, IK_ROWS, ms, bound="latency",
                                 note="serial LM iterations per target: latency / issue bound, HBM fraction reported for completeness",
                                 traffic_key="ik_lm_panda_f32_100k_chan0.1" if name.endswith("chan0.1") else None),
                "cpu_baseline": cpu["configs"].get(name) if cpu else None, "parity": par,
            }
        del qstar, Tep64, Tep32

    # ================================================================ end to end through the public API (host buffers)
    e2e_steps = max(2, min(args.steps, 5))
    qp = [rtb.pinned_empty((ROWS_PER_GPU, N_JOINTS)) for _ in range(2)]
    for b in range(2):
        qp[b][:] = make_q(77 + b + 10 * rank)
    Tp = rtb.pinned_empty((ROWS_PER_GPU, 4, 4))
    Jp = rtb.pinned_empty((ROWS_PER_GPU, 6, N_JOINTS))
    ets.fkine_jacob0_into(qp[0], Tp, Jp)  # warm-up (allocates the pipeline's device staging)
    ets.fkine_jacob0_into(qp[1], Tp, Jp)
    barrier()
    w0 = time.perf_counter()
    for i in range(e2e_steps):
        ets.fkine_jacob0_into(qp[i % 2], Tp, Jp)  # synchronous: results are in Tp / Jp on return
    torch.cuda.synchronize(dev)
    w1 = time.perf_counter()
    e2e_value = ROWS_PER_GPU * world / rank_max((w1 - w0) / e2e_steps)
    checksum = float(Tp[-1, 0, 3]) + float(Jp[-1, 0, 0])
    # the reference's calling convention: q is an ordinary (pageable) numpy array, results are fresh arrays
    qpage = [np.array(qp[b]) for b in range(2)]
    for b in range(2):
        Th, Jh = ets.fkine_jacob0(qpage[b])
    barrier()
    w0 = time.perf_counter()
    for i in range(e2e_steps):
        Th, Jh = ets.fkine_jacob0(qpage[i % 2])
    torch.cuda.synchronize(dev)
    w1 = time.perf_counter()
    e2e_page = ROWS_PER_GPU * world / rank_max((w1 - w0) / e2e_steps)
    page_ok = bool(np.array_equal(Th, Tp) and np.array_equal(Jh, Jp))  # both loops ended on the same q batch
    sampler.stop()

    if rank == 0:
        achieved = BYTES_PER_EVAL * ROWS_PER_GPU / (ms_step * 1e-3) / 1e9
        hb = cpu["headline"] if cpu else None
        line = {
            "metric": METRIC, "value": value, "unit": "evals/s", "n_gpus": world, "steps": args.steps,
            "warmup": W, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": make_config(world),
            "kernel": "k_fkj_fast<double,7,T,J0> (1 launch per step)",
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": load_traffic(), "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": BYTES_PER_EVAL * ROWS_PER_GPU},
            "step_ms": step_ms,
            "cpu_baseline": hb,
            "parity": headline_parity,
            "e2e": {"value": e2e_value, "unit": "evals/s", "h2d_bytes_per_step": ROWS_PER_GPU * N_JOINTS * 8 * world,
                    "d2h_bytes_per_step": ROWS_PER_GPU * (16 + 42) * 8 * world, "steps": e2e_steps,
                    "api": "ETS.fkine_jacob0_into(pinned q, T, J) -> b2k_fkine_jacob0_host", "checksum": checksum,
                    "pageable": {"value": e2e_page, "unit": "evals/s",
                                 "api": "ETS.fkine_jacob0(pageable numpy q) -> fresh result arrays (pooled pinned memory)",
                                 "identical_to_pinned_path": page_ok},
                    "numa": numa},
            "clocks": clocks, "gpu_launches": int(launches),
        }
        if configs:
            line["configs"] = configs
        if not args.headline_only and dist is not None and gather is not None:
            line["gather"] = gather
        if cpu and cpu.get("modules_loaded") is not None:
            line["reference_modules_loaded"] = cpu["modules_loaded"]
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--headline-only", action="store_true", help="skip the secondary configs and the gather")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-fused-gather", action="store_true", help="skip the symmetric-memory store-to-root experiment (N>1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write T and J of the last timed step (a seeded row sample) as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
