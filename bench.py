#!/usr/bin/env python
"""bench.py -- headline benchmark: QP problems/sec, forward + backward, batch 4096, n=100, m=200
(BASELINE.json configs[1], "C2").  One "step" = one pass of the hot path (boundary tensors ->
ingest -> solve -> adjoint -> emit) over one batch of synthetic dense QPs.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--dump-outputs DIR]

* ours      : `value` = device-resident throughput (inputs already in HBM), `e2e` = the same step
              through the reference-facing `_CvxpyLayer.apply` with HOST buffers (H2D + D2H inside
              the timed region).  N > 1: one rank per GPU (torchrun), each rank solves its own
              4096-instance shard (weak scaling), one NCCL gather of solutions + gradients.
* reference : the reference's algorithm on the host cores -- the C oracle (oracle/cone_oracle.c,
              "port": diffcp/SCS are not installable in this image, DESIGN.md) with all threads.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from types import SimpleNamespace

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "QP problems/sec fwd+bwd (batch=4096, n=100, m=200, zero+nonneg cones)"
UNIT = "problems/s"
# Solver settings shared by both arms (SCS defaults for the forward; LSQR rules of diffcp).
SOLVER_ARGS = {"eps": 1e-4, "max_iters": 10000, "lsqr_precond": 2, "adaptive_check": 1}
# DRAM bytes per instance measured by ncu --set full on 296-instance launches (profiles/prof_fwdfast_r1.txt,
# prof_bwdblk_r1b.txt): fwd_fast_kernel 60.54 MB read + 1.28 MB written; bwd_block_kernel 35.15 MB read
# (only the live rows of A are staged) + 9.90 MB written back within the launch (the rest sits in L2).
NCU_DRAM_BYTES_PER_INSTANCE = {"bwd": (35.154432e6 + 9.900288e6) / 296, "fwd": (60.542976e6 + 1.276416e6) / 296}
# Algorithmic HBM bytes per instance (SURVEY.md 8d): fwd reads A,P,b,c + writes x,y,s;
# bwd re-reads data + x,y,s + dx,dy and writes dA,dP,db,dc.
def algo_bytes(n, m, nnzA, nnzP):
    fwd = 8 * (nnzA + nnzP + m + n) + 8 * (n + 2 * m)
    bwd = 8 * (nnzA + nnzP + m + n) + 8 * (n + 2 * m) + 8 * (n + m) + 8 * (nnzA + nnzP + m + n)
    return fwd, bwd


class ClockSampler:
    """Samples SM clocks / throttle reasons DURING the timed region.  Two sources started together: an in-process NVML thread
    (a sample every 5 ms from the first millisecond -- the timed region of the default run is ~150 ms, less than `nvidia-smi`
    sometimes needs to start up) and an `nvidia-smi -lms 100` child as the fallback; `stop()` reports NVML's samples when it has any."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None
        self.nv_sm, self.nv_max, self.nv_mask, self.nv_thread, self.nv_stop = [], None, 0, None, threading.Event()

    def _nvml_loop(self, nv, handle):
        try:
            while not self.nv_stop.is_set():
                self.nv_sm.append(float(nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM)))
                try:
                    self.nv_mask |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(handle))
                except Exception:  # noqa: BLE001
                    pass
                self.nv_stop.wait(0.005)
        except Exception:  # noqa: BLE001  (a failed query ends this source; nvidia-smi remains)
            pass

    def start(self):
        try:
            import pynvml as nv  # noqa: PLC0415

            nv.nvmlInit()
            handle = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.nv_max = float(nv.nvmlDeviceGetMaxClockInfo(handle, nv.NVML_CLOCK_SM))
            self.nv_thread = threading.Thread(target=self._nvml_loop, args=(nv, handle), daemon=True)
            self.nv_thread.start()
        except Exception:  # noqa: BLE001
            self.nv_thread = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        try:
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:  # noqa: BLE001
            pass

    def stop(self) -> dict:
        try:
            self.nv_stop.set()
            if self.nv_thread is not None:
                self.nv_thread.join(timeout=1)
            if self.proc is not None:
                self.proc.terminate()
                try:
                    self.proc.wait(timeout=2)
                except Exception:  # noqa: BLE001
                    self.proc.kill()
            if self.nv_sm:
                bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
                return {"sm_mhz": float(np.median(self.nv_sm)), "sm_max_mhz": self.nv_max,
                        "reasons": [nm for nm in self.NAMES if self.nv_mask & bits[nm]], "samples": len(self.nv_sm), "source": "nvml"}
            if self.proc is None:
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
            rows = list(self.rows)
            sm = [float(r[0]) for r in rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
            mx = [float(r[1]) for r in rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
            reasons = [nm for k, nm in enumerate(self.NAMES) if any(len(r) >= 6 and r[2 + k].lower().startswith("active") for r in rows)]
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                    "reasons": reasons, "samples": len(sm), "source": "nvidia-smi"}
        except Exception as ex:  # noqa: BLE001  (the sampler must never take the bench line down)
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"sampler error: {ex!r}"[:120]], "samples": 0}


CONFIG = "C2"   # BASELINE.json configs[1] is the headline; the others are parity-test cases that can be timed too


def make_workload(batch: int, seed: int):
    from cvxpylayers_b200 import problems as pr

    bt = pr.CONFIGS[CONFIG](B=batch, seed=seed)
    return bt, pr.to_boundary(bt)


def config_block(bt, B: int, world: int, l2: str) -> dict:
    """The `config` object of the JSON line -- identical for both arms so that the driver can tell they ran the same thing."""
    st = bt.structure
    return {"workload": f"{CONFIG} {bt.name}: n={st.n} m={st.m} cones={st.cones.to_dict()}, synthetic, seed = shard index",
            "batch_per_gpu": B, "global_batch": B * world, "parallelism": f"batch-shard x{world}", "l2": l2,
            "solver_args": dict(SOLVER_ARGS)}


def l2_note(st, B: int) -> str:
    nbytes = (st.nnzA + st.m + st.n + 1 + st.nnzP) * B * 8
    return f"inputs ({nbytes / 1e9:.2f} GB/step) vs 126 MB L2" + ("" if nbytes > 130e6 else "; NOT larger than L2 (secondary config, no flush)")


DUMP_BYTES = 60 * 10**6   # --dump-outputs budget (under 64 MB with the .npy headers); beyond it a seeded sample of instances


def dump_outputs(out_dir: str, sol, grads, B: int):
    """Writes what one step of the timed path hands its caller -- the solution (x, y, s, status) and the gradients of the
    boundary tensors (A_eval, q_eval, P_eval) -- as float64 .npy files, for the instances listed in `instances.npy`: all of
    them when that fits DUMP_BYTES, else a sorted sample drawn with a fixed seed, so two builds dump the same instances."""
    import torch

    gA, gq, gP = grads
    per_instance = 8 * (sol.x.shape[1] + sol.y.shape[1] + sol.s.shape[1] + 2 + gA.shape[0] + gq.shape[0] + (gP.shape[0] if gP is not None else 0))
    k = min(B, DUMP_BYTES // per_instance)
    idx = np.arange(B) if k == B else np.sort(np.random.default_rng(0).choice(B, size=k, replace=False))
    it = torch.as_tensor(idx, device=sol.x.device)
    arrays = {"instances": idx, "x": sol.x[it], "y": sol.y[it], "s": sol.s[it], "status": sol.status[it],
              "grad_A_eval": gA[:, it], "grad_q_eval": gq[:, it]}
    if gP is not None:
        arrays["grad_P_eval"] = gP[:, it]
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrays.items():
        v = v.cpu().numpy() if isinstance(v, torch.Tensor) else v
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(v, dtype=np.float64))
    print(f"[bench] outputs of the last timed step ({k} of {B} instances) written to {out_dir}", file=sys.stderr)


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:  # pragma: no cover
        return os.cpu_count() or 1


def cpu_arm(bt, sample: int, steps: int, warmup: int, threads: int = 0, spread: bool = False, repeat: int = 1):
    """Times the oracle (reference algorithm on host cores): forward + adjoint on `sample` instances.
    The thread count is passed explicitly (torchrun exports OMP_NUM_THREADS=1, which would otherwise pin
    the baseline to one core)."""
    from oracle import oracle as orc

    if threads <= 0:
        threads = host_cores()

    st = bt.structure
    sub = bt.select(slice(0, sample))
    rng = np.random.default_rng(123)
    dx, dy = rng.standard_normal((sample, st.n)), rng.standard_normal((sample, st.m))
    args = dict(SOLVER_ARGS)

    def step():
        for _ in range(repeat):
            x, y, s, status, _ = orc.solve_batch(st, sub.A_vals, sub.b, sub.c, sub.P_vals, nthreads=threads, **args)
            orc.vjp_batch(st, sub.A_vals, sub.b, sub.c, x, y, s, dx, dy, sub.P_vals, nthreads=threads, **args)
        return status

    for _ in range(warmup):
        step()
    per_step = []
    t0 = time.perf_counter()
    for _ in range(steps):
        t1 = time.perf_counter()
        status = step()
        per_step.append(1e3 * (time.perf_counter() - t1))
    dt = (time.perf_counter() - t0) / max(steps, 1)
    cores = threads
    if spread:
        return sample * repeat / dt, dt, cores, int((status == 1).sum()), per_step
    return sample * repeat / dt, dt, cores, int((status == 1).sum())


def make_settings_for(solver_args: dict):
    from cvxpylayers_b200.engine import make_settings

    return make_settings({k: v for k, v in solver_args.items() if k != "reuse_setup"})


def fused_param_variant(bt, B: int, dev, solver_args: dict, steps: int, warmup: int) -> dict:
    """End-to-end variant for SURVEY.md 8f.1 / 8f.2: a layer whose PARAMETERS are b and c only -- A and P are constants of the
    problem (the reference's `PA_is_constant` case, interfaces/moreau_if.py:233-241), the same for every instance -- driven through
    `_CvxpyLayerFused` with pinned host tensors.  Only p_stack = [b; c; 1] goes up and only solutions / the parameter gradient come
    down; the parameter -> matrix map runs inside the engine's load stage.  Timed twice: every call sets the problem up from
    scratch (`reuse_setup` off), and with the set-up cached across calls (what the context does by default for this case)."""
    import scipy.sparse as sp
    import torch

    from cvxpylayers_b200 import problems as pr
    from cvxpylayers_b200.interface import B200_ctx, _CvxpyLayerFused

    st = bt.structure
    rng = np.random.default_rng(12345)
    Pv = None if bt.P_vals is None else np.tile(bt.P_vals[:1], (B, 1))
    bs = pr.plant(st, np.tile(bt.A_vals[:1], (B, 1)), Pv, rng, name="shared_A", active_frac=0.2)
    bd = pr.to_boundary(bs)
    nA, nb, n = st.nnzA, bd.A_eval.shape[0] - st.nnzA, st.n
    P1 = nb + n + 1
    A_map = sp.csr_matrix((np.concatenate([bd.A_eval[:nA, 0], np.ones(nb)]),
                           (np.arange(nA + nb), np.concatenate([np.full(nA, P1 - 1), np.arange(nb)]))), shape=(nA + nb, P1))
    q_map = sp.csr_matrix((np.ones(n), (np.arange(n), nb + np.arange(n))), shape=(n + 1, P1))
    P_map = None if bd.P_eval is None else sp.csr_matrix((bd.P_eval[:, 0], (np.arange(bd.P_eval.shape[0]), np.full(bd.P_eval.shape[0], P1 - 1))),
                                                          shape=(bd.P_eval.shape[0], P1))
    p_host = torch.tensor(np.concatenate([bd.A_eval[nA:], bd.q_eval[:n], np.ones((1, B))])).pin_memory()
    g = torch.Generator(device="cpu").manual_seed(7)
    dxh = torch.randn((B, st.n), dtype=torch.float64, generator=g).pin_memory()
    dyh = torch.randn((B, st.m), dtype=torch.float64, generator=g).pin_memory()
    out = {"workload": f"{bt.name}: A and P constant (one copy for the batch), parameters = b ({nb}) and c ({n}) of each of the {B} instances",
           "h2d_bytes_per_step": int((p_host.numel() + dxh.numel() + dyh.numel()) * 8),
           "d2h_bytes_per_step": int((p_host.numel() + B * (st.n + st.m)) * 8), "unit": UNIT}
    pstruct = (st.P_indices, st.P_indptr, (st.n, st.n)) if st.P_indptr is not None else None
    for key, reuse in (("setup_cached", True), ("setup_every_call", False)):
        ctx = B200_ctx(pstruct, (bd.con_indices, bd.con_ptr, bd.shape), bd.dims, options={**solver_args, "reuse_setup": reuse}, device=str(dev))
        ctx.set_param_maps(A_map, q_map, P_map)
        assert ctx.PA_is_constant
        cl = SimpleNamespace(solver_ctx=ctx)

        def step():
            p = p_host.detach().requires_grad_(True)
            primal, dual, _, _ = _CvxpyLayerFused.apply(p, cl, {}, True, None)
            ((primal * dxh).sum() + (dual * dyh).sum()).backward()
            return primal, p.grad

        for _ in range(max(6, warmup + 2)):   # (the first calls allocate the pinned result buffers, cf. the main e2e loop)
            primal, gp = step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            primal, gp = step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        err = float((primal.detach() - torch.tensor(bs.x_star)).abs().max())
        # three more steps taken apart (wall clock, synchronised; medians): where the time of a call goes
        parts = []
        for _ in range(3):
            p = p_host.detach().requires_grad_(True)
            torch.cuda.synchronize(); t0 = time.perf_counter()
            primal, dual, _, _ = _CvxpyLayerFused.apply(p, cl, {}, True, None)
            torch.cuda.synchronize(); t1 = time.perf_counter()
            loss = (primal * dxh).sum() + (dual * dyh).sum()
            t2 = time.perf_counter()
            loss.backward()
            torch.cuda.synchronize(); t3 = time.perf_counter()
            parts.append((t1 - t0, t2 - t1, t3 - t2))
        t0, t1, t2, t3 = 0.0, *np.cumsum(np.median(np.array(parts), axis=0))
        eng = ctx.engine(torch.device(dev))
        A_vals, P_vals, b_, c_ = eng.ingest_params(p_host.to(dev))
        sol = eng.solve(A_vals, b_, c_, P_vals, make_settings_for(solver_args), cache=ctx.setup_cache(eng, torch.device(dev), B, {"reuse_setup": reuse}), reuse=True)
        out[key] = {"value": B / (ms * 1e-3), "ms_per_step": ms, "max_abs_err_vs_planted_x": err,
                    "one_step_wall_ms": {"forward": round(1e3 * (t1 - t0), 2), "loss_on_host": round(1e3 * (t2 - t1), 2), "backward": round(1e3 * (t3 - t2), 2)},
                    "fwd_iters_mean": float(sol.iters.float().mean()), "solved": int((sol.status == 1).sum())}
    return out


def run_reference(a):
    """The reference's algorithm on the host cores over the SAME batch as our arm (all `a.batch` instances per step,
    every host thread, warmed up, threads bound to cores); per-step times are reported so a noisy host shows."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample = a.batch if a.cpu_sample <= 0 or a.cpu_sample >= a.batch or not a.cpu_sample_given else a.cpu_sample
    bt, _ = make_workload(a.batch, seed=0)
    a.cpu_sample = sample
    world = max(int(os.environ.get("WORLD_SIZE", "1")), 1)
    # N > 1: the job's global batch is N shards; the host has no more cores for it, so a step is N passes over a shard
    val, dt, cores, solved, per_step = cpu_arm(bt, sample, a.steps, max(a.warmup, 1), spread=True, repeat=world)
    st = bt.structure
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": config_block(bt, a.batch, world, l2_note(st, a.batch)),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{a.cpu_sample} of the {a.batch} instances of the {CONFIG} batch per step (oracle/cone_oracle.c: the reference's "
                                       "algorithm restated in C, OpenMP over instances like diffcp's thread pool; diffcp/SCS are not installable here)",
                             "ms_per_step_all": [round(v, 1) for v in per_step],
                             "ms_per_step_min_max": [round(min(per_step), 1), round(max(per_step), 1)],
                             "omp_proc_bind": os.environ.get("OMP_PROC_BIND")},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "solved": solved}
    print(json.dumps(line))


def run_ours(a):
    import torch
    import torch.distributed as dist

    from cvxpylayers_b200 import dist as bdist
    from cvxpylayers_b200.engine import make_settings
    from cvxpylayers_b200.interface import B200_ctx, _CvxpyLayer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the engine has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_bound = bdist.bind_to_gpu_numa_node(local) if world > 1 else False   # pinned buffers next to the GPU's PCIe root
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = a.batch
    bt, bd = make_workload(B, seed=rank)
    st = bt.structure
    pstruct = (st.P_indices, st.P_indptr, (st.n, st.n)) if st.P_indptr is not None else None
    ctx = B200_ctx(pstruct, (bd.con_indices, bd.con_ptr, bd.shape), bd.dims, options=dict(SOLVER_ARGS))
    cl_ctx = SimpleNamespace(solver_ctx=ctx)
    eng = ctx.engine(dev)
    settings = make_settings(SOLVER_ARGS)
    f64 = torch.float64
    # host (pinned) boundary tensors and their device-resident copies
    hA = torch.from_numpy(bd.A_eval).pin_memory()
    hq = torch.from_numpy(bd.q_eval).pin_memory()
    hP = torch.from_numpy(bd.P_eval).pin_memory() if bd.P_eval is not None else None
    dA_, dq_, dP_ = hA.to(dev), hq.to(dev), (hP.to(dev) if hP is not None else None)
    g = torch.Generator(device="cpu").manual_seed(7 + rank)
    dxh = torch.randn((B, st.n), dtype=f64, generator=g)
    dyh = torch.randn((B, st.m), dtype=f64, generator=g)
    dx, dy = dxh.to(dev), dyh.to(dev)
    Btot = B * world
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    kt = {"fwd": 0.0, "bwd": 0.0, "pack": 0.0}

    # Every stage writes into buffers allocated once (the engine's `out=` arguments): no allocator call -- and so no
    # cudaMalloc / cudaFree, which one run in five otherwise slipped between two event records -- inside the timed region.
    nb_aug = hA.shape[0]
    dbuf = dict(inp=(torch.empty((B, st.nnzA), dtype=f64, device=dev), torch.empty((B, st.nnzP), dtype=f64, device=dev) if st.nnzP else None,
                     torch.empty((B, st.m), dtype=f64, device=dev), torch.empty((B, st.n), dtype=f64, device=dev)),
                sol=eng.alloc_solution(B),
                g=(torch.empty((B, st.nnzA), dtype=f64, device=dev), torch.empty((B, st.nnzP), dtype=f64, device=dev) if st.nnzP else None,
                   torch.empty((B, st.m), dtype=f64, device=dev), torch.empty((B, st.n), dtype=f64, device=dev), torch.empty(B, dtype=torch.int32, device=dev)),
                ev=(torch.empty((nb_aug, B), dtype=f64, device=dev), torch.empty((st.n + 1, B), dtype=f64, device=dev),
                    torch.empty((dP_.shape[0], B), dtype=f64, device=dev) if (st.nnzP and dP_ is not None) else None))

    def step_device(timed: bool):
        e = [ev() for _ in range(5)] if timed else None
        if timed: e[0].record()
        A_vals, P_vals, b, c = eng.ingest(dA_, dq_, dP_, out=dbuf["inp"])
        if timed: e[1].record()
        sol = eng.solve(A_vals, b, c, P_vals, settings, out=dbuf["sol"])
        if timed: e[2].record()
        gA, gP, gb, gc, its = eng.vjp(A_vals, b, c, sol.x, sol.y, sol.s, dx, dy, P_vals, settings, out=dbuf["g"])
        if timed: e[3].record()
        gA_eval, gq_eval, gP_eval = eng.emit(gA, gP, gb, gc, out=dbuf["ev"])
        if timed: e[4].record()
        return sol, its, e

    # ---- sharded batch (N > 1): two-stream chunk pipeline, each chunk's results pushed to rank 0 behind the next chunk ----
    # The path has no data-path collective; its one exchange (solutions + gradient blocks onto the rank that owns the
    # autograd graph, SURVEY.md 8e) runs peer-to-peer on the copy engines while the next chunk solves.
    from cvxpylayers_b200.engine import Solution  # noqa: E402

    nnz_aug = hA.shape[0]
    offA = 0
    offq = offA + nnz_aug * B * 8
    offP = offq + (st.n + 1) * B * 8
    offx = offP + st.nnzP * B * 8
    offy = offx + B * st.n * 8
    slot_bytes = offy + B * st.m * 8
    xchg = bdist.PeerExchange(eng.lib, dev, slot_bytes) if world > 1 else None
    if world > 1:
        bufs = dict(A_vals=torch.empty((B, st.nnzA), dtype=f64, device=dev), b=torch.empty((B, st.m), dtype=f64, device=dev),
                    c=torch.empty((B, st.n), dtype=f64, device=dev), P_vals=torch.empty((B, st.nnzP), dtype=f64, device=dev) if st.nnzP else None,
                    sol=eng.alloc_solution(B), gA=torch.empty((B, st.nnzA), dtype=f64, device=dev), gb=torch.empty((B, st.m), dtype=f64, device=dev),
                    gc=torch.empty((B, st.n), dtype=f64, device=dev), gP=torch.empty((B, st.nnzP), dtype=f64, device=dev) if st.nnzP else None,
                    its=torch.empty(B, dtype=torch.int32, device=dev), gA_eval=torch.empty((nnz_aug, B), dtype=f64, device=dev),
                    gq_eval=torch.empty((st.n + 1, B), dtype=f64, device=dev), gP_eval=torch.empty((st.nnzP, B), dtype=f64, device=dev) if st.nnzP else None)
        side = [torch.cuda.Stream(dev), torch.cuda.Stream(dev)]
        copy_stream = torch.cuda.Stream(dev)
        chunk_events, recv_bufs = {}, {}

    def chunk_list(Bs: int, chunk: int):
        """Full chunks first, then a tapered tail (half, quarter, quarter of a chunk, never below 256): the only transfer that
        cannot hide behind a later chunk's solve is the last one, so the last chunk is kept small."""
        sizes, rem = [], Bs
        while rem > chunk:
            sizes.append(chunk); rem -= chunk
        if world > 1 and rem >= 1024:
            sizes += [rem // 2, rem // 4, rem - rem // 2 - rem // 4]
        elif world > 1 and rem >= 512:
            sizes += [rem // 2, rem - rem // 2]
        elif rem > 0:
            sizes.append(rem)
        out, lo = [], 0
        for sz in sizes:
            out.append((lo, lo + sz)); lo += sz
        return out

    def step_sharded(Bs: int, chunk: int):
        """One step over instances [0, Bs) of this rank's shard."""
        u = bufs
        cur = torch.cuda.current_stream(dev)
        for s_ in side:
            s_.wait_stream(cur)
        copy_stream.wait_stream(cur)
        sl = lambda t_, lo, hi: None if t_ is None else t_[lo:hi]  # noqa: E731
        for k, (lo, hi) in enumerate(chunk_list(Bs, chunk)):
            with torch.cuda.stream(side[k % 2]):
                eng.ingest_cols(dA_, dq_, dP_, lo, hi, out=(u["A_vals"][lo:hi], sl(u["P_vals"], lo, hi), u["b"][lo:hi], u["c"][lo:hi]))
                so = u["sol"]
                eng.solve(u["A_vals"][lo:hi], u["b"][lo:hi], u["c"][lo:hi], sl(u["P_vals"], lo, hi), settings,
                          out=Solution(so.x[lo:hi], so.y[lo:hi], so.s[lo:hi], so.status[lo:hi], so.iters[lo:hi], so.resid[lo:hi]))
                eng.vjp(u["A_vals"][lo:hi], u["b"][lo:hi], u["c"][lo:hi], so.x[lo:hi], so.y[lo:hi], so.s[lo:hi], dx[lo:hi], dy[lo:hi],
                        sl(u["P_vals"], lo, hi), settings, out=(u["gA"][lo:hi], sl(u["gP"], lo, hi), u["gb"][lo:hi], u["gc"][lo:hi], u["its"][lo:hi]))
                eng.emit_cols(u["gA"][lo:hi], sl(u["gP"], lo, hi), u["gb"][lo:hi], u["gc"][lo:hi], lo, hi, out=(u["gA_eval"], u["gq_eval"], u["gP_eval"]))
                evk = chunk_events.setdefault(k, torch.cuda.Event())
                evk.record()
            copy_stream.wait_event(evk)
            if xchg.p2p:
                w8 = (hi - lo) * 8
                xchg.push(u["gA_eval"][:, lo:hi], offA + lo * 8, copy_stream, rows=nnz_aug, width_bytes=w8, dpitch=B * 8, spitch=B * 8)
                xchg.push(u["gq_eval"][:, lo:hi], offq + lo * 8, copy_stream, rows=st.n + 1, width_bytes=w8, dpitch=B * 8, spitch=B * 8)
                if st.nnzP:
                    xchg.push(u["gP_eval"][:, lo:hi], offP + lo * 8, copy_stream, rows=st.nnzP, width_bytes=w8, dpitch=B * 8, spitch=B * 8)
                xchg.push(so.x[lo:hi], offx + lo * st.n * 8, copy_stream)
                xchg.push(so.y[lo:hi], offy + lo * st.m * 8, copy_stream)
        for s_ in side:
            cur.wait_stream(s_)
        cur.wait_stream(copy_stream)
        if not xchg.p2p:   # no peer mapping: one NCCL gather per tensor (no transposes, no concatenation afterwards)
            for t_ in (u["gA_eval"], u["gq_eval"], u["gP_eval"], u["sol"].x, u["sol"].y):
                if t_ is None:
                    continue
                if rank == 0:
                    dist.gather(t_, recv_bufs.setdefault(id(t_), [torch.empty_like(t_) for _ in range(world)]), dst=0)
                else:
                    dist.gather(t_, None, dst=0)
        return u["sol"], u["its"]

    def step_e2e(pageable: bool = False):
        srcA, srcq, srcP = (pA, pq, pP) if pageable else (hA, hq, hP)
        A = srcA.detach().requires_grad_(True)
        q = srcq.detach().requires_grad_(True)
        P = srcP.detach().requires_grad_(True) if srcP is not None else None
        t0 = time.perf_counter()
        primal, dual, _, _ = _CvxpyLayer.apply(P, q, A, cl_ctx, {}, True, None)
        t1 = time.perf_counter()
        loss = (primal * dxh).sum() + (dual * dyh).sum()
        loss.backward()
        t2 = time.perf_counter()
        if os.environ.get("BENCH_E2E_BREAKDOWN"):
            print(f"[e2e] forward {1e3 * (t1 - t0):.1f} ms, loss+backward {1e3 * (t2 - t1):.1f} ms", file=sys.stderr)
        return float(loss.detach()), A.grad, q.grad, (P.grad if P is not None else None)

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing ----
    # per-kernel times (and the N = 1 step): the plain one-launch-per-stage sequence
    for _ in range(a.warmup):
        step_device(False)
    sync()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = eng.launch_count()
    t_start, t_end = ev(), ev()
    evs = []
    t_start.record()
    for _ in range(a.steps):
        sol, its, e = step_device(True)
        evs.append(e)
    t_end.record()
    sync()
    if world == 1:
        clocks = sampler.stop()
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, sol, dbuf["ev"], B)
    launches = eng.launch_count() - l0
    ms_total = t_start.elapsed_time(t_end)
    for e in evs:
        kt["pack"] += e[0].elapsed_time(e[1]) + e[3].elapsed_time(e[4])
        kt["fwd"] += e[1].elapsed_time(e[2])
        kt["bwd"] += e[2].elapsed_time(e[3])
    for k in kt:
        kt[k] /= a.steps
    ms_step = ms_total / a.steps
    strong = None
    if world > 1:
        def timed_sharded(Bs, chunk):
            for _ in range(a.warmup):
                step_sharded(Bs, chunk)
            sync()
            lA = eng.launch_count()
            t0_, t1_ = ev(), ev()
            t0_.record()
            for _ in range(a.steps):
                sol_, its_ = step_sharded(Bs, chunk)
            t1_.record()
            sync()
            tt = torch.tensor([t0_.elapsed_time(t1_) / a.steps], dtype=f64, device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt), sol_, its_, eng.launch_count() - lA
        ms_step, sol, its, launches = timed_sharded(B, a.chunk)  # weak scaling: every rank its own B instances
        clocks = sampler.stop()
        if a.dump_outputs and rank == 0:   # rank 0's own shard
            dump_outputs(a.dump_outputs, sol, (bufs["gA_eval"], bufs["gq_eval"], bufs["gP_eval"]), B)
        Bs = max(1, B // world)                                  # strong scaling: the BASELINE batch split over the ranks
        ms_strong, _, _, _ = timed_sharded(Bs, a.chunk)
        strong = {"global_batch": Bs * world, "batch_per_gpu": Bs, "ms_per_step": ms_strong, "value": Bs * world / (ms_strong * 1e-3), "unit": UNIT,
                  "chunks_per_gpu": len(chunk_list(Bs, a.chunk)),
                  "note": f"{Bs} instances per GPU = {Bs / 148:.2f} waves of one CTA per SM: wave quantisation and the fixed per-launch costs bound strong scaling"}
        if a.verify_exchange:
            # every slot of rank 0's buffer against an NCCL gather of the same tensors
            ok = True
            for name_, t_, off_ in (("gA_eval", bufs["gA_eval"], offA), ("gq_eval", bufs["gq_eval"], offq), ("x", bufs["sol"].x, offx), ("y", bufs["sol"].y, offy)):
                recv = [torch.empty_like(t_) for _ in range(world)] if rank == 0 else None
                dist.gather(t_.contiguous(), recv, dst=0)
                if rank == 0 and xchg.p2p:
                    for r_ in range(world):
                        got = xchg.read(r_, off_, torch.empty_like(t_))
                        torch.cuda.synchronize()
                        # (the strong-scaling pass overwrote the first Bs instances of every shard: same data, same values)
                        ok = ok and bool(torch.equal(got, recv[r_]))
            if rank == 0:
                print(f"[bench] exchange verified against NCCL gather: {ok} (p2p={xchg.p2p})", file=sys.stderr)
                assert ok
    status = sol.status.cpu().numpy()
    iters = sol.iters.cpu().numpy()
    lits = its.cpu().numpy()
    n_fallback = eng.fallback_count()   # block solver -> equilibrated LSQR fallbacks of the last backward (-1: block solver not in use)

    # ---- end-to-end through the reference-facing call with HOST buffers ----
    # Warm-up with the same object lifetimes as the timed loop.  The first two calls pay ~360 ms each for the pinned
    # result buffers (two generations are alive at a time); at least three steady steps follow them before timing.
    e2e_warm = max(5, a.warmup + 2)
    for _ in range(e2e_warm):
        loss_val, gAh, gqh, gPh = step_e2e()
    sync()
    e0, e1 = ev(), ev()
    n_e2e = a.steps
    per_step = []
    e0.record()
    for _ in range(n_e2e):
        tw = time.perf_counter()
        loss_val, gAh, gqh, gPh = step_e2e()
        per_step.append(1e3 * (time.perf_counter() - tw))
    e1.record()
    sync()
    print("[bench] e2e wall ms per step: " + ", ".join(f"{v:.1f}" for v in per_step), file=sys.stderr)
    ms_e2e = e0.elapsed_time(e1) / n_e2e
    if world > 1:
        tt = torch.tensor([ms_e2e], dtype=f64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_e2e = float(tt)
    # the same call with PAGEABLE host tensors -- what an unmodified reference layer hands over on CPU (its sparse products
    # return torch.from_numpy arrays, torch/cvxpylayer.py:21-24): no two-stream pipeline, staged copies (ADVICE r1)
    e2e_pageable = None
    if world == 1 and CONFIG == "C2":
        pA, pq, pP = hA.clone(), hq.clone(), (hP.clone() if hP is not None else None)   # clone() of a pinned tensor is pageable
        assert not pA.is_pinned()
        for _ in range(3):
            step_e2e(True)
        sync()
        tw = time.perf_counter()
        for _ in range(a.steps):
            step_e2e(True)
        sync()
        e2e_pageable = {"value": Btot / ((time.perf_counter() - tw) / a.steps), "unit": UNIT, "steps": a.steps,
                        "note": "pageable host inputs (the reference's CPU tensors): batch slices gathered into a ring of pinned staging buffers by a background thread, then the same two-stream pipeline"}
        del pA, pq, pP
    # f1 + f2 in one number: only parameters cross PCIe, the matrices are constants of the layer
    e2e_fused = None
    if world == 1 and CONFIG == "C2" and rank == 0:
        try:
            e2e_fused = fused_param_variant(bt, B, dev, SOLVER_ARGS, a.steps, a.warmup)
        except Exception as ex:  # noqa: BLE001  (a secondary measurement must not take the line down)
            e2e_fused = {"error": repr(ex)[:300]}
    npel = hP.numel() if hP is not None else 0
    h2d = (hA.numel() + hq.numel() + npel + dxh.numel() + dyh.numel()) * 8
    d2h = (gAh.numel() + gqh.numel() + npel + B * (st.n + st.m)) * 8

    if rank == 0:
        fwd_b, bwd_b = algo_bytes(st.n, st.m, st.nnzA, st.nnzP)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:  # noqa: BLE001
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        dom = "bwd" if kt["bwd"] >= kt["fwd"] else "fwd"
        dom_bytes = (bwd_b if dom == "bwd" else fwd_b) * B
        ach = dom_bytes / (kt[dom] * 1e-3) / 1e9
        cpu = None
        if world == 1 and a.cpu_sample > 0:
            ns = min(a.cpu_sample, B)
            if CONFIG == "C4":   # the oracle's dense 1000 x 1000 factor makes an instance a multi-second job per core
                ns = min(ns, 128)
            v, dtc, cores, solved_c, per = cpu_arm(bt, ns, 1 if CONFIG == "C4" else 2, 0 if CONFIG == "C4" else 1, spread=True)
            cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": f"first {ns} instances of the same batch, {0 if CONFIG == 'C4' else 1} warm-up + {1 if CONFIG == 'C4' else 2} timed passes ({dtc:.2f} s each), oracle/cone_oracle.c with OpenMP over instances",
                   "ms_per_pass": [round(x, 1) for x in per]}
        info = eng.kernel_info()
        line = {"metric": METRIC, "value": Btot / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": a.steps,
                "warmup": a.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config_block(bt, B, world, l2_note(st, B)),
                # value = mean over exactly `steps` timed steps (the contract's definition).  The per-step wall times and
                # their median are diagnostics only: on shared boxes single steps sometimes take 2x (profiles/README.md).
                "e2e": {"value": Btot / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e,
                        "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "warmup_steps": e2e_warm,
                        "diagnostic_wall_ms_per_step": [round(v, 1) for v in per_step],
                        "diagnostic_wall_ms_median": round(float(np.median(per_step)), 2),
                        "inputs": "pinned host tensors", **({"pageable_inputs": e2e_pageable} if e2e_pageable else {}),
                        **({"fused_params": e2e_fused} if e2e_fused else {})},
                "gpu_launches": int(launches),
                **({"strong_scaling": strong, "exchange": {"kind": "peer-to-peer copy engines (CUDA IPC over NVLink), chunked behind the solve" if xchg.p2p else "NCCL gather into preallocated slots",
                                                          "bytes_per_rank": int(slot_bytes), "chunk": a.chunk, "numa_bound": bool(numa_bound)}} if world > 1 else {}),
                "roofline": {"bound": "hbm", "kernel": eng.path_info()[dom], "achieved": ach, "peak": peak, "unit": "GB/s",
                             "frac": ach / peak, "traffic": (NCU_DRAM_BYTES_PER_INSTANCE.get(dom, 0) * B / 1e9 or None) if CONFIG == "C2" else None,
                             "traffic_unit": "GB per launch (ncu dram__bytes_read+write per instance, profiles/prof_*_r1*.txt, x B)",
                             "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s",
                             "note": "on-chip iterative solve: HBM is touched once in/out per instance, the loop runs in shared memory"},
                "kernel_ms": {k: round(v, 3) for k, v in kt.items()},
                "kernel_geometry": info, "kernel_paths": eng.path_info(),
                "solver": {"solved": int((status == 1).sum()), "of": int(status.size), "fwd_iters_mean": float(iters.mean()),
                           "fwd_iters_max": int(iters.max()), "lsqr_iters_mean": float(lits.mean()), "lsqr_iters_max": int(lits.max()),
                           "lsqr_fallback": n_fallback, "lsqr_fallback_of": int(lits.size)},
                "clocks": clocks}
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=5)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--batch", type=int, default=0, help="instances per GPU (default: the BASELINE.json batch of the config)")
    p.add_argument("--cpu-sample", type=int, default=None,
                   help="instances per CPU pass (default: 2048 for the cpu_baseline leg of our arm, the whole batch for --impl reference)")
    p.add_argument("--config", default="C2", choices=["C1", "C2", "C2SOC", "C3", "C4", "C5", "C5S", "EXP"],
                   help="workload (default: the headline C2; others are secondary measurements)")
    p.add_argument("--chunk", type=int, default=1024, help="N > 1: instances per pipeline chunk (results of a chunk travel to rank 0 behind the next chunk's solve)")
    p.add_argument("--verify-exchange", action="store_true", help="N > 1: check rank 0's gathered buffer against an NCCL gather")
    p.add_argument("--set", action="append", default=[], metavar="KEY=VALUE",
                   help="override a solver argument for both arms, e.g. --set acceleration_lookback=0")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write the solution and gradients of the last timed step as DIR/<name>.npy (float64, at most 64 MB)")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    a.cpu_sample_given = a.cpu_sample is not None
    if a.cpu_sample is None:
        a.cpu_sample = 2048
    global CONFIG, METRIC
    CONFIG = a.config
    for kv in a.set:
        k, v = kv.split("=", 1)
        SOLVER_ARGS[k] = float(v) if ("." in v or "e" in v.lower()) else int(v)
    if a.batch <= 0:
        a.batch = {"C1": 4096, "C2": 4096, "C2SOC": 1024, "C3": 2048, "C4": 512, "C5": 256, "C5S": 256, "EXP": 1024}[CONFIG]
    if CONFIG != "C2":
        METRIC = f"problems/sec fwd+bwd, BASELINE config {CONFIG} (secondary measurement)"
        a.cpu_sample = min(a.cpu_sample, a.batch)
        if CONFIG in ("C4", "C2SOC"):   # no quadratic term for the block factorisation; LPs need thousands of iterations
            SOLVER_ARGS.update({"lsqr_precond": 1, "max_iters": 100000})
    # The contract is ONE JSON line on stdout.  Libraries write there behind Python's back (NCCL prints its version
    # banner on fd 1 when NCCL_DEBUG is set), so fd 1 points at stderr while the run is in progress and the
    # result line is written to the saved descriptor by the print() calls below via sys.stdout.
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(saved, "w", buffering=1)
    if a.impl == "reference":
        # bind the OpenMP team to cores before libgomp initialises (the oracle is the only OpenMP user of this arm)
        os.environ.setdefault("OMP_PROC_BIND", "spread")
        os.environ.setdefault("OMP_PLACES", "threads")
        run_reference(a)
    else:
        run_ours(a)
    sys.stdout.flush()


if __name__ == "__main__":
    main()
