#!/usr/bin/env python
"""bench.py -- atom-steps/s (energy + forces) of the Allegro hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # this framework
    python bench.py --impl reference --gpus N --steps K ...  # CPU reference arm (oracle port)
    python bench.py --gpus 1 ... --dump-outputs DIR          # also write the last timed step's outputs as DIR/<name>.npy

One "step" = one energy+forces evaluation of the configured model on one synthetic frame
(neighbour list given, built outside the timed region).  N=1 workload: BASELINE.json
configs[1] (c2: 10 976-atom Cu FCC, l_max=2, 2 layers, 64 features, r_max=5.0).
Prints ONE JSON line on rank 0.
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "atom-steps/sec (energy+forces)"
UNIT = "atom-steps/s"


# --------------------------------------------------------------------------------------
# clocks sampling (nvidia-smi during the timed region)
# --------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------
# workload
# --------------------------------------------------------------------------------------
def build_workload(cfg: str, dtype: str, device, scale=None):
    from allegro_b200 import data as D
    from allegro_b200 import systems
    from allegro_b200.model import AllegroModel

    d = systems.make_system(cfg, scale)
    n, e = d[D.POSITIONS_KEY].shape[0], d[D.EDGE_INDEX_KEY].shape[1]
    kw = systems.model_kwargs(cfg, e / n, dtype)
    model = AllegroModel(**kw).to(device)
    data = {k: v.to(device) for k, v in d.items()}
    return model, data, d, kw, n, e


PARITY_TOL = {"float64": 1e-9, "float32": 1e-4, "bfloat16": 1e-3}
DUMP_BUDGET_BYTES = 60_000_000  # --dump-outputs: all arrays together (the .npy headers come on top)


def dump_outputs(outputs, path: str, budget: int = DUMP_BUDGET_BYTES):
    """Write every output as <path>/<name>.npy, float64 as float64 and any other floating type as float32, so that two
    builds can be compared array by array.  Arrays are taken smallest first, each against an even share of the bytes
    of ``budget`` that are still left; one larger than its share keeps a sample of its rows: a fixed-seed random subset
    in ascending row order, the same rows for every run with the same shapes."""
    import numpy as np

    os.makedirs(path, exist_ok=True)
    arrays = {k: v.detach().to("cpu", torch.float64 if v.dtype == torch.float64 else torch.float32) for k, v in outputs.items()}
    left = budget
    for i, (name, t) in enumerate(sorted(arrays.items(), key=lambda kv: (kv[1].numel() * kv[1].element_size(), kv[0]))):
        rows = t.shape[0] if t.dim() else 1
        keep = left // (len(arrays) - i) // max(1, t.numel() // max(1, rows) * t.element_size())
        if rows > keep:
            t = t[torch.randperm(rows, generator=torch.Generator().manual_seed(0))[:keep].sort().values]
        left -= t.numel() * t.element_size()
        np.save(os.path.join(path, f"{name}.npy"), t.numpy())


def parity_check(model, out, d_cpu, kw, dtype: str, n_sample: int = 16):
    """Before anything is timed: energies and forces of the model that is about to be timed, on the frame that is about
    to be timed, against the fp64 CPU oracle on a sub-sample of atoms (strict locality, oracle/subsample.py).  The
    oracle is the CHECKER here; it is never part of a timed region.  Raises if the bar is missed."""
    from allegro_b200 import data as D
    from oracle.model_ref import AllegroOracle
    from oracle.subsample import ball, local_reference

    kwo = dict(kw)
    kwo["model_dtype"] = "float64"
    oracle = AllegroOracle(**kwo)
    oracle.load_state_dict({k: v.detach().double().cpu() for k, v in model.state_dict().items()})
    atoms = ball(d_cpu[D.POSITIONS_KEY], n_sample, seed=7)
    t = time.perf_counter()
    centres, e_ref, f_ref = local_reference(oracle, d_cpu, atoms)
    e = out[D.PER_ATOM_ENERGY_KEY].double().cpu()[centres]
    f = out[D.FORCE_KEY].double().cpu()[atoms]
    err_e = float((e - e_ref).abs().max() / e_ref.abs().max())
    err_f = float((f - f_ref).abs().max() / f_ref.abs().max())
    tol = PARITY_TOL[dtype]
    res = {"vs": "fp64 CPU oracle on a locality sub-sample", "atoms_forces": int(atoms.numel()), "centres_energies": int(centres.numel()),
           "rel_err_E": err_e, "rel_err_F": err_f, "tol": tol, "oracle_s": round(time.perf_counter() - t, 2)}
    if not (err_e < tol and err_f < tol):
        raise AssertionError(f"bench.py: the model about to be timed misses the parity bar: {res}")
    return res


def algorithmic_bytes_per_edge(name: str, core) -> float:
    """Bytes that must cross HBM per edge for each kernel of the current (per-kernel) pipeline
    (DESIGN.md section 4); b = bytes per activation element, 4 = fp32 accumulate-type element."""
    b = {torch.float64: 8, torch.float32: 4, torch.bfloat16: 2}[core.dtype]
    a = 8 if core.dtype == torch.float64 else 4
    U, S, D, nw, L = core.U, core.S, core.D, core.nw, core.L
    kern, _, tag = name.partition("@")
    layer = int(tag.split("L")[1]) if ".L" in tag else None
    if kern == "tp_fwd":
        ly = core.layers[layer]
        vin = (b * nw + a * D) if layer == 0 else b * U * ly["d_in"]
        return vin + 4 + b * U * ly["d_out"]
    if kern == "tp_bwd":
        ly = core.layers[layer]
        vin = (b * nw + a * D) if layer == 0 else b * U * ly["d_in"]
        gin = (b * nw + 2 * a * D) if layer == 0 else b * U * ly["d_in"]
        return vin + 4 + b * U * ly["d_out"] + gin
    if kern == "env_sum":
        return b * nw + a * D
    if kern == "env_bwd":
        return 2 * b * nw + 3 * a * D + 4
    return float("nan")


def run_ours(args, rank: int, world: int):
    from allegro_b200 import _lib
    from allegro_b200 import data as D

    if world > 1:
        return run_ours_multi(args, rank, world)
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(dev)
    cfg = args.config
    from allegro_b200 import systems

    dtype = args.dtype or systems.CONFIGS[cfg]["dtype"]
    model, data, d_cpu, kw, n_atoms, n_edges = build_workload(cfg, dtype, dev)
    K, W = args.steps, args.warmup
    graphed = None
    if not args.no_graph:
        from allegro_b200.graph import GraphedEnergyForces

        graphed = GraphedEnergyForces(model, data)

    def step():
        return graphed() if graphed is not None else model(data)

    def step_eager():
        return model(data)

    for _ in range(W):
        out = step()
    torch.cuda.synchronize()
    parity = None if args.no_parity_check else parity_check(model, out, d_cpu, kw, dtype)
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    # ---- leg 1: inputs resident in HBM, device-timed ----
    _lib.PROF.reset()
    _lib.PROF.enabled = False
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record()
    for _ in range(K):
        out = step()
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / K
    launches = _lib.PROF.launches
    # what a caller of the timed path receives from its last step: the computed arrays, not the inputs echoed back
    # (copied now: the graph's static output buffers are overwritten by the legs below)
    last = {k: v.detach().clone() for k, v in out.items() if k not in data and torch.is_floating_point(v)} if args.dump_outputs else None
    # ---- leg 2: same K steps with per-kernel CUDA events (roofline of the dominant kernel) ----
    _lib.PROF.reset()
    _lib.PROF.enabled = True
    for _ in range(K):
        out = step_eager()
    times = _lib.PROF.times_ms()
    _lib.PROF.enabled = False
    # ---- leg 3: end to end through the public API with HOST buffers ----
    pos_host = d_cpu[D.POSITIONS_KEY].clone().pin_memory()
    f_host = torch.empty(n_atoms, 3, dtype=out[D.FORCE_KEY].dtype).pin_memory()
    e_host = torch.empty(1, 1, dtype=out[D.TOTAL_ENERGY_KEY].dtype).pin_memory()
    data_e2e = dict(data)

    def step_e2e():
        if graphed is not None:
            o = graphed(pos_host)  # H2D of the positions into the graph's static buffer, then replay
        else:
            data_e2e[D.POSITIONS_KEY] = pos_host.to(dev, non_blocking=True)
            o = model(data_e2e)
        f_host.copy_(o[D.FORCE_KEY], non_blocking=True)
        e_host.copy_(o[D.TOTAL_ENERGY_KEY], non_blocking=True)

    for _ in range(2):
        step_e2e()
    torch.cuda.synchronize()
    t0.record()
    for _ in range(K):
        step_e2e()
    t1.record()
    torch.cuda.synchronize()
    ms_e2e = t0.elapsed_time(t1) / K
    clocks = sampler.stop()

    core = model.model.core()
    per_kernel = {k: sum(v) / K for k, v in times.items()}  # ms per step
    kernel_total = sum(per_kernel.values())
    dom = max(per_kernel, key=per_kernel.get)
    # the roofline is quoted for the dominant tensor-product kernel (the path's named hot loop)
    tp_like = {k: v for k, v in per_kernel.items() if k.split("@")[0] in ("tp_fwd", "tp_bwd", "env_sum", "env_bwd")}
    dom_tp = max(tp_like, key=tp_like.get)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    n_l = len(times[dom_tp]) / K
    avg_ms = per_kernel[dom_tp] / n_l
    bpe = algorithmic_bytes_per_edge(dom_tp, core)
    achieved = bpe * n_edges / (avg_ms * 1e-3) / 1e9
    # DRAM traffic of that kernel from the latest committed `ncu --set full` capture (tools/ncu_summary.py writes
    # profiles/ncu_traffic.json: dram__bytes_read.sum + dram__bytes_write.sum per launch, measured at the c2 shapes)
    traffic = traffic_src = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        pat = {"tp_bwd@bwd.L0": "tp_bwd3_kernel", "tp_fwd@fwd.L0": "tp_stream_kernel<float, float, 9, 9, 1, 0,",
               "tp_bwd@bwd.L1": "tp_smem_kernel<float, float, 9, 1,",
               "env_bwd@bwd.L0": "env_bwd_stream_kernel<float, 2,", "env_bwd@bwd.L1": "env_bwd_stream_kernel<float, 2,"}.get(dom_tp)
        if cfg == "c2" and dtype == "float32" and pat:
            for kname, rec in tj["per_kernel"].items():
                if pat in kname:
                    traffic = rec["dram_bytes_per_launch"]
                    traffic_src = f"profiles/{tj['tag']}_ncu_full_summary.md ({tj['source']}: ncu --set full, dram__bytes_read+write per launch)"
    except Exception:
        pass
    roofline = {
        "kernel": dom_tp, "bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
        "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": traffic_src,
        "launches_per_call": int(round(n_l)), "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 (of fallback)",
        "algorithmic_bytes_per_edge": bpe, "avg_launch_ms": round(avg_ms, 5), "share_of_kernel_time": round(per_kernel[dom_tp] / kernel_total, 4),
    }
    res = {
        "metric": METRIC, "value": n_atoms * 1e3 / ms, "unit": UNIT, "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": {"float64": "f64", "float32": "f32", "bfloat16": "bf16"}[dtype], "data": "synthetic",
        "config": {"workload": f"{cfg}: {systems.CONFIGS[cfg]['system']}, {n_atoms} atoms, {n_edges} edges, l_max={kw['l_max']}, "
                               f"n_layers={kw['num_layers']}, S={kw['num_scalar_features']}, U={kw['num_tensor_features']}, r_max={kw['r_max']}",
                   "global_atoms": n_atoms, "parallelism": "1 GPU", "cuda_graph": graphed is not None, "timing": "CUDA events, inputs larger than L2 (per-step working set "
                   f"~{n_edges * 5e3 / 1e9:.1f} GB >> 126 MB L2), neighbour list resident"},
        "ns_per_day_at_1fs": 1e3 / ms * 0.0864,
        "clocks": clocks,
        "e2e": {"value": n_atoms * 1e3 / ms_e2e, "unit": UNIT, "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": pos_host.numel() * pos_host.element_size(),
                "d2h_bytes_per_step": f_host.numel() * f_host.element_size() + e_host.numel() * e_host.element_size()},
        "gpu_launches": launches,
        "parity_check": parity,
        "roofline": roofline,
        "kernels_ms_per_step": {k: round(v, 4) for k, v in sorted(per_kernel.items(), key=lambda kv: -kv[1])},
        "kernel_time_ms_per_step": round(kernel_total, 4),
        "dominant_kernel": dom,
    }
    if not args.no_cpu_baseline:
        res["cpu_baseline"] = cpu_baseline(cfg, steps=3)
    if last is not None:
        dump_outputs(last, args.dump_outputs)
    print(json.dumps(res))


def run_ours_multi(args, rank, world):
    """N>1: weak scaling by spatial domain decomposition (SURVEY 8e).  The c2 crystal is
    replicated `world` times along x; each rank owns one 14x14x14-cell slab (fixed per-GPU
    work) and exchanges a single-r_max halo with its two neighbours every step:
    positions forward, ghost gradients back, one scalar sum (over NVLink peer memory by default, NCCL with --halo nccl).
    At N = 8 the line additionally carries BASELINE configs[3] -- the ~1M-atom water-like box split into 8 slabs -- under
    the key "c4" (measured after the main timed region, guarded by a watchdog so that it can never cost the main line)."""
    import torch.distributed as dist

    local = int(os.environ.get("LOCAL_RANK", rank))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    res = _measure_multi(args, rank, world, dev, args.config, args.steps, args.warmup)
    want_c4 = world == 8 and args.config == "c2" and not args.no_c4 and not args.reps
    if want_c4:
        state = {"printed": False}
        lock = threading.Lock()

        def emit(extra):
            with lock:
                if state["printed"]:
                    return
                state["printed"] = True
                if rank == 0:
                    res["c4"] = extra
                    print(json.dumps(res), flush=True)

        def bail():  # the c4 leg hangs (or takes too long): every rank leaves, rank 0 with the main line
            emit({"error": "c4 leg exceeded its time limit"})
            sys.stdout.flush()
            os._exit(0)

        timer = threading.Timer(float(os.environ.get("AB2_BENCH_C4_LIMIT_S", "420")), bail)
        timer.daemon = True
        timer.start()
        try:
            torch.cuda.empty_cache()
            c4 = _measure_multi(args, rank, world, dev, "c4", min(args.steps, 10), min(args.warmup, 3))
            extra = None
            if rank == 0:
                extra = {k: c4[k] for k in ("value", "unit", "ms_per_step", "scaling", "ns_per_day_at_1fs", "e2e", "gpu_launches")}
                extra["workload"] = c4["config"]["workload"]
                extra["steps"] = c4["steps"]
                extra["halo"] = c4["config"]["halo"]
            emit(extra)
        except Exception as exc:  # noqa: BLE001 -- anything here must not cost the main line
            emit({"error": f"{type(exc).__name__}: {exc}"[:300]})
        timer.cancel()
    elif rank == 0:
        print(json.dumps(res), flush=True)
    sys.stdout.flush()
    sys.stderr.flush()
    # CUDA graphs holding captured NCCL kernels keep the communicator busy: tearing the process group down under them
    # blocks.  Every rank is past its last collective and rank 0 has printed, so leave without running the destructors.
    try:
        torch.cuda.synchronize()
    except Exception:  # noqa: BLE001
        pass
    os._exit(0)


def _measure_multi(args, rank, world, dev, cfg, K, W):
    """One multi-GPU measurement (all ranks call it; rank 0 gets the result dict, the others None)."""
    import torch.distributed as dist

    from allegro_b200 import _lib, systems
    from allegro_b200 import data as D
    from allegro_b200.halo import DistributedAllegro, SlabDecomposition
    from allegro_b200.model import AllegroModel

    dtype = args.dtype or systems.CONFIGS[cfg]["dtype"]
    base = args.reps or {"c1": 2, "c2": 14, "c5": 14, "c3": 46, "c4": 69}[cfg]
    # c4 IS the multi-GPU configuration (BASELINE configs[3]: the 1M-atom water box split into N slabs, fixed total
    # size); every other config is replicated N times along x (fixed per-GPU work, weak scaling)
    strong = cfg == "c4"
    reps = (base, base, base) if strong else (base * world, base, base)
    pos, cell, types = systems.make_positions(cfg, reps)
    n_global = pos.shape[0]
    dec = SlabDecomposition(pos, cell, types, systems.CONFIGS[cfg]["r_max"], rank, world, device=dev)
    n_edges = dec.n_edges
    cnt = torch.tensor([float(n_edges), float(dec.n_owned)], device=dev, dtype=torch.float64)
    dist.all_reduce(cnt)  # one model for the whole frame: the global average neighbour count on every rank
    kw = systems.model_kwargs(cfg, float(cnt[0] / cnt[1]), dtype)
    model = AllegroModel(**kw).to(dev).model  # energy model; forces via the halo-aware runner
    pos_owned = dec.local_positions_from_global(pos)[: dec.n_owned].to(dev)
    dec.to(dev)
    eager = DistributedAllegro(model, dec)
    # halo over NVLink peer memory (kernels only, no NCCL call per step); checked once against the NCCL path on this
    # very frame, and abandoned on every rank if any rank disagrees
    halo_mode = args.halo
    if halo_mode == "p2p":
        from allegro_b200.halo import P2PHalo

        ok = 1
        try:
            p2p = P2PHalo(dec, dev)
            cand = DistributedAllegro(model, dec, p2p=p2p)
            e1, f1, _ = eager(pos_owned)
            e2, f2, _ = cand(pos_owned)
            e3, f3, _ = cand(pos_owned)  # second step: the other mailbox parity
            torch.cuda.synchronize()
            scale = float(f1.abs().max())
            if p2p.error() != 0 or float((f2 - f1).abs().max()) > 1e-5 * scale or float((f3 - f1).abs().max()) > 1e-5 * scale or \
                    abs(float(e2) - float(e1)) > 1e-6 * abs(float(e1)) + 1e-9:
                ok = 0
        except Exception as exc:  # IPC not available, ...
            print(f"[bench] rank {rank}: p2p halo unavailable: {exc}", file=sys.stderr)
            ok = 0
        okt = torch.tensor([ok], device=dev)
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        if int(okt) == 1:
            eager = cand
        else:
            halo_mode = "nccl (p2p self-check failed)"
    for _ in range(W):
        e, f, _ = eager(pos_owned)
    # host-side launch cost of the eager step (wall clock of the Python loop, no sync inside)
    torch.cuda.synchronize()
    dist.barrier()
    tw = time.perf_counter()
    for _ in range(5):
        eager(pos_owned)
    host_ms = (time.perf_counter() - tw) / 5 * 1e3
    torch.cuda.synchronize()
    graphed = False
    runner = eager
    if not args.no_graph:
        from allegro_b200.halo import GraphedDistributedAllegro

        runner = GraphedDistributedAllegro(eager, pos_owned)
        graphed = True
        for _ in range(W):
            e, f, _ = runner(pos_owned)
        torch.cuda.synchronize()
    sampler = ClockSampler(dev.index or 0)
    if rank == 0:
        sampler.start()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    _lib.PROF.reset()
    dist.barrier()
    torch.cuda.synchronize()
    t0.record()
    for _ in range(K):
        e, f, _ = runner(pos_owned)
    t1.record()
    torch.cuda.synchronize()
    dist.barrier()
    ms_t = torch.tensor([t0.elapsed_time(t1) / K], device=dev, dtype=torch.float64)
    dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)
    ms = float(ms_t)
    launches = _lib.PROF.launches
    host_t = torch.tensor([host_ms], device=dev, dtype=torch.float64)
    dist.all_reduce(host_t, op=dist.ReduceOp.MAX)
    # end to end: owned positions from pinned host memory, forces + energy back to the host
    pos_host = pos_owned.cpu().pin_memory()
    f_host = torch.empty(dec.n_owned, 3, dtype=f.dtype).pin_memory()
    e_host = torch.empty(1, dtype=e.dtype).pin_memory()

    def step_e2e():
        p = pos_host.to(dev, non_blocking=True)
        ee, ff, _ = runner(p)  # graphed: p is copied into the static position buffer, then one replay
        f_host.copy_(ff, non_blocking=True)
        e_host.copy_(ee, non_blocking=True)

    step_e2e()
    dist.barrier()
    torch.cuda.synchronize()
    t0.record()
    for _ in range(K):
        step_e2e()
    t1.record()
    torch.cuda.synchronize()
    dist.barrier()
    ms_e = torch.tensor([t0.elapsed_time(t1) / K], device=dev, dtype=torch.float64)
    dist.all_reduce(ms_e, op=dist.ReduceOp.MAX)
    ms_e2e = float(ms_e)
    ghosts = torch.tensor([dec.n_ghost], device=dev)
    dist.all_reduce(ghosts, op=dist.ReduceOp.MAX)
    if rank == 0:
        clocks = sampler.stop()
        res = {
            "metric": METRIC, "value": n_global * 1e3 / ms, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": {"float64": "f64", "float32": "f32", "bfloat16": "bf16"}[dtype], "data": "synthetic",
            "config": {"workload": f"{cfg} " + (f"split into {world} slabs" if strong else f"replicated x{world}") + f" along x: {n_global} atoms, {dec.n_owned} owned + <= {int(ghosts)} ghost atoms and "
                                   f"{n_edges} edges per GPU, l_max={kw['l_max']}, n_layers={kw['num_layers']}, S={kw['num_scalar_features']}, "
                                   f"U={kw['num_tensor_features']}, r_max={kw['r_max']}",
                       "global_atoms": n_global, "parallelism": f"spatial slab decomposition x{world}, ghost-atom halo (positions fwd, gradients rev) "
                       "+ 1 scalar energy sum per step", "halo": halo_mode + (": NVLink peer-memory mailboxes (CUDA IPC), kernels only, inside the CUDA graph"
                                                                              if halo_mode == "p2p" else ": torch.distributed P2P + all_reduce inside the CUDA graph"), "timing": "CUDA events, barrier + synchronize both sides, max over ranks; per-step working set >> L2",
                       "halo_bytes_per_step_per_gpu": dec.halo_bytes_per_step(8),
                       "cuda_graph": graphed, "eager_host_ms_per_step_max": float(host_t),
                       "host_cpus_visible": len(os.sched_getaffinity(0))},
            "ns_per_day_at_1fs": 1e3 / ms * 0.0864,
            "clocks": clocks,
            "e2e": {"value": n_global * 1e3 / ms_e2e, "unit": UNIT, "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": pos_host.numel() * 8 * world, "d2h_bytes_per_step": (f_host.numel() * f_host.element_size() + 8) * world},
            "gpu_launches": launches,
        }
        return res
    return None


# --------------------------------------------------------------------------------------
# CPU reference arm / baseline: the oracle port on the host cores
# --------------------------------------------------------------------------------------
def _host_threads() -> int:
    """CPU threads this process may really use: affinity mask capped by the cgroup CPU quota.  torchrun exports
    OMP_NUM_THREADS=1 to its workers; the CPU arm is a single process (rank 0), so it takes the whole allowance."""
    n = len(os.sched_getaffinity(0))
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return n


def _oracle_setup(cfg: str, scale: int):
    torch.set_num_threads(_host_threads())
    from allegro_b200 import data as D
    from allegro_b200 import systems
    from oracle.model_ref import AllegroOracle

    d = systems.make_system(cfg, scale)
    n, e = d[D.POSITIONS_KEY].shape[0], d[D.EDGE_INDEX_KEY].shape[1]
    kw = systems.model_kwargs(cfg, e / n, "float32")
    return AllegroOracle(**kw), d, n, e, kw


def cpu_baseline(cfg: str, steps: int = 3, scale: int = 4):
    oracle, d, n, e, _ = _oracle_setup(cfg, scale)
    oracle(d)
    t = time.perf_counter()
    for _ in range(steps):
        oracle(d)
    dt = (time.perf_counter() - t) / steps
    return {"value": n / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{cfg} architecture (fp32 eager PyTorch oracle, edge-chunked dense contraction) on a {scale}^3 supercell: "
                      f"{n} atoms, {e} edges, {steps} evaluations of {dt:.2f} s; cost is linear in edges",
            "host_cpus": os.cpu_count()}


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    cfg = args.config
    K, W = args.steps, args.warmup
    scale = 3 if K + W > 60 else 4  # 4^3 cells = 256 atoms / 10.8k edges per step (0.4 s on 16 threads): less threading overhead per edge than 3^3
    oracle, d, n, e, kw = _oracle_setup(cfg, scale)
    for _ in range(max(W, 1)):
        oracle(d)
    t = time.perf_counter()
    for _ in range(K):
        oracle(d)
    dt = (time.perf_counter() - t) / K
    val = n / dt
    from allegro_b200 import systems

    res = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": W,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{cfg}: {systems.CONFIGS[cfg]['system']} architecture l_max={kw['l_max']}, n_layers={kw['num_layers']}, "
                               f"S={kw['num_scalar_features']}, U={kw['num_tensor_features']}; bounded sample {n} atoms / {e} edges per step",
                   "note": "plain-PyTorch restatement of the reference (nequip/e3nn are not installable here), CPU, all host threads"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                         "sample": f"{scale}^3 supercell, {n} atoms, {e} edges per step"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(res))


def run_reference_gpu(args, rank: int, world: int, triton: bool = False):
    """GPU baseline (SURVEY 8d "GPU reference baseline"): the oracle -- a plain-PyTorch restatement of the reference's
    default path, autograd forces -- evaluated on one B200 at the full benchmark size, fp32, eager.  With ``triton``
    every eligible Contracter is replaced by the reference's own TritonContracter (oracle/_ref, staged verbatim from
    /root/reference by oracle/build_ref.py), i.e. the reference's accelerated inference path."""
    if rank != 0:
        return
    from allegro_b200 import data as D
    from allegro_b200 import systems
    from oracle.model_ref import AllegroOracle

    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(dev)
    cfg = args.config
    d = systems.make_system(cfg)
    n, e = d[D.POSITIONS_KEY].shape[0], d[D.EDGE_INDEX_KEY].shape[1]
    kw = systems.model_kwargs(cfg, e / n, "float32")
    oracle = AllegroOracle(**kw)
    swapped = 0
    if triton:
        from oracle import build_ref

        ref = build_ref.load()
        inner = oracle.model if hasattr(oracle, "model") else oracle
        tps = inner.allegro.tps
        for i, tp in enumerate(tps):
            if tp.w3j.dim() != 4:
                continue  # the reference's Triton path only takes [P,I,J,K] tables (_flashallegro.py:315)
            new = ref.TritonContracter(irreps_in1=repr(tp.irreps_in1).replace(" ", ""), irreps_in2=repr(tp.irreps_in2).replace(" ", ""), irreps_out=repr(tp.irreps_out).replace(" ", ""), mul=tp.mul,
                                       instructions=tp.instructions, path_channel_coupling=tp.path_channel_coupling,
                                       scatter_factor=tp.scatter_factor, irrep_normalization=tp.irrep_normalization)
            new.load_state_dict(tp.state_dict())
            tps[i] = new
            swapped += 1
    oracle = oracle.to(dev).eval()
    dd = {k: v.to(dev) for k, v in d.items()}
    dd[D.POSITIONS_KEY] = dd[D.POSITIONS_KEY].float()
    dd[D.CELL_KEY] = dd[D.CELL_KEY].float()
    dd[D.EDGE_CELL_SHIFT_KEY] = dd[D.EDGE_CELL_SHIFT_KEY].float()
    K, W = args.steps, args.warmup
    for _ in range(max(W, 1)):
        out = oracle(dd)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(K):
        out = oracle(dd)
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / K
    res = {"impl": args.impl, "metric": METRIC, "value": n * 1e3 / ms, "unit": UNIT, "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": ms,
           "higher_is_better": True, "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"{cfg}: {n} atoms, {e} edges (full size)", "what": "oracle/ (plain PyTorch restatement of the reference, autograd forces) on 1 B200, eager"
                      + (f", {swapped} Contracter(s) replaced by the reference's TritonContracter" if triton else ""),
                      "peak_mem_gb": round(torch.cuda.max_memory_allocated() / 2**30, 1)}}
    print(json.dumps(res))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu", "reference-gpu-triton"],
                    help="reference = CPU oracle (the driver's reference arm); reference-gpu(-triton) = the same oracle on the B200 "
                         "(eager PyTorch; -triton swaps in the reference's own Triton tensor-product kernel staged under oracle/_ref): "
                         "the GPU baseline of the >=10x target, NOT the driver's anchor")
    ap.add_argument("--config", default="c2")
    ap.add_argument("--dtype", default="float32", choices=["float64", "float32", "bfloat16"],
                    help="activation storage; default float32 (GEMMs on tcgen05 as split-bf16, fp32-accurate): bfloat16 storage, the dtype BASELINE names for c2, measured 4e-3/4e-2 (E/F) against the fp64 oracle, outside the 1e-3 parity bar")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity-check", action="store_true", help="skip the pre-timing E/F check against the CPU oracle sub-sample")
    ap.add_argument("--halo", default="p2p", choices=["p2p", "nccl"], help="N>1: ghost-atom exchange over NVLink peer memory (default) or NCCL")
    ap.add_argument("--reps", type=int, default=0, help="N>1: lattice repetitions per box edge instead of the config's own (smaller boxes for tests)")
    ap.add_argument("--no-c4", action="store_true", help="N=8: skip the extra 1M-atom c4 measurement")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from Python instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the outputs of the last one as DIR/<name>.npy "
                                                             "(float32 / float64; rows of large arrays sampled with a fixed seed, at most "
                                                             f"{DUMP_BUDGET_BYTES // 10**6} MB of data in all)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.dump_outputs and (args.impl != "ours" or world > 1):
        ap.error("--dump-outputs is supported for --impl ours on one GPU")
    if args.impl == "reference":
        return run_reference(args, rank, world)
    if args.impl.startswith("reference-gpu"):
        return run_reference_gpu(args, rank, world, triton=args.impl.endswith("triton"))
    return run_ours(args, rank, world)


if __name__ == "__main__":
    main()
