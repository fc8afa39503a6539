#!/usr/bin/env python
"""Headline benchmark: modal solves/s on the synthetic 200k quadratic-tet cube (BASELINE.json
configs[2]; SURVEY.md section 8d config 3).

One step = one modal solve of the hot path, from vertex positions already on the device:
    sparsity pattern + fused K/M assembly  ->  LOBPCG, 32 elastic modes (+6 rigid), cold start
    ->  get_vals() forward  ->  backward to all vertex positions (upstream grad 1/lambda).
`value` times that with CUDA events (inputs resident in HBM); `e2e` times the same through the public
API (`DiffSoundObj`) from pinned HOST buffers: H2D of the linear mesh, linear->quadratic promotion,
solve, D2H of eigenvalues and the vertex gradient.

N > 1 (torchrun): the path shards by independent candidates (the thickness / material sweeps of the
reference, SURVEY.md section 8e) -- every rank solves its own mesh, no data-path collective; NCCL is
used for the barriers and the max-over-ranks timing only ("scaling": "weak").

`--impl reference` times the CPU restatement of the reference algorithm (oracle/, kind "port": the
reference itself is Python + SciPy ARPACK and cannot travel to the GPU box) on a bounded sample.

`--dump-outputs DIR` writes what the last timed step returned to its caller as DIR/<name>.npy: the eigenvalues (fp64),
get_vals() (fp32) and the gradient to the quadratic vertex positions (fp32).  The input mesh is generated, not random, so
two builds run with the same arguments can be compared output for output.
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

METRIC = "modal solves/s (assemble+LOBPCG k=32+dlambda/dtheta) @200k ord-2 tets"
UNIT = "solves/s"
STEEL = (7850.0, 2.0e11, 0.29, 20, 3e-8)
CUBE_N = 32          # 32^3 cells x 6 Kuhn tets = 196 608 tets
MODES = 32


def kuhn_cube(N):
    """Synthetic procedurally tetrahedralised cube (SURVEY.md 8d config 3): (N+1)^3 grid on [0,1]^3,
    six Kuhn tets per cell, permutation-major.  numpy, host side."""
    import itertools
    import numpy as np
    import torch
    lin = torch.linspace(0, 1, N + 1).numpy()      # fp32, the rounding SURVEY.md 8d config 3 specifies
    gx, gy, gz = np.meshgrid(lin, lin, lin, indexing="ij")
    verts = np.stack([gx, gy, gz], axis=-1).reshape(-1, 3).astype(np.float32)
    ii, jj, kk = np.meshgrid(np.arange(N), np.arange(N), np.arange(N), indexing="ij")
    base = np.stack([ii, jj, kk], axis=-1).reshape(-1, 3)
    tets = []
    for perm in itertools.permutations(range(3)):
        p = base.copy()
        ids = [(p[:, 0] * (N + 1) + p[:, 1]) * (N + 1) + p[:, 2]]
        for ax in perm:
            p = p.copy()
            p[:, ax] += 1
            ids.append((p[:, 0] * (N + 1) + p[:, 1]) * (N + 1) + p[:, 2])
        tets.append(np.stack(ids, axis=1))
    return verts, np.concatenate(tets, axis=0).astype(np.int64)


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons while the timed region runs: through NVML in this process (what nvidia-smi
    itself reads; a query costs microseconds), falling back to the nvidia-smi command line of B200_PROFILING.md when the
    binding is missing.  (A forked nvidia-smi every 0.2 s put a 5-100 ms hiccup into the timed step it landed in.)"""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False
        self.nvml = self.handle = None
        try:                                    # initialised here, before the timed region
            import pynvml
            import torch
            pynvml.nvmlInit()
            try:
                p = torch.cuda.get_device_properties(index)
                bus = f"{p.pci_domain_id:08x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
                self.handle = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.nvml = pynvml
            # The first queries made while the GPU is busy are slow and hold a driver lock that kernel launches wait on (one
            # 96 .. 198 ms step among 88 ms steps, always the one in which the second sample fell): take them here, under load.
            busy = torch.empty(1 << 26, device=f"cuda:{index}")
            for _ in range(40):
                busy.add_(1.0)
            for _ in range(3):
                self._sample_nvml()
            torch.cuda.synchronize(index)
            del busy
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n, h = self.nvml, self.handle
        sm = n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM)
        pw = 0.0            # power is not sampled: the PMU read behind nvmlDeviceGetPowerUsage can take tens of milliseconds and
                            # holds a driver lock that kernel launches wait on (one 96 .. 198 ms step among 88 ms steps)
        get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        r = int(get(h))
        flag = lambda bit: "Active" if r & bit else "Not Active"      # noqa: E731
        # NVML reason bits: sw_power_cap 0x4, hw_slowdown 0x8, sw_thermal_slowdown 0x20, hw_thermal_slowdown 0x40
        return [str(sm), str(mx), f"{pw:.1f}", flag(0x8), flag(0x40), flag(0x20), flag(0x4)]

    def run(self):
        while not self.stop_flag:
            try:
                if self.nvml is not None:
                    self.samples.append(self._sample_nvml())
                else:
                    out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                          str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                    if out:
                        self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1 if self.nvml is not None else 0.2)

    def summary(self):
        import statistics
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        reasons = []
        for i, name in ((3, "hw_slowdown"), (4, "hw_thermal_slowdown"), (5, "sw_thermal_slowdown"), (6, "sw_power_cap")):
            if any(len(s) > i and s[i].lower().startswith("active") for s in self.samples):
                reasons.append(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.samples), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def measured_hbm_peak():
    """HBM GB/s for the roofline denominator: MEASURED_PEAKS.json (driver-written; the sustained figure when the file
    distinguishes burst and sustained, since the kernel is timed inside a long step), else the fallback of
    B200_PROFILING.md."""
    fallback = (6650.0, "fallback 6650 GB/s (B200_PROFILING.md)")
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return fallback
    found = []

    def walk(node, path):
        if isinstance(node, dict):
            for k, v in node.items():
                walk(v, path + [str(k)])
        elif isinstance(node, (int, float)) and not isinstance(node, bool):
            name = "/".join(path).lower()
            if any(t in name for t in ("hbm", "copy", "bandwidth", "gbs", "gb_s", "gbps")) and "tflop" not in name:
                val = float(node)
                if 0.5 <= val <= 20.0:          # TB/s
                    val *= 1000.0
                if 1000.0 <= val <= 20000.0:
                    found.append((name, val))

    walk(peaks, [])
    if not found:
        return fallback
    sustained = [f for f in found if "sustain" in f[0]]
    name, val = (sustained or found)[0]
    return val, f"measured (MEASURED_PEAKS.json {name})"


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


DUMP_LIMIT = 64 * 10 ** 6       # bytes --dump-outputs writes in all


def step_outputs(obj, vals, grad):
    """What one step of the timed path hands its caller, copied to the host."""
    return {"eigenvalues": obj.eigenvalues.detach().cpu().numpy(), "vals": vals.detach().cpu().numpy(),
            "vertex_grad": grad.detach().cpu().numpy()}


def dump_outputs(out_dir, arrays, limit=DUMP_LIMIT):
    """Writes every array as out_dir/<name>.npy.  Arrays of at most limit / 64 bytes are written whole.  If the larger ones do
    not fit in the rest of the limit, each is cut to a fixed, seeded sample of its rows (the same rows for the same row count),
    whose ids go to out_dir/<name>_rows.npy as float64."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    header = 256                                    # bytes of .npy header allowed per file
    small = {k for k, a in arrays.items() if a.nbytes <= limit // 64}
    large = [a for k, a in arrays.items() if k not in small]
    room = limit - sum(arrays[k].nbytes + header for k in small) - 2 * header * len(large)
    keep = 1.0
    if sum(a.nbytes for a in large) > room:
        keep = room / sum(a.nbytes + 8 * a.shape[0] for a in large)
    for name, a in arrays.items():
        if a.dtype not in (np.float32, np.float64):
            raise TypeError(f"--dump-outputs: {name} is {a.dtype}, not float32 / float64")
        if name not in small and keep < 1.0:
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], int(a.shape[0] * keep), replace=False))
            np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


# ----------------------------------------------------------------------------------------------
# CPU arm: the oracle's restatement of the reference algorithm on the host cores
# ----------------------------------------------------------------------------------------------
def cpu_reference_solve(N, order, k, threads):
    """One modal solve with the reference algorithm on the CPU: fp64 COO-free assembly, SciPy ARPACK
    shift-invert (sigma = 20000, as diff_model.py:356-358), eigenvalue gradient by autograd."""
    import numpy as np
    import torch
    from oracle import modal_oracle as mo
    torch.set_num_threads(threads)
    v, t = mo.kuhn_cube(N)
    t0 = time.perf_counter()
    pv, pt = mo.promote(v, t, order)
    K, M = mo.assemble(pv, pt, order, STEEL[1], STEEL[2], STEEL[0])
    lam, U, _, _ = mo.eig_arpack(K, M, k)
    g = mo.eigval_grad_shape(pv, pt, order, STEEL[1], STEEL[2], STEEL[0], U, lam, 1.0 / lam)
    dt = time.perf_counter() - t0
    return dt, pt.shape[0], float(np.abs(g.numpy()).sum())


CPU_CUBE_N = 10      # the CPU arm's bounded sample: 10^3 x 6 = 6 000 quadratic tets (n = 27 783 dofs), ~20 s per solve on
                     # 16 host threads; 16^3 x 6 = 24 576 tets measured 266.6 s per solve (gpurun_out/r2a_bench.json)


def cpu_baseline(sample_N, steps=1, warmup=0, budget_s=150.0):
    """Times the oracle port on ONE stated size -- no scaling to the full workload.  `value` is solves/s measured on the
    sample_N^3 x 6-tet cube; as many of the requested steps as fit in `budget_s` are run (at least one)."""
    threads = os.cpu_count() or 1
    t_begin = time.perf_counter()
    ts, tets = [], 0
    for i in range(warmup + steps):
        dt, tets, _ = cpu_reference_solve(sample_N, 2, MODES, threads)
        if i >= warmup or dt > 0.2 * budget_s:       # a warm-up pass that already eats the budget counts as a step
            ts.append(dt)
        if time.perf_counter() - t_begin + dt > budget_s and ts:
            break
    per_step = sum(ts) / len(ts)
    full_tets = 6 * CUBE_N ** 3
    return {"value": 1.0 / per_step, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": (f"oracle port of the reference algorithm (numpy/torch-CPU assembly + SciPy ARPACK shift-invert + autograd "
                       f"gradient) on a {sample_N}^3 x 6 = {tets}-tet quadratic Kuhn cube, k={MODES}: {per_step:.2f} s/solve, "
                       f"{len(ts)} timed solve(s), NOT scaled; the {full_tets}-tet workload does not finish on the host "
                       f"(SuperLU fill-in; SURVEY.md 8d)"),
            "sample_tets": int(tets), "steps_timed": len(ts),
            "extrapolated_full_size_solves_per_s_linear_in_tets": tets / (per_step * full_tets)}, per_step


def workload_name(cube):
    return f"synthetic {6 * cube ** 3}-tet quadratic Kuhn cube ({cube}^3 x 6), {MODES} elastic modes (+6 rigid), shape gradient"


def run_reference_arm(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    t0 = time.perf_counter()
    base, per_step = cpu_baseline(args.cpu_cube, steps=max(1, args.steps), warmup=min(args.warmup, 1))
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_step * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(CUBE_N),
                       "bounded_sample": workload_name(args.cpu_cube),
                       "note": ("value and ms_per_step are MEASURED on bounded_sample, not scaled; the GPU arm reports the "
                                "same size under same_size_as_reference_arm")},
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def verify_solution(obj, leaf, solve, native, torch):
    """FP64 checks of the solution the timed region produced (device side, after the timed region):
    max ||K u - lam M u|| / (lam ||M u||) and ||U^T M U - I|| over the wanted modes, the relative gap between the last
    wanted and the first unwanted eigenvalue (a cluster cut there would make sum_i g_i dlambda_i basis dependent), and
    the distance to a second solve at eig_tol = 1e-9 (eigenvalues: max relative difference; gradient: relative L2)."""
    k = obj.mode_num
    pat = obj.deform.pattern
    X = obj._Xpad
    lam_all = obj.ritz_values[:X.shape[1]]
    KX, MX = native.spmm_k_and_m(pat, obj._Kval, obj._Mblk, X)
    R = KX - MX * lam_all
    res = (R.norm(dim=0) / (lam_all.abs() * MX.norm(dim=0)))[6:6 + k]
    G = torch.cat([native.gram(X[:, c:c + 16].contiguous(), MX) for c in range(0, X.shape[1], 16)], dim=0)
    G = G[6:6 + k, 6:6 + k]
    ortho = float((G - torch.eye(k, dtype=G.dtype, device=G.device)).abs().max())
    rv = obj.ritz_values
    gap = float((rv[6 + k] - rv[6 + k - 1]) / rv[6 + k]) if rv.numel() > 6 + k else None
    lam5 = obj.eigenvalues.clone()
    g5 = leaf.grad.clone()
    it5 = obj.eig_stats["iterations"]
    tol_saved = obj.eig_tol
    try:
        obj.eig_tol = 1e-9
        solve(obj, leaf)
        lam9, g9, it9 = obj.eigenvalues.clone(), leaf.grad.clone(), obj.eig_stats["iterations"]
    finally:
        obj.eig_tol = tol_saved
    return {"max_rel_residual_fp64": float(res.max()), "max_abs_UtMU_minus_I": ortho,
            "rel_gap_lambda_k_to_k+1": gap,
            "max_rel_dlambda_vs_tol1e-9": float(((lam5 - lam9).abs() / lam9).max()),
            "rel_l2_dgradient_vs_tol1e-9": float((g5.double() - g9.double()).norm() / g9.double().norm()),
            "iterations_tol1e-5": it5, "iterations_tol1e-9": it9}


def run_rowpart(args):
    """ONE mesh on N GPUs ("scaling": "strong"): assembly replicated on every rank, LOBPCG on row slabs
    (diffsound_b200/parallel/rowpart_lobpcg.py: halo rows of the FP32 smoother read over NVLink inside the SpMM kernel, NCCL
    all-reduce of Gram strips / residual sums / partial coarse residuals, all-gather of the new search block), shape gradient
    replicated.  The partition and the peer-visible buffers are set up once per topology, outside the timed region."""
    import torch
    import torch.distributed as dist
    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    from diffsound_b200 import native
    from diffsound_b200.diffelastic.diff_model import DiffSoundObj
    from diffsound_b200.parallel.rowpart_lobpcg import eigen_decomposition_rowpart
    v_np, t_np = kuhn_cube(args.cube)
    leaf0 = torch.from_numpy(v_np).to(dev)
    obj = DiffSoundObj(leaf0, torch.from_numpy(t_np).to(dev), mode_num=MODES, order=2, mat=STEEL)
    leaf = obj.tetmesh.vertices.detach().clone().requires_grad_(True)
    obj.tetmesh.vertices = leaf
    state = {"solver": None}

    def solve():
        obj._X = None
        obj._warm = []
        obj._Kval = obj._Mblk = None
        stats, state["solver"] = eigen_decomposition_rowpart(obj, solver=state["solver"], keep=True)
        vals = state["vals"] = obj.get_vals()
        leaf.grad = None
        (vals[:, 0] * (1.0 / obj.eigenvalues).float()).sum().backward()
        return stats

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # host-side preparation first, then the warm-up steps straight into the timed region (see the sweep mode)
    lib = native._lib.load()
    stats = solve()                                # first call: arena growth, lazy module loading
    sampler = ClockSampler(local)
    import gc
    gc.collect()
    gc.disable()                                   # no cyclic-GC pass inside the timed region
    lib.ds_prof_reserve(8192)                      # every CUDA event of the region exists before it starts
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    for ev in [e0, e1] + marks:
        ev.record()
    for _ in range(max(3, args.warmup)):
        stats = solve()
    sampler.start()
    barrier()
    launches0 = lib.ds_launch_count()
    e0.record()
    for k in range(args.steps):
        stats = solve()
        marks[k].record()
    e1.record()
    barrier()
    launches = int(lib.ds_launch_count() - launches0)
    sampler.stop_flag = True
    outputs = step_outputs(obj, state["vals"], leaf.grad) if args.dump_outputs and rank == 0 else None
    each_ms = [a.elapsed_time(b) for a, b in zip([e0] + marks[:-1], marks)]
    tms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms_max = float(tms.item())
    gc.enable()
    with native.prof() as pf_all:
        for _ in range(2):
            solve()
        torch.cuda.synchronize()
    prof_all = pf_all.read()
    # wall time per phase of the driver with a device synchronize at every boundary (diagnostic pass, untimed)
    import time as _time
    sv = state["solver"]
    sv.profile, sv.phase_ms = True, {}
    t_a = _time.perf_counter()
    solve()
    torch.cuda.synchronize()
    t_total = (_time.perf_counter() - t_a) * 1e3
    phases = dict(sv.phase_ms)
    phases["outside_solver (assembly, start block, gradient)"] = t_total - sum(phases.values())
    sv.profile = False
    # the eigenvalues against the single-GPU driver on the same mesh (rank 0)
    lam_rp = obj.eigenvalues.clone()
    check = None
    if rank == 0:
        obj._X, obj._warm, obj._Kval, obj._Mblk = None, [], None, None
        obj.eigen_decomposition()
        check = float(((obj.eigenvalues - lam_rp).abs() / lam_rp).max())
    pat = obj.deform.pattern
    line = {"metric": METRIC, "value": args.steps / (ms_max * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "mode": "rowpart", "ms_each_step_rank0": each_ms,
            "config": {"workload": workload_name(args.cube),
                       "sizes": f"n={pat.n} dofs, nnz={9 * pat.nnzb}; ONE mesh, rows split over {world} GPU(s)",
                       "eig_tol": DiffSoundObj.eig_tol, "lobpcg_iterations": stats["iterations"],
                       "nested_p1_iterations": stats.get("nested_iterations"),
                       "replicated": "assembly, nested P1 eigen-solve, P1 coarse Chebyshev solves, small eigen-solves, gradient",
                       "max_rel_dlambda_vs_single_gpu_driver": check},
            "gpu_launches": launches, "clocks": sampler.summary(),
            "kernel_ms_per_step_rank0": {k: v["ms"] / 2 for k, v in prof_all.items()},
            "phase_wall_ms_rank0_synchronised": phases}
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    if rank == 0:
        print(json.dumps(line), flush=True)
    state["solver"].close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--cube", type=int, default=CUBE_N, help="cells per side (default 32 -> 196 608 tets)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-cube", type=int, default=CPU_CUBE_N, help="cells per side of the CPU arm's bounded sample")
    ap.add_argument("--no-verify", action="store_true", help="skip the FP64 verification of the timed solve")
    ap.add_argument("--mode", default="sweep", choices=["sweep", "rowpart"],
                    help="sweep: one independent mesh per GPU (weak scaling, the default and the driver's line); rowpart: ONE "
                         "mesh, eigen-solve row-partitioned over the GPUs (strong scaling)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs the native arm (the reference arm keeps no outputs)")
    if args.impl == "reference":
        run_reference_arm(args)
        return
    if args.mode == "rowpart":
        run_rowpart(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"       # keep NCCL's version banner off stdout: one JSON line only
        dist.init_process_group("nccl", device_id=dev)
    from diffsound_b200 import native
    from diffsound_b200.diffelastic.diff_model import DiffSoundObj
    from diffsound_b200.diffelastic.deform import Deform

    # ---- synthetic input (host, pinned) and the device-resident copy for the kernel-only number
    v_np, t_np = kuhn_cube(args.cube)
    # N > 1: every rank solves its own copy of the named configuration (weak scaling: the per-GPU work is exactly the
    # N = 1 work; a perturbed geometry per rank changes the LOBPCG iteration count and with it the work)
    v_host = torch.from_numpy(v_np).pin_memory()
    t_host = torch.from_numpy(t_np).pin_memory()

    def build(vh, th):
        leaf = vh.to(dev, non_blocking=True).requires_grad_(True)
        obj = DiffSoundObj(leaf, th.to(dev, non_blocking=True), mode_num=MODES, order=2, mat=STEEL)
        return leaf, obj

    _, obj = build(v_host, t_host)
    # kernel-only number: the promoted (quadratic) mesh is the device-resident input
    leaf = obj.tetmesh.vertices.detach().clone().requires_grad_(True)
    obj.tetmesh.vertices = leaf

    def solve(obj, leaf):
        """the hot path on device-resident inputs"""
        obj.deform = Deform(obj.tetmesh)        # pattern + incidence lists rebuilt: nothing topological is cached
        obj._X = None                           # cold start of the eigensolver
        obj._warm = []
        obj._Kval = obj._Mblk = None
        obj.eigen_decomposition()
        vals = obj.get_vals()
        up = (1.0 / obj.eigenvalues).float()
        leaf.grad = None
        (vals[:, 0] * up).sum().backward()
        return vals, leaf.grad

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # Warm-up in exactly the call pattern of the timed loop -- results BOUND to the names the loop rebinds.  While step k runs,
    # the previous step's `vals` (and, through its autograd graph, 0.25 GB of saved eigenvectors) is still alive; a warm-up
    # that drops its results never reaches that footprint, so the second timed step made torch's caching allocator call
    # cudaMalloc: one step of 96 .. 220 ms among 88 ms steps in about half of the runs.  Host-side preparation (NVML, garbage
    # collection, event creation) comes first, so that the warm-up steps run straight into the timed region.
    lib = native._lib.load()
    vals, grad = solve(obj, leaf)                  # first call: arena growth, lazy module loading
    sampler = ClockSampler(local)
    import gc
    gc.collect()
    gc.disable()                                   # no cyclic-GC pass inside the timed regions
    lib.ds_prof_reserve(8192)                      # every CUDA event of the region exists before it starts
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    for ev in [e0, e1] + marks:
        ev.record()
    for _ in range(max(3, args.warmup)):
        vals, grad = solve(obj, leaf)
    # ---- timed region (device time, CUDA events on the current stream = the kernels' stream)
    sampler.start()
    barrier()
    launches0 = lib.ds_launch_count()
    # only the dominant kernel class is bracketed by events inside the timed region (the roofline's launch time);
    # the per-class breakdown comes from a second, untimed pass below
    with native.prof(classes=["cheb_step"]) as pf:
        e0.record()
        for k in range(args.steps):
            vals, grad = solve(obj, leaf)
            marks[k].record()
        e1.record()
        barrier()
    prof = pf.read()
    launches = int(lib.ds_launch_count() - launches0)
    sampler.stop_flag = True
    outputs = step_outputs(obj, vals, grad) if args.dump_outputs and rank == 0 else None
    ms = e0.elapsed_time(e1)
    each_ms = [a.elapsed_time(b) for a, b in zip([e0] + marks[:-1], marks)]
    with native.prof() as pf_all:
        for _ in range(2):
            solve(obj, leaf)
        torch.cuda.synchronize()
    prof_all = pf_all.read()
    tms = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms_max = float(tms.item())
    ms_per_step = ms_max / args.steps
    value = world * args.steps / (ms_max * 1e-3)
    stats = obj.eig_stats

    # ---- end to end through the public API from host buffers (a new model per step, as the sweeps build one
    # per candidate); one untimed pass first so that the caching allocator owns the blocks a second model needs
    e2e_steps = args.steps                  # as many end-to-end steps as device-timed steps

    def e2e_step():
        lf, ob = build(v_host, t_host)
        ob.eigen_decomposition()
        vv = ob.get_vals()
        (vv[:, 0] * (1.0 / ob.eigenvalues).float()).sum().backward()
        return ob.eigenvalues.cpu(), lf.grad.cpu()

    lam_h, grad_h = e2e_step()
    barrier()
    t_e2e = time.perf_counter()
    for _ in range(e2e_steps):
        lam_h, grad_h = e2e_step()
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = world * e2e_steps / float(e2e_s.item())
    gc.enable()
    h2d = v_host.numel() * 4 + t_host.numel() * 8
    d2h = lam_h.numel() * 8 + grad_h.numel() * 4

    # ---- the answer at the size that was timed (verdict r1, item 1): FP64 residuals and M-orthonormality of the 32
    # modes of the timed configuration, and a re-solve at eig_tol = 1e-9 to bound the eigenvalue / gradient error
    verify = None
    if not args.no_verify:
        verify = verify_solution(obj, leaf, solve, native, torch)
        if verify["max_rel_dlambda_vs_tol1e-9"] > 1e-6:
            raise SystemExit(f"bench.py: eigenvalues of the timed solve differ from the 1e-9 solve by "
                             f"{verify['max_rel_dlambda_vs_tol1e-9']:.3e} > 1e-6")

    # ---- the reference arm's bounded sample on the GPU, through the public API from host buffers (same_config ratio)
    same = None
    if rank == 0 and args.cpu_cube != args.cube:
        vs_np, ts_np = kuhn_cube(args.cpu_cube)
        vs_h, ts_h = torch.from_numpy(vs_np).pin_memory(), torch.from_numpy(ts_np).pin_memory()

        def small_step():
            lf, ob = build(vs_h, ts_h)
            ob.eigen_decomposition()
            vv = ob.get_vals()
            (vv[:, 0] * (1.0 / ob.eigenvalues).float()).sum().backward()
            return ob.eigenvalues.cpu(), lf.grad.cpu()

        for _ in range(2):
            small_step()
        torch.cuda.synchronize()
        t_s = time.perf_counter()
        for _ in range(5):
            small_step()
        torch.cuda.synchronize()
        dt_s = (time.perf_counter() - t_s) / 5
        same = {"workload": workload_name(args.cpu_cube), "value": 1.0 / dt_s, "unit": UNIT, "ms_per_step": dt_s * 1e3,
                "how": "end to end through DiffSoundObj from pinned host buffers (H2D, promotion, pattern, assembly, "
                       "eigen-solve, backward, D2H), new model per step, 5 timed steps"}

    # ---- roofline of the dominant kernel class, from the event times of the timed region
    pat = obj.deform.pattern
    n, nnzb, n_nodes = pat.n, pat.nnzb, pat.n_nodes
    roof = None
    peak, peak_src = measured_hbm_peak()
    if stats and "cheb_step" in prof and stats.get("cheb_steps"):
        # One fine-level FP32 SpMM launch (k_spmm32v) streams one 40-byte record per 3x3 block (9 fp32 K
        # values + bcol), brow (4 B) and the 3x3 block-Jacobi inverse (36 B) per node, reads the gathered
        # block Z once plus R and Zprev, and writes Znew: 4 x n x c x 4 B (3 for the residual launch of a
        # V-cycle, which has no Zprev).
        c_avg = stats["cheb_cols_avg"]
        steps_total = stats["cheb_steps"]          # V-cycle smoothing + residual launches + the 20 power-iteration launches
        n_resid = stats["iterations"] if stats.get("two_level") else 0
        streams = 4.0 - n_resid / steps_total
        per_launch_bytes = nnzb * 40 + n_nodes * (4 + 36) + streams * n * c_avg * 4
        t_avg = prof["cheb_step"]["ms"] / prof["cheb_step"]["count"] * 1e-3     # seconds per launch
        # DRAM traffic of the same kernel from the committed ncu --set full capture (per launch at the captured
        # column count), scaled to this run's average column count by the algorithmic-byte ratio
        traffic = None
        try:
            cap = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))["k_spmm32v"]
            cap_alg = nnzb * 40 + n_nodes * (4 + 36) + 4.0 * n * cap["ncols"] * 4
            traffic = cap["dram_bytes_per_launch"] * per_launch_bytes / cap_alg
        except Exception:
            pass
        roof = {"bound": "hbm", "kernel": "k_spmm32v (FP32 block-CSR SpMM on 40 B records, L1-resident gather in a Morton "
                                          "node numbering, packed FFMA2, fused Chebyshev update; the fine-level smoother "
                                          "of the eigensolver's preconditioner)",
                "achieved": per_launch_bytes / t_avg / 1e9, "peak": peak, "unit": "GB/s",
                "frac": per_launch_bytes / t_avg / 1e9 / peak, "traffic": traffic, "peak_source": peak_src,
                "launches_per_step": steps_total, "avg_launch_ms": t_avg * 1e3, "avg_cols": c_avg,
                "bytes_per_launch": per_launch_bytes, "share_of_step": prof["cheb_step"]["ms"] / ms}
    # ---- every kernel class against the roofline that bounds it (algorithmic bytes / flops accounted at the launch sites,
    # csrc/prof.cu; device time from the CUDA events of the untimed profiling pass)
    fp64_peak = None
    try:
        fp64_peak = json.load(open(os.path.join(ROOT, "profiles", "fp64_peak.json")))["dmma_m8n8k4_tflops"]
    except Exception:
        pass
    roofline_all = {}
    names = {"spmm": "k_spmm_dual_z32 / k_spmm_dual (FP64 K.W, M.W)", "assemble": "k_tet_geometry + k_assemble_rows",
             "gram": "k_gram_strip / k_gram_sym2 / k_gram (DMMA)", "block_gemm": "k_rr_update2 / k_block_gemm (DMMA)",
             "grad_shape": "k_eigval_grad_shape"}
    for cls, kname in names.items():
        v = prof_all.get(cls)
        if not v or not v["ms"]:
            continue
        sec = v["ms"] * 1e-3
        ent = {"kernels": kname, "ms_per_step": v["ms"] / 2, "launches_per_step": v["count"] / 2,
               "algorithmic_GB_per_step": v["bytes"] / 2 / 1e9, "achieved_GBps": v["bytes"] / sec / 1e9,
               "hbm_frac": v["bytes"] / sec / 1e9 / peak}
        if v["flops"]:
            ent["algorithmic_GFLOP_per_step"] = v["flops"] / 2 / 1e9
            ent["achieved_TFLOPs"] = v["flops"] / sec / 1e12
            if fp64_peak:
                ent["fp64_frac"] = v["flops"] / sec / 1e12 / fp64_peak
        roofline_all[cls] = ent
    if roof:
        roofline_all["cheb_step"] = {"kernels": "k_spmm32v (fine-level FP32 SpMM)", "ms_per_step": prof_all["cheb_step"]["ms"] / 2,
                                     "achieved_GBps": roof["achieved"], "hbm_frac": roof["frac"]}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "ms_each_step": each_ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(args.cube),
                       "sizes": f"n={n} dofs, nnz={9 * nnzb}; one independent mesh per GPU",
                       "bounded_sample": workload_name(args.cpu_cube),
                       "l2_policy": "inputs larger than L2 (K values alone 553 MB vs 126 MB L2); no flush needed",
                       "host_gc": "Python cyclic GC collected before and disabled inside the timed regions",
                       "eig_tol": DiffSoundObj.eig_tol, "lobpcg_iterations": stats["iterations"] if stats else None,
                       "nested_p1_iterations": stats.get("nested_iterations") if stats else None,
                       "preconditioner": ("fp32 two-level p-multigrid (P2 Chebyshev-Jacobi smoother, P1 coarse Chebyshev)"
                                          if stats and stats.get("two_level") else "fp32 block-Jacobi Chebyshev"),
                       "pattern_rebuilt_each_step": True, "eigensolver_cold_start": True, "verification": verify},
            "same_size_as_reference_arm": same,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps},
            "gpu_launches": launches, "clocks": sampler.summary(),
            "kernel_ms_per_step": {k: v["ms"] / 2 for k, v in prof_all.items()},
            "roofline": roof, "roofline_all": roofline_all,
            "fp64_peak_tflops": fp64_peak}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"], _ = cpu_baseline(args.cpu_cube, steps=1, warmup=0, budget_s=120.0)
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
