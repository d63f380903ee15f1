#!/usr/bin/env python
"""bench.py -- LVG solves/s of the batched forward-model sweep (BASELINE.json configs[1]) and, beside it, the other
quantities BASELINE.json's metric names: walker-steps/s of the sharded stretch-move sampler and the flux rel-err.

One "step" = one pass of the hot path over one batch: 2^20 random (Tkin, n_H2, N_CO/dv) CO LVG
solves (41 levels / 40 lines), drawn as SURVEY.md 8(d) config 2, each carried to the reference's
own stop rule (pyradex: sum|dx| < 1e-16 after > 10 iterations, cap 200) unless --stop radex.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--log2n 20] [--stop pyradex|radex]
                  [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  `value`: inputs resident in HBM, kernel timed with CUDA events on
its launch stream, L2 flushed between timed steps.  `e2e`: same workload through the C ABI's
host-pointer entry (rb_solve_batch) with pinned host buffers, H2D and D2H inside the timed region.
Outside the timed region, at every N (extra keys of the same line):
  `parity`      first 2000 draws of rank 0's sweep, the arrays of the timed launch against oracle/ (the bit-exact C
                restatement of the reference): rel-err of populations and fluxes on ALL models, the well-posed
                fraction, counts per excluded class (oracle/parity.py);
  `stop_radex`  the same sweep under RADEX's own convergence rule (Fortran matrix()'s conv flag): solves/s and the
                error of every model against the fixed point (the pyradex-rule arrays of the timed launch);
  `sampler`     BASELINE.json configs[4] shape: two-component model, 2^20 walkers in total sharded over the N
                ranks, NCCL all-gather of the complementary half per half-step, burnt-in start: walker-steps/s,
                solves/s, all-gather share;
  `sampler_small` (N = 1) configs[0] and configs[3] shapes: 100 walkers; 16 sources x 100 walkers in one ensemble.
`--impl reference`: the reference's CPU implementation of the same path (the bit-exact C
restatement in oracle/, since the reference ships only a macOS binary) on all host threads.
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TBG = 2.7315 * (1 + 3)          # config 2: z = 3 background (SURVEY.md 8d)
# algorithmic flops (SURVEY.md 8d): per matrix iteration and per solve prologue/epilogue, CO
F_ITER = 72368.0
F_PRO = 1.3e4
F_EPI = 4.0e3
MOLFILE = os.path.join(ROOT, "radex_emcee_b200", "data", "co.dat")
DUMP_BYTES = 48 << 20           # --dump-outputs: larger batches are sampled down to this many bytes of models
DUMP_SEED = 20240601


def draw(n, seed):
    rng = np.random.default_rng(seed)
    out = np.empty((0, 3))
    while out.shape[0] < n:
        m = int(1.6 * (n - out.shape[0])) + 16
        ln, lt, lN = rng.uniform(2, 7, m), rng.uniform(np.log10(TBG), 3, m), rng.uniform(15.5, 19.5, m)
        ok = (lN - ln > 10.0) & (lN - ln < 17.5)
        out = np.vstack([out, np.column_stack([10 ** lt, 10 ** ln, 10 ** lN])[ok]])
    out = out[:n]
    return np.ascontiguousarray(out[:, 0]), np.ascontiguousarray(out[:, 1]), np.ascontiguousarray(out[:, 2])


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


def source_hash():
    """Identifies the kernel sources a profile under profiles/ was taken with."""
    h = hashlib.sha256()
    for f in ("radex_b200.cu", "lvg_v2.cuh", "lvg_small.cuh", "stretch.cuh"):
        with open(os.path.join(ROOT, "radex_emcee_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def measured_traffic(log2n, kernel, stop_rule):
    """DRAM bytes of one step (all launches) from the committed ncu pass -- only if it was taken with THESE kernel
    sources and this workload; otherwise null (bench.py cannot measure DRAM traffic itself)."""
    p = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if not os.path.exists(p):
        return None, "no ncu pass committed for this build"
    with open(p) as f:
        t = json.load(f)
    if t.get("source_hash") != source_hash():
        return None, "profiles/r2_traffic.json was taken with other kernel sources (%s)" % t.get("source_hash")
    if (t.get("log2n"), t.get("kernel"), t.get("stop_rule")) != (log2n, kernel, stop_rule):
        return None, "profiles/r2_traffic.json holds another workload"
    return float(t["dram_bytes_per_step"]), t.get("how", "")


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.stop_flag = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 6:
                    self.rows.append(parts)
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for i, nm in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]),
                "reasons": reasons, "samples": len(self.rows)}


def cpu_reference(tk, nh2, cd, stop_rule, max_seconds, threads):
    """Time the oracle (bit-exact restatement of the reference's CPU path) on `threads` host threads."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle.oracle import Oracle
    # calibrate on a few solves, then size the sample for ~max_seconds of wall time
    o = Oracle(MOLFILE)
    t0 = time.perf_counter()
    o.solve_batch(tk[:24], 0.25 * nh2[:24], 0.75 * nh2[:24], cd[:24], tbg=TBG, stop_rule=stop_rule)
    per = (time.perf_counter() - t0) / 24
    n = int(min(tk.size, max(threads * 8, max_seconds / per * threads)))
    chunks = np.array_split(np.arange(n), threads)
    oracles = [Oracle(MOLFILE) for _ in range(threads)]

    def work(i):
        idx = chunks[i]
        r = oracles[i].solve_batch(tk[idx], 0.25 * nh2[idx], 0.75 * nh2[idx], cd[idx], tbg=TBG, stop_rule=stop_rule)
        return int(r["niter"].sum())

    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:
        iters = sum(ex.map(work, range(threads)))
    dt = time.perf_counter() - t0
    return n / dt, n, dt, iters


def make_config(log2n, stop):
    """`config` of the JSON line: the same dict on both arms (the reference arm times a sample of this workload)."""
    return {"workload": "batched forward-model sweep: 2^%d random (Tkin,n_H2,N_CO/dv) CO LVG solves, 41 levels, "
                        "tbg=%.3f K, stop=%s" % (log2n, TBG, stop),
            "models_per_gpu": 1 << log2n, "outputs": "xpop,tex,tau,surf,niter,status",
            "l2": "GPU arm: 256 MiB flush write between timed steps"}


# ---- extra records (outside the timed region) ------------------------------------------------------------------
def parity_record(n_par, tk, nh2, cd, arrays):
    """First n_par draws of the sweep: the timed launch's own arrays against the oracle, per class of model."""
    from oracle import parity
    got = {k: v[:n_par] for k, v in arrays.items()}
    rec, ref, cls, w, att = parity.summary(got, MOLFILE, tk[:n_par], nh2[:n_par], cd[:n_par], TBG)
    rec["excluded"]["nonfinite"]["gpu_flags_nonfinite"] = int(((got["status"] & 8) != 0)[cls["nonfinite"]].sum())
    rec["against"] = ("oracle/ (bit-exact C restatement of the reference binary), %d host threads; arrays of the last "
                      "timed launch" % (os.cpu_count() or 1))
    return rec


def sampler_models():
    from radex_emcee_b200 import emcee_radex as er1, emcee_radex_2comp as er2
    from radex_emcee_b200.data import get_source, read_data
    return er1, er2, get_source, read_data


def sampler_record(ctx, world, rank, dev, log2w, burn, steps, stop_rule):
    """configs[4]: two-component model, 2^log2w walkers in total over the ranks, burnt-in start."""
    import torch
    import torch.distributed as dist
    from radex_emcee_b200 import _lib
    from radex_emcee_b200.sampler import CudaEngine, SLEDModel, StretchSampler
    er1, er2, get_source, read_data = sampler_models()
    z, T_d, lw, jup, flux, eflux = get_source("G09v1.97", read_data(ROOT + "/data/flux_for2p.dat"))
    tbg, ra, bounds, p0 = er2.source_setup(z)
    p0 = p0.copy()
    p0[3] += 0.1
    nw = 1 << log2w
    # a spread of the order of the posterior's width (0.3 dex in n and N, 0.1 in T, 0.2 in size), redrawn until the
    # prior is finite, then `burn` untimed steps: the ensemble the timed steps see is not a point
    rng = np.random.default_rng(20170914)
    sig = np.array([0.3, 0.1, 0.3, 0.2, 0.3, 0.1, 0.3, 0.2])
    pos = p0 + sig * rng.standard_normal((nw, 8))
    for _ in range(60):
        bad = ~np.isfinite(er2.lnprior(pos, bounds, T_d=T_d))
        if not bad.any():
            break
        pos[bad] = p0 + sig * rng.standard_normal((int(bad.sum()), 8))
    opts = _lib.default_opts(stop_rule=stop_rule)
    eng = CudaEngine(ctx, SLEDModel(2, jup, flux, eflux, bounds, tbg, T_d=T_d, opts=opts))
    s = StretchSampler(nw, 8, eng, seed=1, time_gather=True)
    s.run_mcmc(pos, burn, store=False)
    torch.cuda.synchronize(dev)
    s.gather_ms()
    if world > 1:
        dist.barrier()
    solves0 = int(eng.total_solves.item()) + s.total_solves
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    s.run_mcmc(None, steps, store=False)
    e1.record()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    t = torch.tensor([e0.elapsed_time(e1), s.gather_ms(), float(int(eng.total_solves.item()) + s.total_solves - solves0)],
                     dtype=torch.float64, device=dev)
    if world > 1:
        mx = t.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = t.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        t_ms, g_ms, solves = float(mx[0]), float(mx[1]), float(sm[2])
    else:
        t_ms, g_ms, solves = float(t[0]), float(t[1]), float(t[2])
    acc = s.acceptance_fraction          # collective
    x, lnp = s.get_last_sample()         # collective
    return {"config": "configs[4] shape: two-component CO model (G09v1.97, T_d prior), 2^%d walkers in total over %d "
                      "rank(s), stretch move a=2, randomized split, stop=%s" % (log2w, world, "pyradex" if stop_rule == 0 else "radex"),
            "walkers": nw, "walkers_per_gpu": nw // world, "burn_steps": burn, "steps": steps,
            "start": "p0 + N(0, [0.3,0.1,0.3,0.2]x2 dex), prior-finite, then the burn steps",
            "walker_steps_per_s": nw * steps / (t_ms * 1e-3), "solves_per_s": solves / (t_ms * 1e-3),
            "ms_per_step": t_ms / steps, "solves_per_walker_step": solves / (nw * steps),
            "allgather": {"ms_per_step": g_ms / steps, "fraction": g_ms / t_ms,
                          "bytes_per_rank_per_half_step": (nw // world // 2) * 8 * 8,
                          "collective": "NCCL all_gather_into_tensor of the complementary half's positions" if world > 1 else "none (1 rank)"},
            "acceptance_fraction": float(np.mean(acc)), "lnprob_finite_fraction": float(np.isfinite(lnp).mean()),
            "spread_dex_after": [float(v) for v in np.std(x, axis=0)],
            "native_loop": bool(s.native), "scaling": "strong (fixed 2^%d walkers)" % log2w,
            "timing": "CUDA events on the launch stream around the timed steps, max over ranks"}


def sampler_small_records(ctx, dev, stop_rule):
    """configs[0] (100 walkers, one source) and configs[3] (all 16 flux.dat sources x 100 walkers in one ensemble)."""
    import torch
    from radex_emcee_b200 import _lib
    from radex_emcee_b200.sampler import CudaEngine, SLEDModel, StretchSampler
    er1, er2, get_source, read_data = sampler_models()
    data = read_data(ROOT + "/data/flux.dat")
    opts = _lib.default_opts(stop_rule=stop_rule)
    out = []
    for label, names in (("configs[0] shape: one source (G09v1.97), 100 walkers", list(data)[:1]),
                         ("configs[3] shape: all %d flux.dat sources concurrently, 100 walkers each, one ensemble" % len(data),
                          list(data))):
        models, starts = [], []
        for k, nm in enumerate(names):
            z, lw, jup, flux, eflux = get_source(nm, data)
            tbg, ra, bounds, p0 = er1.source_setup(z)
            models.append(SLEDModel(1, jup, flux, eflux, bounds, tbg, opts=opts))
            starts.append(p0 + 1e-3 * np.random.default_rng(20170914 + k).standard_normal((100, 4)))
        eng = CudaEngine(ctx, models)
        s = StretchSampler(100 * len(names), 4, eng, seed=1, nsources=len(names))
        s.run_mcmc(np.vstack(starts), 30, store=False)          # the drivers' burn-in, shortened
        torch.cuda.synchronize(dev)
        solves0 = s.total_solves
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        steps = 100
        e0.record()
        s.run_mcmc(None, steps, store=False)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1)
        out.append({"config": label, "walkers": 100 * len(names), "sources": len(names), "steps": steps,
                    "walker_steps_per_s": 100 * len(names) * steps / (ms * 1e-3), "ms_per_step": ms / steps,
                    "solves_per_s": (s.total_solves - solves0) / (ms * 1e-3),
                    "acceptance_fraction": float(np.mean(s.acceptance_fraction)), "native_loop": bool(s.native),
                    "loop": "rb_stretch_run_dev: CUDA graph of one step replayed; second half-step proposed speculatively "
                            "(rb_opts.spec_half = 0: one lnprob launch of 1.5 N candidates per step, same chain bit for bit; "
                            "solves_per_s counts the speculative solves as well)"})
    return out


def dump_outputs(out_dir, arrays):
    """Write the per-model device arrays `arrays` (name -> tensor with one row per model) as out_dir/<name>.npy in
    float64.  Where all of them together exceed DUMP_BYTES, the same seeded sample of models is kept in every array.
    Every file holds finite numbers only: the solver returns an infinite or NaN brightness where the reference does
    (status bit RB_ST_NONFINITE), so each floating-point output is written with 0 in place of a non-finite entry, and
    <name>_nonfinite.npy (float32, same shape) says what stood there: 0 finite, 1 NaN, 2 +inf, 3 -inf."""
    import torch
    n = next(iter(arrays.values())).shape[0]
    row_bytes = sum((12 if a.is_floating_point() else 8) * (a[0].numel() if a.dim() > 1 else 1) for a in arrays.values())
    keep = DUMP_BYTES // row_bytes
    idx = None
    if n > keep:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, keep, replace=False))
        idx = torch.from_numpy(idx).to(next(iter(arrays.values())).device)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = (a if idx is None else a[idx]).to(torch.float64)
        if arrays[name].is_floating_point():
            code = torch.zeros(a.shape, dtype=torch.float32, device=a.device)
            code[torch.isnan(a)] = 1
            code[torch.isposinf(a)] = 2
            code[torch.isneginf(a)] = 3
            np.save(os.path.join(out_dir, name + "_nonfinite.npy"), code.cpu().numpy())
            a = torch.where(code == 0, a, torch.zeros_like(a))
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())


def emit(line):
    """The ONE JSON line of the contract goes to the process's real stdout; everything else that libraries write to fd 1
    while the bench runs (NCCL prints its version there) is sent to stderr by main()."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)          # fd 1 -> stderr for the duration of the run (C libraries included)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log2n", type=int, default=20)
    ap.add_argument("--stop", default="pyradex", choices=["pyradex", "radex"])
    ap.add_argument("--abs-tol", type=float, default=1e-16, help="pyradex stop rule: run_radex's abs_convergence_threshold (core.py:857)")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--no-cpu", action="store_true", help="skip cpu_baseline and the oracle-side parity record")
    ap.add_argument("--no-extras", action="store_true", help="skip the parity / stop_radex / sampler records")
    ap.add_argument("--no-e2e", action="store_true", help="profiling aid: skip the host-buffer leg (e2e is then null)")
    ap.add_argument("--parity-n", type=int, default=2000)
    ap.add_argument("--sampler-log2w", type=int, default=20)
    ap.add_argument("--sampler-burn", type=int, default=20)
    ap.add_argument("--sampler-steps", type=int, default=10)
    ap.add_argument("--keep", default="", help="debug: small | big | k57 | k8 -- keep only the models whose lead block (from a first pass) has <= 16 | > 16 | 20..28 | > 28 levels, tiled to n")
    ap.add_argument("--park-max", type=int, default=0, help="rb_opts.park_max (profiling aid: 7 gives the 20/24/28-level engines their own launches on small batches)")
    ap.add_argument("--kernel", type=int, default=0, help="rb_opts.kernel: 0 default, 1 v1 LU, 2 v2 without caching, 3 single launch, 4 without the half-warp engine")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed launch returned (xpop, tex, tau, surf, niter, "
                         "status) as DIR/<name>.npy in float64, rank 0 only, non-finite entries as 0 with their kind "
                         "in DIR/<name>_nonfinite.npy; batches of more than %d MiB are sampled to that size, the same "
                         "models on every run (fixed seed)" % (DUMP_BYTES >> 20))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl b200: the reference arm times a sample whose size depends on its speed")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n = 1 << args.log2n
    stop_rule = 0 if args.stop == "pyradex" else 1
    config = make_config(args.log2n, args.stop if args.abs_tol == 1e-16 else "%s(abs_tol=%g)" % (args.stop, args.abs_tol))
    cores = os.cpu_count() or 1

    if args.impl == "reference":
        if rank != 0:
            return
        tk, nh2, cd = draw(n, 0)
        vals = []
        per_step = max(5.0, min(30.0, 120.0 / max(1, args.steps + args.warmup)))
        sample = 0
        for s in range(args.warmup + args.steps):
            v, sample, dt, _ = cpu_reference(tk, nh2, cd, stop_rule, per_step, cores)
            if s >= args.warmup:
                vals.append((v, dt))
        value = float(np.mean([v for v, _ in vals]))
        line = {"impl": "reference", "metric": "LVG solves/s", "value": value, "unit": "solves/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean([d for _, d in vals]) * 1e3),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config,
                "cpu_baseline": {"value": value, "unit": "solves/s", "cores": cores, "kind": "port",
                                 "sample": "first %d draws of the sweep per step, %d threads; oracle/ is the bit-exact C "
                                           "restatement of the reference (its Fortran ships only as a macOS binary)" % (sample, cores)},
                "e2e": {"value": value, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        emit(line)
        return

    import torch
    import torch.distributed as dist
    from radex_emcee_b200 import _lib

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback in the product path)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    mol = _lib.MolData(MOLFILE)
    ctx = _lib.Context(mol, local_rank)
    L = _lib.load()
    nl, nn, npart = mol.nlev, mol.nline, mol.npart

    tk, nh2, cd = draw(n, rank)                      # weak scaling: every rank gets its own 2^k draws
    dens = np.zeros((n, npart))
    for p, pid in enumerate(mol.partner_id):
        dens[:, p] = {2: 0.25, 3: 0.75}.get(int(pid), 0.0) * nh2
    d_tk, d_dens, d_cd = (torch.from_numpy(a).to(dev) for a in (tk, dens, cd))
    d_x = torch.empty((n, nl), dtype=torch.float64, device=dev)
    d_tex = torch.empty((n, nn), dtype=torch.float64, device=dev)
    d_tau = torch.empty_like(d_tex)
    d_surf = torch.empty_like(d_tex)
    d_it = torch.empty(n, dtype=torch.int32, device=dev)
    d_st = torch.empty(n, dtype=torch.int32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2
    opts = _lib.default_opts(stop_rule=stop_rule, kernel=args.kernel, abs_tol=args.abs_tol, park_max=args.park_max)
    stream = torch.cuda.current_stream(dev)
    ctx.set_stream(stream.cuda_stream)

    def launch(o=opts, surf=d_surf, x=d_x, it=d_it, st=d_st):
        _lib.check(L.rb_solve_batch_dev(ctx.handle, n, d_tk.data_ptr(), d_dens.data_ptr(), d_cd.data_ptr(), 1.0, TBG, 2,
                                        C.byref(o), x.data_ptr(), d_tex.data_ptr(), d_tau.data_ptr(),
                                        surf.data_ptr(), it.data_ptr(), st.data_ptr()))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    if args.keep in ("small", "big", "k57", "k8"):
        launch()
        torch.cuda.synchronize(dev)
        tau = d_tau.cpu().numpy()
        thick = ~(np.abs(tau) * 0.5 < np.float32(0.01))
        top = np.where(thick.any(axis=1), thick.shape[1] - np.argmax(thick[:, ::-1], axis=1), -1)   # upper level of the highest thick line
        key = np.maximum(3, (top + 1 + 4) >> 2)
        sel = np.nonzero({"small": key <= 4, "big": key > 4, "k57": (key > 4) & (key < 8), "k8": key >= 8}[args.keep])[0]
        o = np.resize(sel, n)
        tk, nh2, cd, dens = tk[o].copy(), nh2[o].copy(), cd[o].copy(), dens[o].copy()
        d_tk.copy_(torch.from_numpy(tk)); d_cd.copy_(torch.from_numpy(cd)); d_dens.copy_(torch.from_numpy(dens))
    for _ in range(args.warmup):
        launch()
    torch.cuda.synchronize(dev)
    launches_before = ctx.counters()[1]
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # ---- kernel-only: K steps, each bracketed by events on the launch stream, L2 flushed between ----
    barrier()
    t_wall0 = time.perf_counter()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for k in range(args.steps):
        flush.fill_(k & 0xFF)
        ev[k][0].record(stream)
        launch()
        ev[k][1].record(stream)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    step_ms = [a.elapsed_time(b) for a, b in ev]
    kern_ms = float(sum(step_ms))
    total_iters, launches_after = ctx.counters()      # iterations of the last step (device-counted)
    launches_timed = launches_after - launches_before  # kernels launched inside the kernel-only timed region
    cache_stats = ctx.cache_stats()                   # (cached iterations, captures, invalidations), last launch
    niter_host = d_it.cpu().numpy()
    status_host = d_st.cpu().numpy()
    npar = min(args.parity_n, n)      # the arrays the parity record checks are the timed launch's own
    par_arrays = {"xpop": d_x[:npar].cpu().numpy(), "tex": d_tex[:npar].cpu().numpy(), "tau": d_tau[:npar].cpu().numpy(),
                  "surf": d_surf[:npar].cpu().numpy(), "niter": niter_host[:npar].copy(), "status": status_host[:npar].copy()}
    if args.dump_outputs and rank == 0:         # before the extra records: their launches write into d_tex and d_tau
        dump_outputs(args.dump_outputs, {"xpop": d_x, "tex": d_tex, "tau": d_tau, "surf": d_surf, "niter": d_it,
                                         "status": d_st})

    # ---- e2e: host buffers through the C ABI (pinned), H2D + D2H inside the timed region --------------
    def pinned(shape, dtype):
        return torch.empty(shape, dtype=dtype, pin_memory=True)

    h_tk, h_cd = pinned(n, torch.float64), pinned(n, torch.float64)
    h_dens = pinned((n, npart), torch.float64)
    h_tk.copy_(torch.from_numpy(tk)); h_cd.copy_(torch.from_numpy(cd)); h_dens.copy_(torch.from_numpy(dens))
    h_x, h_tex, h_tau, h_surf = pinned((n, nl), torch.float64), pinned((n, nn), torch.float64), \
        pinned((n, nn), torch.float64), pinned((n, nn), torch.float64)
    h_it, h_st = pinned(n, torch.int32), pinned(n, torch.int32)

    def e2e_call():
        _lib.check(L.rb_solve_batch(ctx.handle, n, h_tk.data_ptr(), h_dens.data_ptr(), h_cd.data_ptr(), 1.0, TBG, 2,
                                    C.byref(opts), h_x.data_ptr(), h_tex.data_ptr(), h_tau.data_ptr(),
                                    h_surf.data_ptr(), h_it.data_ptr(), h_st.data_ptr()))

    if not args.no_e2e:
        e2e_call()                                    # warm-up (allocates the ctx scratch)
    barrier()
    t0 = time.perf_counter()
    for _ in range(0 if args.no_e2e else args.steps):
        e2e_call()                                    # synchronous: returns after the D2H copies
    barrier()
    e2e_s = time.perf_counter() - t0
    if rank == 0:
        sampler.stop_flag.set()
        sampler.join(timeout=5)
    h2d = (2 * n + n * npart) * 8
    d2h = (n * nl + 3 * n * nn) * 8 + 2 * n * 4

    # ---- max over ranks ------------------------------------------------------------------------------------
    t = torch.tensor([kern_ms, e2e_s * 1e3, float(total_iters)], dtype=torch.float64, device=dev)
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        kern_ms, e2e_ms, iters_all = float(tmax[0]), float(tmax[1]), float(tsum[2])
    else:
        kern_ms, e2e_ms, iters_all = float(t[0]), float(t[1]), float(t[2])

    # ---- extra records: every rank takes part in the collective ones ---------------------------------------
    extras = {}
    if not args.no_extras and not args.keep and args.kernel == 0 and args.abs_tol == 1e-16:
        # (1) the same sweep under the other stop rule, against the arrays of the timed launch
        other = 1 - stop_rule
        o2 = _lib.default_opts(stop_rule=other, kernel=args.kernel)
        x2, s2 = torch.empty_like(d_x), torch.empty_like(d_surf)
        it2, st2 = torch.empty_like(d_it), torch.empty_like(d_st)
        for _ in range(2):
            launch(o2, s2, x2, it2, st2)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        flush.fill_(1)
        e0.record(stream)
        launch(o2, s2, x2, it2, st2)
        e1.record(stream)
        barrier()
        it_other, _ = ctx.counters()
        tt = torch.tensor([e0.elapsed_time(e1), float(it_other)], dtype=torch.float64, device=dev)
        if world > 1:
            tm = tt.clone(); dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            ts = tt.clone(); dist.all_reduce(ts, op=dist.ReduceOp.SUM)
            ms_o, it_o = float(tm[0]), float(ts[1])
        else:
            ms_o, it_o = float(tt[0]), float(tt[1])
        # error of the RADEX-rule answer against the fixed point (the pyradex-rule answer), every model of this rank
        fix_x, fix_s, rx, rs = (d_x, d_surf, x2, s2) if stop_rule == 0 else (x2, s2, d_x, d_surf)
        sig = fix_x > 1e-9
        ex = torch.where(sig, (rx - fix_x).abs() / fix_x, torch.zeros_like(fix_x)).amax(dim=1)
        bright = (fix_s.abs() > 1e-6 * torch.nan_to_num(fix_s.abs(), nan=0.0).amax(dim=1, keepdim=True)) & (fix_s.abs() > 1e-25)
        es = torch.where(bright, (rs - fix_s).abs() / fix_s.abs(), torch.zeros_like(fix_s)).amax(dim=1)
        fin = torch.isfinite(ex) & torch.isfinite(es)
        qs = torch.tensor([0.5, 0.9, 0.99, 0.999], dtype=torch.float64, device=dev)

        def quant(v):
            v = v[fin]
            idx = (qs * (v.numel() - 1)).long()
            return [float(a) for a in torch.sort(v).values[idx]] + [float(v.max())]

        qx, qf = quant(ex), quant(es)
        st_r = (st2 if stop_rule == 0 else d_st)
        it_r = (it2 if stop_rule == 0 else d_it).double()
        extras["stop_radex" if stop_rule == 0 else "stop_pyradex"] = {
            "rule": "RADEX's own conv flag (Fortran matrix(): iter >= 10 and mean |dTex/Tex| of the thick lines < 1e-6), "
                    "dropped by f2py (core.py:910)" if stop_rule == 0 else "pyradex: sum|dx| < 1e-16, iter > 10, cap 200",
            "value": world * n / (ms_o * 1e-3), "unit": "solves/s", "ms_per_step": ms_o, "steps": 1,
            "iters_per_solve": it_o / (world * n), "matrix_iterations_per_s": it_o / (ms_o * 1e-3),
            "roofline_frac": ((it_o / world * F_ITER + n * (F_PRO + F_EPI)) / (ms_o * 1e-3) * 1e-12),   # TFLOP/s; divided by the peak below
            "frac_at_maxiter": float(((st_r & 4) != 0).double().mean()),
            "iters_histogram": {"p10": float(it_r.quantile(0.1)) if n <= (1 << 24) else None, "p50": float(it_r.median()),
                                "p90": float(torch.sort(it_r).values[int(0.9 * (n - 1))]), "max": float(it_r.max())},
            "error_vs_fixed_point": {"what": "per model, RADEX-rule answer against the pyradex-rule answer (sum|dx| < 1e-16) of "
                                             "the same kernels; populations > 1e-9; lines brighter than 1e-6 of the brightest",
                                     "models": int(fin.sum()), "quantiles": [0.5, 0.9, 0.99, 0.999, 1.0],
                                     "pops_rel_err": qx, "flux_rel_err": qf,
                                     "frac_flux_within_1e-5": float((es[fin] < 1e-5).double().mean()),
                                     "frac_pops_within_1e-5": float((ex[fin] < 1e-5).double().mean())}}
        del x2, s2, it2, st2, ex, es, sig, bright
        # (1b) size-independent properties of the whole timed batch (this rank's n models): populations normalised and
        # above RADEX's floor; the answer of a model does not depend on where it sits in the batch (the launches order,
        # park and hand models between kernels by lead-block size: a permuted batch must give the same bits per model)
        ran_ok = (d_st & 3) == 0
        conv = d_st == 0          # stopped by the criterion (a model at the cap need not be normalised in the reference either:
        sums = d_x.sum(dim=1)     # calls whose solution breaks down leave every level on the floor, and 0.3/0.7 of that is kept)
        perm = torch.randperm(n, device=dev, generator=torch.Generator(device=dev).manual_seed(12345))
        keep_in = (d_tk.clone(), d_dens.clone(), d_cd.clone())
        xp, sp_ = torch.empty_like(d_x), torch.empty_like(d_surf)
        itp, stp = torch.empty_like(d_it), torch.empty_like(d_st)
        d_tk.copy_(keep_in[0][perm]); d_dens.copy_(keep_in[1][perm]); d_cd.copy_(keep_in[2][perm])
        launch(opts, sp_, xp, itp, stp)
        torch.cuda.synchronize(dev)
        d_tk.copy_(keep_in[0]); d_dens.copy_(keep_in[1]); d_cd.copy_(keep_in[2])
        same_x = (xp == d_x[perm]) | (torch.isnan(xp) & torch.isnan(d_x[perm]))
        same_s = (sp_ == d_surf[perm]) | (torch.isnan(sp_) & torch.isnan(d_surf[perm]))
        extras["properties"] = {
            "models": n, "what": "the timed 2^20 batch of this rank: sum of the populations, floor, and the same batch solved "
                                 "in a random order (same bits per model wanted: the schedule must not leak into the answer)",
            "converged_models": int(conv.sum()),
            "max_abs_sum_xpop_minus_1_converged": float((sums[conv] - 1.0).abs().max()),
            "models_at_the_cap_with_sum_xpop_off_by_1e-9": int((((sums - 1.0).abs() > 1e-9) & ran_ok & ~conv).sum()),
            "min_xpop": float(d_x[ran_ok].min()),
            "permuted_batch_models_with_identical_populations": int(same_x.all(dim=1).sum()),
            "permuted_batch_models_with_identical_brightness": int(same_s.all(dim=1).sum()),
            "permuted_batch_identical_niter_and_status": int(((itp == d_it[perm]) & (stp == d_st[perm])).sum())}
        del xp, sp_, itp, stp, same_x, same_s, keep_in, perm, sums
        # (2) the sampler the north star shards over the GPUs
        extras["sampler"] = sampler_record(ctx, world, rank, dev, args.sampler_log2w, args.sampler_burn,
                                           args.sampler_steps, 0)
        if world == 1:
            extras["sampler_small"] = sampler_small_records(ctx, dev, 0)
        ctx.set_stream(stream.cuda_stream)

    if rank == 0:
        peaks, peak_src = load_peaks()
        fp64_peak = ctx.fp64_peak_tflops()
        ms_per_step = kern_ms / args.steps
        value = world * n / (ms_per_step * 1e-3)
        e2e_value = world * n / (e2e_ms / args.steps * 1e-3)
        flops_launch = iters_all / world * F_ITER + n * (F_PRO + F_EPI)          # per launch (one rank)
        achieved = flops_launch / (ms_per_step * 1e-3) * 1e-12
        bytes_launch = h2d + d2h                                                  # algorithmic HBM bytes
        traffic, traffic_how = measured_traffic(args.log2n, args.kernel, stop_rule) if not args.keep else (None, "debug subset")
        for k in ("stop_radex", "stop_pyradex"):
            if k in extras:
                extras[k]["roofline_frac"] = extras[k]["roofline_frac"] / fp64_peak
        line = {
            "metric": "LVG solves/s", "value": value, "unit": "solves/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config,
            "kernels": {0: "k_lvg_solve_v2 launches A, B, C (frozen-top caching, ordered by lead-block size) + k_lvg_small<3..7> (cached engines per lead-block size, two models per warp up to 16 levels)",
                        1: "k_lvg_solve_v1", 2: "k_lvg_solve_v2 (no caching)",
                        3: "k_lvg_solve_v2 (frozen-top caching, single launch)",
                        4: "k_lvg_solve_v2 (frozen-top caching, two launches ordered by lead-block size)"}[args.kernel],
            "iters_per_solve": iters_all / (world * n),
            "matrix_iterations_per_s": iters_all / (ms_per_step * 1e-3),
            "frac_iterations_cached": cache_stats[0] / max(1, total_iters),
            "captures_per_solve": cache_stats[1] / n, "invalidations_per_solve": cache_stats[2] / n,
            "frac_at_maxiter": float((status_host & 4).astype(bool).mean()),
            "frac_nonfinite": float((status_host & 8).astype(bool).mean()),
            "e2e": None if args.no_e2e else {"value": e2e_value, "unit": "solves/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches_timed,
            "roofline": {"bound": "fp64", "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s",
                         "frac": achieved / fp64_peak,
                         "traffic": traffic,
                         "traffic_unit": "bytes per step, all launches; algorithmic bytes = h2d + d2h = %d" % bytes_launch,
                         "traffic_source": traffic_how, "kernel_sources": source_hash(),
                         "peak_source": "rb_fp64_peak DFMA probe measured in this run (MEASURED_PEAKS.json has no FP64 "
                                        "figure); nominal 148 SM x 64 FMA x 2 x 1.965 GHz = 37.2",
                         "flops_per_iter": F_ITER,
                         "hbm": {"achieved_gbs": bytes_launch / (ms_per_step * 1e-3) * 1e-9,
                                 "peak_gbs": peaks.get("hbm_gbs"), "peak_source": peak_src}},
            "clocks": sampler.summary(),
            "wall_s_timed_region": t_wall,
        }
        line.update(extras)
        if not args.no_cpu and not args.keep:
            if stop_rule == 0 and npar > 0 and args.abs_tol == 1e-16:
                line["parity"] = parity_record(npar, tk, nh2, cd, par_arrays)
            if world == 1:
                v, sample, dt, _ = cpu_reference(tk, nh2, cd, stop_rule, args.cpu_seconds, 1)
                line["cpu_baseline"] = {"value": v, "unit": "solves/s", "cores": 1, "kind": "port",
                                        "sample": "first %d draws of the same sweep, 1 thread, %.1f s; oracle/ is the "
                                                  "bit-exact C restatement of the reference" % (sample, dt)}
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
