#!/usr/bin/env python
"""bench.py — marker x trait LOD tests/sec on the BXD-shape bulkscan (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
                    [--workload alt-grid|null-grid|null-exact|scaled-null-exact|perms] [--dump-outputs DIR]

One "step" = one full scan call through the C-ABI (rotation by U' -> per-trait null statistics / Brent
fit -> marker operand -> fused DMMA scan with the LOD epilogue) on synthetic data (SURVEY 8d):

  alt-grid (default)  BASELINE.json configs[2], the north-star target: n=79, p=7321, m=35554, 10-point grid
  null-grid           configs[1]: same shape, bulkscan default method (the reference's published 2.11 s)
  null-exact          same shape, per-trait REML Brent + per-trait-weight scan (bulkscan_null)
  scaled-null-exact   configs[4]: n=1000, p=100000, m=20000, c=3, REML
  perms               configs[3]: scan, 1 trait x 10000 permutations x 7321 markers

The kinship eigendecomposition is setup (one-off, timed separately and reported as `setup_ms`).

  value      : whole-job tests/s, inputs resident in HBM, outputs left in HBM
  e2e        : the same call through the C-ABI with HOST (pinned) buffers: H2D of Y,G,Covar,U,lambda
               and D2H of the outputs inside the timed region
  roofline   : the fused scan kernel against the measured FP64 tensor peak (profiles/fp64_peak_r01.json)
  cpu_baseline: the CPU oracle (numpy restatement of the reference algorithm), all host cores, on a
               bounded sample of the same workload

N > 1 (torchrun, one rank per GPU): traits (bulkscan) or permutations (scan) are sharded across ranks
(strong scaling: the problem is fixed), G/U are replicated, there is no data-path collective; NCCL is
used for the barrier and the max-over-ranks time.

--dump-outputs DIR (one GPU) writes the results of the last timed step as DIR/<name>.npy (float64), named and
oriented as the Python API returns them (markers x traits / permutations); an output of more than DUMP_ENTRIES
entries is cut to a fixed, seeded sample of its traits (permutations) and markers.  The inputs are seeded too, so two
builds run with the same arguments can be compared output for output.
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
for sub in ("bulklmm.jl_b200", "oracle"):
    sys.path.insert(0, os.path.join(ROOT, sub))
sys.dont_write_bytecode = True  # the source tree may be read-only: nothing is cached there

import numpy as np  # noqa: E402

GRID = np.arange(10) / 10.0  # 0.0:0.1:0.9, src/bulkscan.jl:82
README_REF = {"value": 1.23e8, "what": "reference README.md:336-339: bulkscan null-grid, 2.112 s, 16 Julia threads, "
                                       "48x Xeon Silver 4214 (other hardware)"}
METRIC = "marker x trait LOD tests/sec, BXD-shape bulkscan"

# name -> shape, method, covariate columns (incl. intercept), opts, flops per test / n, outputs, cpu sample
WORKLOADS = {
    "alt-grid": dict(n=79, p=7321, m=35554, c=1, method="alt-grid", opts=dict(h2_grid=GRID), fmult=len(GRID),
                     cfg="BASELINE.json configs[2]", outputs="L and h2_panel (p x m f64 each)", cpu_m=8192),
    "null-grid": dict(n=79, p=7321, m=35554, c=1, method="null-grid", opts=dict(h2_grid=GRID), fmult=1,
                      cfg="BASELINE.json configs[1]", outputs="L (p x m f64) and h2_null_list", cpu_m=35554),
    "null-exact": dict(n=79, p=7321, m=35554, c=1, method="null-exact", opts=dict(reml=True, prior_variance=0.0),
                       fmult=3, cfg="BXD shape, bulkscan_null", outputs="L (p x m f64) and h2_null_list", cpu_m=1024),
    "scaled-null-exact": dict(n=1000, p=100000, m=20000, c=3, method="null-exact",
                              opts=dict(reml=True, prior_variance=0.0), fmult=5, cfg="BASELINE.json configs[4]",
                              outputs="L (p x m f64) and h2_null_list", cpu_m=16),
    "perms": dict(n=79, p=7321, m=10001, c=1, method="perms", opts=dict(prior_variance=0.0), fmult=1,
                  cfg="BASELINE.json configs[3]", outputs="lod, L_perms (p x nperms f64), per-permutation max", cpu_m=10000),
}
DUMP_ENTRIES = 1 << 21  # 16 MB of float64; no workload has more than two outputs this large, so a dump is <= 64 MB


def fp64_peak():
    path = os.path.join(ROOT, "profiles", "fp64_peak_r01.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return d["cublas_dgemm_tflops_sustained"], ("measured: cuBLAS DGEMM 8192^3 sustained on this pool "
                                                    "(profiles/fp64_peak_r01.json); MEASURED_PEAKS.json has no FP64 entry")
    return 37.0, "fallback: B200 datasheet FP64 tensor 37 TFLOP/s (no measured file)"


# ------------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                mx = max(mx, float(f[1]))
                if t0 - 0.05 <= ts <= t1 + 0.15:
                    sm.append(float(f[0]))
                    for nm, v in zip(names, f[3:7]):
                        if v.lower().startswith("active"):
                            reasons.add(nm)
            except ValueError:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# synthetic inputs (SURVEY 8d): same generator and seeds on every rank
# ------------------------------------------------------------------------------------------------
def make_inputs(w, m_limit=None, seed=0):
    from blmm_b200 import synth
    n, p, c = w["n"], w["p"], w["c"]
    m = w["m"] if m_limit is None else min(m_limit, w["m"])
    G = synth.make_geno(n, p, seed=p)
    K = synth.calc_kinship_host(G)
    if w["method"] == "perms":
        Y = synth.make_pheno(G, K, 1112, seed=35554)[:, 1111:1112]  # trait column 1112 (SURVEY C4)
    else:
        Y = synth.make_pheno(G, K, m, seed=w["m"] + seed)
    Cv = np.ones((n, 1)) if c == 1 else np.hstack([np.ones((n, 1)), synth.make_covar(n)[:, :c - 1]])
    return Y, G, K, Cv


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle, threaded over trait blocks like the reference (Threads.@threads over nb blocks
# with BLAS pinned to one thread, src/bulkscan.jl:252-286)
# ------------------------------------------------------------------------------------------------
def cpu_baseline(name, repeats=1, warmup=0):
    """Time the oracle on a bounded sample of the workload (inputs generated once); returns the mean of
    `repeats` timed runs after `warmup` untimed ones."""
    import blmm_oracle as orc
    from blmm_b200 import synth
    from concurrent.futures import ThreadPoolExecutor
    try:
        from threadpoolctl import threadpool_limits
    except Exception:  # pragma: no cover
        threadpool_limits = None
    w = WORKLOADS[name]
    cores = os.cpu_count() or 1
    sample_m = w["cpu_m"]
    Y, G, K, Cv = make_inputs(w, m_limit=sample_m)
    n, p = G.shape
    Ut, lam = orc.decompose(K)
    covar = None if w["c"] == 1 else Cv[:, 1:]
    if w["method"] == "perms":
        perm = synth.make_perm_indices(n, sample_m, 0)
        run = lambda: orc.scan(Y, G, K, permutation_test=True, perm_idx=perm, Ut=Ut, lam=lam)  # BLAS-threaded GEMM
        tests = p * (sample_m + 1)
        what = f"{sample_m} of 10000 permutations, OpenBLAS threads"
    else:
        nb = max(1, min(cores * 2, sample_m // 4))
        edges = np.linspace(0, sample_m, nb + 1).astype(int)
        if w["method"] == "alt-grid":
            fn = lambda Ys: orc.bulkscan_alt_grid(Ys, G, K, GRID, Covar=covar, Ut=Ut, lam=lam)
        elif w["method"] == "null-grid":
            fn = lambda Ys: orc.bulkscan_null_grid(Ys, G, K, GRID, Covar=covar, Ut=Ut, lam=lam)
        else:
            fn = lambda Ys: orc.bulkscan_null(Ys, G, K, Covar=covar, reml=True, prior_variance=0.0, Ut=Ut, lam=lam)

        def pool():
            with ThreadPoolExecutor(cores) as ex:
                return list(ex.map(lambda i: fn(Y[:, edges[i]:edges[i + 1]]), range(nb)))

        def run():
            if threadpool_limits is not None:
                with threadpool_limits(limits=1):
                    pool()
            else:
                pool()

        tests = p * sample_m
        what = f"first {sample_m} of {w['m']} synthetic traits, threaded over {nb} trait blocks"
    times = []
    for i in range(warmup + repeats):
        t0 = time.perf_counter()
        run()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    dt = float(np.mean(times))
    return {"value": tests / dt, "unit": "tests/s", "cores": cores, "kind": "port",
            "sample": f"{name}, all {p} markers x {what}, {dt:.2f} s per run; numpy oracle (CPU restatement of the "
                      f"reference algorithm; the Julia reference cannot run: no Julia in the image)",
            "seconds": dt}


def workload_config(name, gpus):
    w = WORKLOADS[name]
    unit = "permutations" if w["method"] == "perms" else "traits"
    return {"workload": f"{'scan with permutations' if w['method'] == 'perms' else 'bulkscan ' + w['method']}, "
                        f"n={w['n']} p={w['p']} {'nperms+1' if w['method'] == 'perms' else 'm'}={w['m']}, c={w['c']}"
                        f"{', h2 grid 0:0.1:0.9, ML' if 'grid' in w['method'] else ''} ({w['cfg']})",
            "n": w["n"], "p": w["p"], "m": w["m"], "c": w["c"], "outputs": w["outputs"],
            "sharding": f"{unit} over {gpus} GPU(s), G/U replicated, no data-path collective",
            "l2": "explicit 512 MB L2 flush between timed steps (each step also writes > L2 of output)"}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path = the oracle port (Julia is not
    installed, so oracle/_ref does not exist), all host cores, bounded sample per step."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    last = cpu_baseline(args.workload, repeats=args.steps, warmup=args.warmup)
    dt, value = last["seconds"], last["value"]
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "tests/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args.workload, args.gpus),
            "cpu_baseline": {"value": value, "unit": "tests/s", "cores": last["cores"], "kind": "port",
                             "sample": last["sample"]},
            "e2e": {"value": value, "unit": "tests/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="alt-grid", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer e2e leg")
    ap.add_argument("--no-other", action="store_true", help="skip the short runs of the other configs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's results (sampled above DUMP_ENTRIES entries) as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's results; it does not apply to --impl reference")
    if args.dump_outputs and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        ap.error("--dump-outputs needs one GPU: at N > 1 each rank holds only its shard of the results")
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    from blmm_b200 import Engine, synth, _lib as L

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))

    def wait_for_rank0(tag):
        """CPU-side wait (the rendezvous store, no GPU work) for the phases in which rank 0 drives every GPU through
        ONE multi-GPU context: the other ranks must not sit in an NCCL barrier meanwhile — a spinning kernel on their
        GPU would time-slice with rank 0's work there."""
        if world == 1:
            return
        import datetime
        store = dist.distributed_c10d._get_default_store()
        if rank == 0:
            store.set(tag, "1")
        else:
            store.wait([tag], datetime.timedelta(seconds=3600))
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    METHODS = {"alt-grid": L.METHOD_ALT_GRID, "null-grid": L.METHOD_NULL_GRID, "null-exact": L.METHOD_NULL_EXACT,
               "perms": L.METHOD_NULL_EXACT}

    eng = Engine(local)
    stream = torch.cuda.ExternalStream(eng.stream, device=dev)
    eng.set_profiling(True)
    flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def colmajor(a):
        return torch.from_numpy(np.ascontiguousarray(np.asarray(a, dtype=np.float64).T))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        eng.sync()

    class Job:
        """One workload resident on this rank's GPU: step() = one C-ABI call with device pointers."""

        def __init__(self, name):
            w = self.w = WORKLOADS[name]
            self.name = name
            n, p, c = w["n"], w["p"], w["c"]
            Y, G, K, Cv = make_inputs(w)
            self.K = K
            self.perms = w["method"] == "perms"
            t0 = time.perf_counter()
            U, lam, _ = eng.decompose(K)  # setup: cuSOLVER syevd
            self.setup_ms = (time.perf_counter() - t0) * 1e3
            cols = w["m"] - 1 if self.perms else w["m"]  # sharded units: traits or permutations
            self.cols = cols
            j0, j1 = rank * cols // world, (rank + 1) * cols // world
            self.j0, self.j1 = j0, j1
            self.ml = ml = j1 - j0
            self.tests_total = p * w["m"]
            # full host inputs (the e2e leg passes them whole to a context that shards them itself)
            self.host_full = [Y, G, Cv, U, lam]
            self.h = [colmajor(Y if self.perms else Y[:, j0:j1]), colmajor(G), colmajor(Cv), colmajor(U),
                      torch.from_numpy(lam.copy())]
            self.d = [t.to(dev) for t in self.h]
            self.method = METHODS[w["method"]]
            self.alt = alt = w["method"] == "alt-grid"
            self.out_shapes = [(ml, p), (ml, p) if alt else (ml,)]
            if self.perms:
                self.perm_full = synth.make_perm_indices(n, cols, 0)
                self.hperm = torch.from_numpy(np.ascontiguousarray(self.perm_full[:, j0:j1].T))
                self.dperm = self.hperm.to(dev)
                self.out_shapes = [(ml, p), (ml,), (p,), (2,)]  # L_perms, max, lod, (sigma2, h2)
                self.gathered_max = torch.empty(world * ((cols + world - 1) // world), dtype=torch.float64, device=dev)
                self.max_pad = torch.zeros((cols + world - 1) // world, dtype=torch.float64, device=dev)
            self.dout = [torch.empty(s, dtype=torch.float64, device=dev) for s in self.out_shapes]
            self.opts, self._keep = eng.make_opts(method=self.method, mem_space=L.MEM_DEVICE, **w["opts"])
            self.pr = eng.make_problem(n, p, 1 if self.perms else ml, c, *[t.data_ptr() for t in self.d])
            self.flops = 2.0 * n * p * (ml + (1 if self.perms else 0)) * w["fmult"]
            self.out_bytes = 8.0 * sum(int(np.prod(s)) for s in self.out_shapes[:2])

        def outputs(self):
            """(name, device tensor) of each result a caller of the path receives, named as in blmm_b200's results;
            matrices are traits (permutations) x markers here, the transpose of the caller's layout"""
            if self.perms:
                Lp, mx, lod, s = self.dout
                return [("L_perms", Lp), ("max_lod", mx), ("lod", lod), ("sigma2_e", s[:1]), ("h2_null", s[1:])]
            return [("L", self.dout[0]), ("h2_panel" if self.alt else "h2_null_list", self.dout[1])]

        @staticmethod
        def call(E, perms, pr, opts, outs, perm_ptr, nperms):
            if perms:
                E.scan_perms_raw(pr, opts, perm_ptr, nperms, outs[2], outs[0], outs[1], outs[3], outs[3] + 8)
            else:
                E.bulkscan_raw(pr, opts, outs[0], outs[1])

        def step(self):
            self.call(eng, self.perms, self.pr, self.opts, [t.data_ptr() for t in self.dout],
                      self.dperm.data_ptr() if self.perms else None, self.ml)
            if self.perms and world > 1:
                # configs[3]: NCCL gather of the per-permutation maximum LODs (what get_thresholds consumes), on the
                # library's stream, inside the timed region
                with torch.cuda.stream(stream):
                    self.max_pad[: self.ml].copy_(self.dout[1], non_blocking=True)
                    dist.all_gather_into_tensor(self.gathered_max, self.max_pad)

        def timed(self, steps, warmup):
            for _ in range(warmup):
                self.step()
                eng.sync()
                torch.cuda.synchronize(dev)
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            scan_ms = []
            barrier()
            l0, w0 = eng.launch_count, time.time()
            for a, b in evs:
                with torch.cuda.stream(stream):
                    flush.zero_()  # L2 flush, outside the step's event pair
                a.record(stream)
                self.step()
                b.record(stream)
                eng.sync()
                torch.cuda.synchronize(dev)
                scan_ms.append(eng.last_scan_ms())
            barrier()
            w1 = time.time()
            total_ms = sum(a.elapsed_time(b) for a, b in evs)
            local_ms = total_ms
            if world > 1:
                tt = torch.tensor([total_ms], dtype=torch.float64, device=dev)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                total_ms = float(tt.item())
            return dict(total_ms=total_ms, local_ms=local_ms, scan_ms=float(np.mean(scan_ms)),
                        launches=eng.launch_count - l0, wall=(w0, w1))

        def e2e(self, E, steps):
            """The call a user of the boundary makes: ONE blocking C-ABI call on the WHOLE problem with HOST buffers
            (H2D of Y, G, Covar, U, lambda and D2H of every result inside the timed region), on a context that owns all
            `world` GPUs (blmm_create_multi shards the traits / permutations itself).  Timed twice: with ordinary
            pageable numpy arrays (what the Julia shim and the Python mirror pass) and with pinned buffers."""
            w = self.w
            n, p, c = w["n"], w["p"], w["c"]
            Y, G, Cv, U, lam = self.host_full
            mfull = self.cols if self.perms else w["m"]
            shapes = ([(mfull, p), (mfull,), (p,), (2,)] if self.perms else
                      [(mfull, p), (mfull, p) if self.alt else (mfull,)])
            hopts, keep2 = E.make_opts(method=self.method, mem_space=L.MEM_HOST, **w["opts"])
            res = {}
            for kind in ("pageable", "pinned"):
                ins = [colmajor(Y), colmajor(G), colmajor(Cv), colmajor(U), torch.from_numpy(lam.copy())]
                outs = [torch.zeros(s, dtype=torch.float64) for s in shapes]  # zeros: pages touched before timing
                perm = torch.from_numpy(np.ascontiguousarray(self.perm_full.T)) if self.perms else None
                if kind == "pinned":
                    ins = [t.pin_memory() for t in ins]
                    outs = [t.pin_memory() for t in outs]
                    perm = perm.pin_memory() if self.perms else None
                hpr = E.make_problem(n, p, 1 if self.perms else mfull, c, *[t.data_ptr() for t in ins])
                optr = [t.data_ptr() for t in outs]
                pptr = perm.data_ptr() if self.perms else None
                self.call(E, self.perms, hpr, hopts, optr, pptr, mfull)  # warm (allocates staging)
                per = []
                for _ in range(steps):
                    t1 = time.perf_counter()
                    self.call(E, self.perms, hpr, hopts, optr, pptr, mfull)  # blocking: results are on the host
                    per.append((time.perf_counter() - t1) * 1e3)
                h2d = sum(t.numel() * t.element_size() for t in ins) + (perm.numel() * 4 if self.perms else 0)
                d2h = sum(t.numel() * 8 for t in outs)
                # the host-buffer result equals this rank's device-resident slab bit for bit
                assert torch.equal(outs[0][self.j0:self.j1], self.dout[0].cpu()), "host-buffer result differs"
                if self.alt:
                    assert torch.equal(outs[1][self.j0:self.j1], self.dout[1].cpu()), "host-buffer h2 panel differs"
                ms = float(np.mean(per))
                res[kind] = {"ms_per_step": ms, "ms_each_step": [round(x, 2) for x in per],
                             "value": self.tests_total / (ms * 1e-3)}
                del ins, outs
            idx = self.alt and p * mfull >= 1e8  # the library decides the encoding on the whole panel
            pcie_d2h = d2h - (p * mfull * 7 if idx else 0)
            head = res["pinned"]
            return {"value": head["value"], "unit": "tests/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(pcie_d2h), "host_output_bytes_per_step": int(d2h),
                    "ms_per_step": head["ms_per_step"], "ms_each_step": head["ms_each_step"], "steps": steps,
                    "buffers": "pinned", "n_gpus_in_call": E.device_count,
                    "pageable": res["pageable"],
                    "note": "ONE blocking C-ABI call on the whole problem per step, wall clock, host buffers; value = "
                            "page-locked host buffers as the bench contract prescribes (direct DMA into the caller's "
                            "arrays); `pageable` = the same call on ordinary numpy arrays, what Julia / numpy callers pass "
                            "unless they register their arrays (the library stages those through its pinned ring and "
                            "drain threads: one extra pass over host memory, so it is bound by the host's memory "
                            "bandwidth and stops scaling with the GPU count; DESIGN.md section 6).  "
                            "At n_gpus > 1 the call runs on a blmm_create_multi context that shards the traits / "
                            "permutations over all GPUs itself, each GPU writing its slab of the caller's arrays over "
                            "its own PCIe link.  alt-grid: the copy-back overlaps the scan in trait-tile chunks; with "
                            ">= 1e8 panel entries per GPU the h2 panel crosses PCIe as one-byte grid indices "
                            "(d2h_bytes_per_step = bytes over PCIe; host_output_bytes_per_step = the caller's Float64 arrays)"}

    def pcie_rates():
        """measured pinned copy rates of this rank's GPU (1 GiB, best of 3): the floor of any host-buffer call"""
        nb = 1 << 30
        hbuf = torch.empty(nb, dtype=torch.uint8).pin_memory()
        dbuf = torch.empty(nb, dtype=torch.uint8, device=dev)
        out = {}
        for nm, (dst, src) in (("d2h_gbs", (hbuf, dbuf)), ("h2d_gbs", (dbuf, hbuf))):
            best = 1e9
            for _ in range(3):
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                dst.copy_(src, non_blocking=True)
                torch.cuda.synchronize(dev)
                best = min(best, time.perf_counter() - t0)
            out[nm] = nb / best / 1e9
        return out

    def dump_outputs(job, outdir):
        """job's results as outdir/<name>.npy in the caller's orientation (markers x traits); a matrix of more than
        DUMP_ENTRIES entries is cut to the same seeded, sorted sample of its rows and columns on every run"""
        os.makedirs(outdir, exist_ok=True)
        for name, t in job.outputs():
            if t.dim() == 2 and t.numel() > DUMP_ENTRIES:
                r, c = t.shape
                kc = min(c, DUMP_ENTRIES // min(r, 256))
                kr = min(r, DUMP_ENTRIES // kc)
                rng = np.random.default_rng(0)
                rows = torch.from_numpy(np.sort(rng.choice(r, kr, replace=False))).to(dev)
                cols = torch.from_numpy(np.sort(rng.choice(c, kc, replace=False))).to(dev)
                t = t.index_select(0, rows).index_select(1, cols)
            np.save(os.path.join(outdir, name + ".npy"), np.ascontiguousarray(t.cpu().numpy().T))

    def run_e2e(job, steps):
        """rank 0 drives all `world` GPUs through one context; the other ranks wait on the CPU barrier"""
        out = None
        if rank == 0:
            try:
                if world > 1 and torch.cuda.device_count() >= world:
                    E = Engine(devices=list(range(world)))
                else:
                    E = eng
                out = job.e2e(E, steps)
                if E is not eng:
                    E.close()
                if world > 1 and E is eng:
                    out["note"] += "  [only this rank's GPU was visible: single-GPU call]"
            except (RuntimeError, MemoryError) as ex:  # pinned allocation of a very large result can fail on small hosts
                out = {"value": None, "unit": "tests/s", "error": str(ex)[:200]}
        wait_for_rank0("blmm_e2e_done")
        return out

    job = Job(args.workload)
    w = job.w
    t0 = time.perf_counter()
    eng.decompose(job.K)
    setup_ms_warm = (time.perf_counter() - t0) * 1e3

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    r = job.timed(args.steps, args.warmup)
    clocks = sampler.stop(*r["wall"]) if rank == 0 else None
    value = job.tests_total * args.steps / (r["total_ms"] * 1e-3)
    if args.dump_outputs:
        dump_outputs(job, args.dump_outputs)

    # ---- roofline of the dominant kernel (the fused scan), measured live with CUDA events inside the library
    peak, peak_src = fp64_peak()
    hbm = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"] if os.path.exists(
        os.path.join(ROOT, "MEASURED_PEAKS.json")) else 6650.0
    t_tensor = job.flops / (peak * 1e12)
    t_hbm = job.out_bytes / (hbm * 1e9)
    ach = job.flops / (r["scan_ms"] * 1e-3) / 1e12
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "scan_traffic_r02.json")
    if not os.path.exists(tpath):
        tpath = os.path.join(ROOT, "profiles", "scan_traffic_r01.json")
    if os.path.exists(tpath) and world == 1:
        traffic = json.load(open(tpath)).get(args.workload)
    kname = ("blmm::scan_stream_kernel (FP64 DMMA.8x8x4, K-streamed TMA bulk copies)" if "exact" in args.workload
             else "blmm::scan_kernel (FP64 DMMA.8x8x4, TMA bulk copies)")
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    dmma_issue = 148 * 4 * 512 / 16 * sm_mhz * 1e6 / 1e12  # SMs x sub-partitions x flop per DMMA.8x8x4 / 16 clk
    roofline = {"bound": "tensor" if t_tensor >= t_hbm else "hbm", "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                "frac": ach / peak, "traffic": traffic, "kernel": kname, "kernel_ms": r["scan_ms"],
                "kernel_share_of_step": r["scan_ms"] * args.steps / r["local_ms"],
                "algorithmic_flops_per_launch": job.flops, "algorithmic_output_bytes_per_launch": job.out_bytes,
                "t_roof_ms": max(t_tensor, t_hbm) * 1e3, "frac_of_t_roof": max(t_tensor, t_hbm) * 1e3 / r["scan_ms"],
                "frac_vs_dmma_issue": ach / dmma_issue, "dmma_issue_tflops": dmma_issue,
                "peak_source": peak_src, "hbm_gbs": hbm}

    e2e = None
    if not args.no_e2e:
        pcie = pcie_rates() if rank == 0 else None
        e2e = run_e2e(job, max(2, min(args.steps, 5)))
        if rank == 0 and e2e is not None:
            e2e["pcie_measured"] = pcie
            if pcie and e2e.get("d2h_bytes_per_step"):
                nd = e2e.get("n_gpus_in_call", 1)
                e2e["pcie_floor_ms"] = (e2e["d2h_bytes_per_step"] / nd / (pcie["d2h_gbs"] * 1e9) +
                                        e2e["h2d_bytes_per_step"] / (pcie["h2d_gbs"] * 1e9)) * 1e3

    # ---- the other BASELINE.json configs, device-resident, a few steps each, at this N (context for the headline
    # number, not part of it): configs[1] null-grid, configs[3] permutations (with the NCCL gather of the maxima at
    # N > 1), configs[4] the scaled null-exact problem, and null-exact at BXD shape
    other = None
    if not args.no_other and args.workload == "alt-grid":
        other = {}
        del job.dout, job.d
        torch.cuda.empty_cache()
        names = ("null-grid", "null-exact", "perms", "scaled-null-exact") if world == 1 else ("perms", "scaled-null-exact")
        for nm in names:
            j2 = Job(nm)
            r2 = j2.timed(3 if nm.startswith("scaled") else 5, 3)
            k = 3 if nm.startswith("scaled") else 5
            other[nm] = {"workload": workload_config(nm, world)["workload"], "ms_per_step": r2["total_ms"] / k,
                         "tests_per_s": j2.tests_total * k / (r2["total_ms"] * 1e-3), "scan_kernel_ms": r2["scan_ms"],
                         "scan_kernel_tflops_this_rank": j2.flops / (r2["scan_ms"] * 1e-3) / 1e12,
                         "scan_kernel_frac_of_peak": j2.flops / (r2["scan_ms"] * 1e-3) / 1e12 / peak}
            if nm == "perms" and world > 1:
                other[nm]["collective"] = "NCCL all_gather of the per-permutation maximum LODs inside the timed step"
            del j2
            torch.cuda.empty_cache()

    cpu = None
    if rank == 0 and not args.no_cpu and world == 1:
        cpu = cpu_baseline(args.workload)
        cpu.pop("seconds", None)

    if rank == 0:
        vs = value / README_REF["value"] if args.workload == "null-grid" else None
        line = {"metric": METRIC, "value": value, "unit": "tests/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": r["total_ms"] / args.steps, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": vs, "dtype": "f64", "data": "synthetic",
                "config": workload_config(args.workload, world), "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
                "gpu_launches": int(r["launches"]), "clocks": clocks, "other_workloads": other,
                "setup_ms": {"eigendecomposition_first_call": job.setup_ms, "eigendecomposition_warm": setup_ms_warm},
                "reference_published": README_REF}
        print(json.dumps(line), flush=True)
    if world > 1:
        wait_for_rank0("blmm_line_printed")
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
