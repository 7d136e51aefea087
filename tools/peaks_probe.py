"""Per-trait peaks (blmm_bulkscan_peaks) against the dense scan (blmm_bulkscan) on one GPU.

    python tools/peaks_probe.py [--steps 10] [--warmup 3] [--out FILE.json]

For BXD alt-grid, BXD null-grid and the configs[4] null-exact shape (bench.py's WORKLOADS and seeded inputs):
  * the device-resident step of each call (CUDA events on the library's stream, the 512 MB L2 flush of bench.py
    between steps, outside the event pair), and the scan kernel's own time (blmm_last_scan_ms);
  * one blocking host-buffer call of each, with pinned and with ordinary (pageable) arrays, after one warm-up call;
  * a check that the peaks are the findmax of the dense L, bit for bit.
The card's name and power limit are read with a read-only nvidia-smi query and printed with the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402

import bench  # noqa: E402  (puts the package and the oracle on sys.path)

SHAPES = ("alt-grid", "null-grid", "scaled-null-exact")


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out
    except Exception as e:  # the numbers are still printed; the card line says why it is missing
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--out", help="also write the results as JSON to this file")
    args = ap.parse_args()

    import torch
    from blmm_b200 import Engine, _lib as L

    dev = torch.device("cuda:0")
    eng = Engine(0)
    stream = torch.cuda.ExternalStream(eng.stream, device=dev)
    eng.set_profiling(True)
    flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=dev)
    methods = {"alt-grid": L.METHOD_ALT_GRID, "null-grid": L.METHOD_NULL_GRID, "null-exact": L.METHOD_NULL_EXACT}

    def colmajor(a):
        return torch.from_numpy(np.ascontiguousarray(np.asarray(a, dtype=np.float64).T))

    def timed(step):
        for _ in range(args.warmup):
            step()
            eng.sync()
        torch.cuda.synchronize(dev)
        ms, scan = [], []
        for _ in range(args.steps):
            with torch.cuda.stream(stream):
                flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            step()
            b.record(stream)
            eng.sync()
            torch.cuda.synchronize(dev)
            ms.append(a.elapsed_time(b))
            scan.append(eng.last_scan_ms())
        return {"step_ms": round(float(np.median(ms)), 3), "step_ms_each": [round(x, 3) for x in ms],
                "scan_kernel_ms": round(float(np.median(scan)), 3)}

    def host_call(call):
        call()  # warm: staging buffers
        t = time.perf_counter()
        call()
        return round((time.perf_counter() - t) * 1e3, 2)

    results = {"card": card(), "l2": "512 MB flush between timed device steps", "shapes": {}}
    for name in args.shapes.split(","):
        w = bench.WORKLOADS[name]
        n, p, m, c = w["n"], w["p"], w["m"], w["c"]
        method = methods[w["method"]]
        alt = method == L.METHOD_ALT_GRID
        Y, G, K, Cv = bench.make_inputs(w)
        U, lam, _ = eng.decompose(K)
        hin = [colmajor(Y), colmajor(G), colmajor(Cv), colmajor(U), torch.from_numpy(lam.copy())]
        din = [t.to(dev) for t in hin]
        pr = eng.make_problem(n, p, m, c, *[t.data_ptr() for t in din])
        dopts, keep = eng.make_opts(method=method, mem_space=L.MEM_DEVICE, **w["opts"])
        Ld = torch.empty((m, p), dtype=torch.float64, device=dev)
        Hd = torch.empty((m, p) if alt else (m,), dtype=torch.float64, device=dev)
        pl = torch.empty(m, dtype=torch.float64, device=dev)
        pm = torch.empty(m, dtype=torch.int64, device=dev)
        ph = torch.empty(m, dtype=torch.float64, device=dev)
        r = {"shape": f"n={n} p={p} m={m} c={c}, {w['method']}", "dense_output_bytes": 8 * p * m * (2 if alt else 1)}
        r["dense_device"] = timed(lambda: eng.bulkscan_raw(pr, dopts, Ld.data_ptr(), Hd.data_ptr()))
        r["peaks_device"] = timed(lambda: eng.bulkscan_peaks_raw(pr, dopts, pl.data_ptr(), pm.data_ptr(), ph.data_ptr()))
        # the peaks are the findmax of the dense L (rows of Ld are traits), bit for bit
        b = Ld.view(torch.int64)
        key = torch.where(b >= 0, b, b ^ 0x7FFFFFFFFFFFFFFF)
        key = torch.where(torch.isnan(Ld), torch.full_like(key, 0x7FFFFFFFFFFFFFFF), key)
        idx = torch.argmax(key, dim=1)
        del key, b
        ar = torch.arange(m, device=dev)
        ok = torch.equal(idx, pm) and torch.equal(Ld[ar, idx].view(torch.int64), pl.view(torch.int64))
        ok = ok and torch.equal((Hd[ar, idx] if alt else Hd).view(torch.int64), ph.view(torch.int64))
        r["peaks_equal_findmax_of_dense"] = bool(ok)
        del Ld, Hd
        torch.cuda.synchronize(dev)
        hopts, keep2 = eng.make_opts(method=method, mem_space=L.MEM_HOST, **w["opts"])
        for kind in ("pinned", "pageable"):
            ins = [t.pin_memory() for t in hin] if kind == "pinned" else hin
            hpr = eng.make_problem(n, p, m, c, *[t.data_ptr() for t in ins])
            outs = [torch.zeros(m, dtype=torch.float64), torch.zeros(m, dtype=torch.int64),
                    torch.zeros(m, dtype=torch.float64)]
            if kind == "pinned":
                outs = [t.pin_memory() for t in outs]
            r[f"peaks_host_{kind}_ms"] = host_call(
                lambda: eng.bulkscan_peaks_raw(hpr, hopts, *[t.data_ptr() for t in outs]))
            dl = torch.zeros((m, p), dtype=torch.float64)
            dh = torch.zeros((m, p) if alt else (m,), dtype=torch.float64)
            if kind == "pinned":
                dl, dh = dl.pin_memory(), dh.pin_memory()
            r[f"dense_host_{kind}_ms"] = host_call(lambda: eng.bulkscan_raw(hpr, hopts, dl.data_ptr(), dh.data_ptr()))
            assert torch.equal(outs[1], pm.cpu()), "host-buffer peaks differ from the device-resident call"
            del dl, dh, ins, outs
        print(json.dumps({name: r}), flush=True)
        results["shapes"][name] = r
    print(json.dumps({"card": results["card"]}), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
