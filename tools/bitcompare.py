"""Bit-for-bit comparison of two builds of libblmm_b200 on every output of the library's scans and fits.

    python tools/bitcompare.py LIB_A LIB_B [--out DIR]

Each build runs in its own process (BLMM_B200_LIB selects it) on the same seeded inputs, which this process generates
once.  The shapes are the grid-edge cases of tests/test_gpu_grid_edges.py (CASES and CEILING_SHAPES, read from that
file), which between them reach every trait-statistics / marker-operand / scan-kernel path of the grid scans, and
scans with permutations at n = 79 and n = 137, through the fused single-trait prologue and the separate kernels
(BLMM_B200_NO_CHAIN).  Called: bulkscan (null-grid, alt-grid, null-exact), bulkscan_peaks (the same three),
grid_loglik, fit_h2, scan_null, scan_alt and scan_perms.  A refactor that must not change the arithmetic should report
every output identical; the exit code is 1 otherwise.  Needs one GPU."""
from __future__ import annotations

import argparse
import ast
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "bulklmm.jl_b200"))


def grid_edge_shapes():
    """CASES + CEILING_SHAPES of tests/test_gpu_grid_edges.py, evaluated from its source (the test module itself
    imports the oracle and pytest)."""
    path = os.path.join(ROOT, "tests", "test_gpu_grid_edges.py")
    shapes = {}
    for node in ast.parse(open(path).read()).body:
        name = node.targets[0].id if isinstance(node, ast.Assign) and isinstance(node.targets[0], ast.Name) else None
        if name in ("CASES", "CEILING_SHAPES"):
            shapes[name] = eval(compile(ast.Expression(node.value), path, "eval"), {"dict": dict})
    return [dict(p=130, m=150, **s) if "p" not in s else s for s in shapes["CASES"] + shapes["CEILING_SHAPES"]]


def make_inputs(path):
    from blmm_b200 import synth
    cases = [dict(s, kind="grid") for s in grid_edge_shapes()]
    cases += [dict(n=79, p=500, m=1, c=1, nk=1, kind="perms"), dict(n=137, p=500, m=1, c=2, nk=1, kind="perms")]
    arrays = {}
    for i, s in enumerate(cases):
        n, p, m, c = s["n"], s["p"], s["m"], s["c"]
        G = synth.make_geno(n, p, seed=1000 + i)
        K = synth.calc_kinship_host(G)
        lam, U = np.linalg.eigh(K)
        rng = np.random.default_rng(2000 + i)
        Cv = np.hstack([np.ones((n, 1)), rng.standard_normal((n, c - 1))])
        arrays.update({f"{i}_G": G, f"{i}_U": U, f"{i}_lam": np.clip(lam, 0.0, None), f"{i}_Cv": Cv,
                       f"{i}_Y": synth.make_pheno(G, K, max(m, 1), seed=3000 + i),
                       f"{i}_perm": synth.make_perm_indices(n, 255 if s["kind"] == "perms" else 20, 4000 + i),
                       f"{i}_grid": np.arange(s["nk"]) / max(s["nk"], 10)})
    np.savez(path, cases=json.dumps(cases), **arrays)


def run_build(inputs, out):
    """In the child process: every call on every case with the build named by BLMM_B200_LIB; results to out (.npz)."""
    from blmm_b200 import Engine, _lib as L
    z = np.load(inputs)
    cases = json.loads(str(z["cases"]))
    eng = Engine(0)
    res = {}

    def record(key, fn):
        try:
            r = fn()
        except Exception as ex:  # an error is an outcome too: both builds must raise the same one
            res[key + "/error"] = np.frombuffer(repr(ex).encode(), dtype=np.uint8)
            return
        r = vars(r) if hasattr(r, "__dict__") else r
        items = r.items() if isinstance(r, dict) else enumerate(r if isinstance(r, tuple) else (r,))
        for name, v in items:
            if v is not None:
                res[f"{key}/{name}"] = np.asarray(v)

    methods = {"null-grid": L.METHOD_NULL_GRID, "alt-grid": L.METHOD_ALT_GRID, "null-exact": L.METHOD_NULL_EXACT}
    for i, s in enumerate(cases):
        G, U, lam, Cv, Y, perm, grid = (z[f"{i}_{k}"] for k in ("G", "U", "lam", "Cv", "Y", "perm", "grid"))
        tag = f"{i}:{s['kind']}-n{s['n']}-p{s['p']}-m{s['m']}-c{s['c']}-k{s['nk']}"
        y1 = Y[:, :1]
        if s["kind"] == "grid":
            for nm, meth in methods.items():
                reml = nm == "null-exact"
                record(f"{tag}/bulkscan-{nm}", lambda: eng.bulkscan_host(Y, G, Cv, U, lam, meth, grid, reml, 0.0, 0.0))
                record(f"{tag}/bulkscan_peaks-{nm}",
                       lambda: eng.bulkscan_peaks_host(Y, G, Cv, U, lam, meth, grid, reml, 0.0, 0.0))
            record(f"{tag}/grid_loglik", lambda: eng.grid_loglik(Y, Cv, U, lam, grid, prior_variance=0.0))
            record(f"{tag}/fit_h2", lambda: eng.fit_h2(Y, Cv, U, lam, reml=True))
            record(f"{tag}/scan_null", lambda: eng.scan_null_host(Y, G, Cv, U, lam, reml=True))
            if s["c"] + 1 <= 8:  # scan_alt takes the marker as one more covariate column
                record(f"{tag}/scan_alt", lambda: eng.scan_alt_host(y1, G, Cv, U, lam))
        for path in ("chain", "separate"):
            if path == "separate":
                os.environ["BLMM_B200_NO_CHAIN"] = "1"
            record(f"{tag}/scan_perms-{path}", lambda: eng.scan_perms_host(y1, G, Cv, U, lam, perm))
            os.environ.pop("BLMM_B200_NO_CHAIN", None)
    eng.close()
    np.savez(out, **res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("libs", nargs="*")
    ap.add_argument("--out", help="directory for the inputs and both builds' results (default: a temporary one)")
    ap.add_argument("--child", nargs=2, metavar=("INPUTS", "OUT"), help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.child:
        run_build(*args.child)
        return 0
    if len(args.libs) != 2:
        ap.error("give the two library builds to compare")
    out = args.out or tempfile.mkdtemp(prefix="blmm_bitcompare_")
    os.makedirs(out, exist_ok=True)
    inputs = os.path.join(out, "inputs.npz")
    make_inputs(inputs)
    results = []
    for k, lib in enumerate(args.libs):
        dst = os.path.join(out, f"build{k}.npz")
        env = dict(os.environ, BLMM_B200_LIB=os.path.abspath(lib), PYTHONDONTWRITEBYTECODE="1")
        subprocess.run([sys.executable, os.path.abspath(__file__), "--child", inputs, dst], env=env, check=True)
        results.append(np.load(dst))
    a, b = results
    keys = sorted(set(a.files) | set(b.files))
    differ = [k for k in keys if k not in a.files or k not in b.files or a[k].dtype != b[k].dtype
              or a[k].shape != b[k].shape or a[k].tobytes() != b[k].tobytes()]
    errors = [k for k in keys if k.endswith("/error")]
    for k in differ:
        print(f"DIFFERS {k}")
    for k in errors:
        print(f"error (both builds) {k}: {bytes(a[k]).decode() if k in a.files else ''}")
    print(json.dumps({"builds": args.libs, "outputs": len(keys), "identical": len(keys) - len(differ),
                      "differ": len(differ), "errors": len(errors), "results": out}))
    return 1 if differ else 0


if __name__ == "__main__":
    sys.exit(main())
