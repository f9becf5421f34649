"""Forward + d acq / dX of the C5 JESMOC acquisition (6 black boxes x (1 + 16) MFDGPs, M = 256, d = 6, L = 3, S = 25,
fidelity 2; bench.py's models), through the fused chain (mobo_acq_moments + mobo_acq_moments_bwd) and through the
composable autograd path (one _LayerRows per layer, torch glue), which every acquisition took before the fused
backward existed.

    python tools/acq_grad_bench.py [--runs 5] [--n-small 1024] [--n-large 125000] [--out DIR]

prints one JSON line (and writes it to DIR/acq_grad_bench.json with --out).
Records, with the device name and power limit read in the same run:
  * forward + dX candidates/s at n_small, fused and composable alternating, `runs` runs each;
  * fused forward + dX at n_large (C5's candidates per GPU), with the peak memory; the composable path keeps
    ~21 MB of saved rows per candidate and cannot run this size;
  * the forward-only jes_sweep at n_large as the reference point.
Times are CUDA events around work that ends in a device synchronisation; every shape is warmed up first."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def device_info(index=0):
    q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(index)


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--n-small", type=int, default=1024)
    ap.add_argument("--n-large", type=int, default=125000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import bench
    from mobocmf_b200.acquisition_functions.JESMOC_MFDGP import jes_sweep
    from mobocmf_b200.models.mfdgp import MFDGP

    dev = torch.device("cuda:0")
    cfg = bench.C4
    x, y, fid = bench.c4_data(cfg)
    boxes = bench.acq_models(bench.build_model(cfg, x, y, fid, dev), dev, K=6, P=16)
    fidelity = cfg["L"] - 1
    g = torch.Generator().manual_seed(1)
    X = torch.rand(args.n_large, cfg["d"], dtype=torch.float64, generator=g).to(dev)
    fused_applies = MFDGP._fused_acquisition_applies

    def fwd_dx(n):
        Xg = X[:n].clone().requires_grad_(True)
        v = jes_sweep(Xg, fidelity, boxes)
        v.sum().backward()
        return v.detach(), Xg.grad

    def composable(on):
        MFDGP._fused_acquisition_applies = (lambda self, x: False) if on else fused_applies

    res = {"device": device_info(), "workload": "C5 acquisition: 6 black boxes x (1 + 16) MFDGPs = 102 chains, "
                                                "M=256, d=6, L=3, S=25, fidelity 2"}
    # n_small: fused and composable alternating (each warmed up once)
    v_ref = jes_sweep(X[:args.n_small], fidelity, boxes)
    for path in ("fused", "composable"):
        composable(path == "composable")
        fwd_dx(args.n_small)
    times = {"fused": [], "composable": []}
    grads = {}
    for _ in range(args.runs):
        for path in ("fused", "composable"):
            composable(path == "composable")
            ms, (v, gx) = timed(lambda: fwd_dx(args.n_small))
            times[path].append(ms)
            grads[path] = (v, gx)
    composable(False)
    gf, gc = grads["fused"][1], grads["composable"][1]
    res["small"] = {"n": args.n_small}
    for path, ts in times.items():
        res["small"][path] = {"ms": ts, "candidates_per_s": [args.n_small / (t * 1e-3) for t in ts],
                              "median_candidates_per_s": args.n_small / (statistics.median(ts) * 1e-3),
                              "spread_pct": 100.0 * (max(ts) - min(ts)) / statistics.median(ts)}
    res["small"]["dX_max_rel_diff_fused_vs_composable"] = float((gf - gc).abs().max() / gc.abs().max())
    res["small"]["values_fused_minus_forward_only_max_abs"] = float((grads["fused"][0] - v_ref).abs().max())

    # n_large: forward only, then fused forward + dX with its peak memory
    jes_sweep(X[:4096], fidelity, boxes)
    ms_f, v_large = timed(lambda: jes_sweep(X, fidelity, boxes))
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    ms_g, (v_g, gx) = timed(lambda: fwd_dx(args.n_large))
    peak = torch.cuda.max_memory_allocated() - base
    res["large"] = {"n": args.n_large,
                    "forward_only": {"ms": ms_f, "candidates_per_s": args.n_large / (ms_f * 1e-3)},
                    "fused_fwd_plus_dX": {"ms": ms_g, "candidates_per_s": args.n_large / (ms_g * 1e-3),
                                          "peak_memory_growth_gib": peak / 2 ** 30,
                                          "values_equal_forward_only": bool(torch.equal(v_g, v_large)),
                                          "grad_finite": bool(torch.isfinite(gx).all())}}
    res["acq_grad_chunk"] = MFDGP.ACQ_GRAD_CHUNK
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "acq_grad_bench.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
