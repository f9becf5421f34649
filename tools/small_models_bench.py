"""Microseconds per model-step of the ELBO step + Adam for K small black-box models, three ways:
  (a) GraphedELBOStep, one model after the other on one stream;
  (b) one stream and one GraphedELBOStep per model (BlackBoxMFDGPFitter(concurrent_models=True) before the single-kernel
      step; bench.py's small_configs does the same);
  (c) GraphedSmallModelsELBOStep: mobo_elbo_step_small (one CTA per model) + the K Adam updates in one graph.
Configurations: C2 Forrester (d = 1, 2 fidelities, N = M = B = 16) and the N = 75 synthetic set (d = 2, M = 75: beyond
the single-CTA limit, so (c) does not apply there), K = 1, 3, 6; then a sweep over M = 16 ... 64 and B = 16 ... 256
(K = 1, 3, 6, S = 1 as the fitter trains) that places the fitter's selection bounds (`selection`).  Device events around each timed
window after a warm-up; the card's name and power limit are read in the same run.  Also compares one step of (a) and
(c) on the same seeded inputs.  Writes JSON (--out).  Run on a GPU box: python tools/small_models_bench.py"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mobocmf_b200.fused import (Adam, FusedELBOStep, GraphedELBOStep, GraphedSmallModelsELBOStep,  # noqa: E402
                                SmallModelsELBOStep)
from mobocmf_b200.mlls.variational_elbo_mf import VariationalELBOMF  # noqa: E402
from mobocmf_b200.models.mfdgp import MFDGP  # noqa: E402
from tests.helpers import forrester_data, relerr, synthetic_data  # noqa: E402

DEV = torch.device("cuda:0")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.stdout else ""}


def data(cfg):
    if cfg == "C2_forrester_N16":
        x, ys, fid = forrester_data()
        return x, [ys["obj1"], ys["obj2"], ys["con1"]], fid, None
    if cfg == "synthetic_N75":
        x, y, fid = synthetic_data([50, 25], 2, seed=4)
        return x, [y, -y, 0.5 * y], fid, None
    M = int(cfg.split("_")[1][1:])           # "rows_M64"
    x, y, fid = synthetic_data([400, 200], 2, seed=5)
    return x, [y, -y, 0.5 * y], fid, M


def models(cfg, K):
    x, ys, fid, M = data(cfg)
    out = []
    for k in range(K):
        torch.manual_seed(k)
        m = MFDGP(x, ys[k % 3], fid, 2, num_inducing=M, init_lengthscale=0.3 if M else None)
        m.double().to(DEV)
        m.fix_variational_hypers(False)
        out.append((m, VariationalELBOMF(m, x.shape[0], 2)))
    return x, ys, fid, out


def batches_for(x, ys, fid, K, B, seed):
    g = torch.Generator().manual_seed(seed)
    out = []
    for k in range(K):
        idx = torch.randperm(x.shape[0], generator=g)[:B] if B <= x.shape[0] else \
            torch.randint(0, x.shape[0], (B,), generator=g)
        if B == x.shape[0] and torch.equal(idx, torch.arange(B)):
            idx = torch.roll(idx, 1)
        out.append((x[idx].to(DEV), ys[k % 3][idx].to(DEV), fid[idx].to(DEV)))
    return out


def timed(fn, steps, reps=3, warmup=20):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    res = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        res.append(e0.elapsed_time(e1) * 1e3 / steps)
    return sorted(res)[len(res) // 2], res


def run_a(ms, batches):
    gs = []
    for (m, e), b in zip(ms, batches):
        o = Adam([{"params": m.parameters()}], lr=1e-3, capturable=True)
        gs.append((GraphedELBOStep(FusedELBOStep(m, e), o, b[0].shape[0]), b))

    def fn():
        for g, b in gs:
            g(*b, check_shortcut=False)
    return fn


def run_b(ms, batches):
    cur = torch.cuda.current_stream()
    gs = []
    for (m, e), b in zip(ms, batches):
        o = Adam([{"params": m.parameters()}], lr=1e-3, capturable=True)
        gs.append((GraphedELBOStep(FusedELBOStep(m, e), o, b[0].shape[0]), b, torch.cuda.Stream(device=DEV)))

    def fn():
        for g, b, st in gs:
            st.wait_stream(cur)
            with torch.cuda.stream(st):
                g(*b, check_shortcut=False)
        for _, _, st in gs:
            cur.wait_stream(st)
    return fn


def run_c(ms, batches):
    small = SmallModelsELBOStep([m for m, _ in ms], [e for _, e in ms])
    opts = [Adam([{"params": m.parameters()}], lr=1e-3, capturable=True) for m, _ in ms]
    g = GraphedSmallModelsELBOStep(small, opts)

    def fn():
        g(batches, check_shortcut=False)
    return fn


def compare(cfg, K, B):
    """One step of FusedELBOStep and of SmallModelsELBOStep on the same models, minibatches and normals."""
    x, ys, fid, ms = models(cfg, K)
    batches = batches_for(x, ys, fid, K, B, seed=11)
    g = torch.Generator().manual_seed(12)
    eps = [[None, torch.randn(B, generator=g).double().to(DEV)] for _ in range(K)]
    worst_loss, worst_grad = 0.0, 0.0
    ref = []
    for (m, e), b, ep in zip(ms, batches, eps):
        f = FusedELBOStep(m, e)
        loss, _ = f(*b, eps=ep)
        ref.append((loss.clone(), f.flat.flat.clone()))
    small = SmallModelsELBOStep([m for m, _ in ms], [e for _, e in ms])
    res = small(batches, eps=eps)
    for (l1, _), (l0, g0), st in zip(res, ref, small.steps):
        worst_loss = max(worst_loss, relerr(l1, l0))
        worst_grad = max(worst_grad, relerr(st.flat.flat, g0))
    return {"loss_relerr_max": worst_loss, "flat_grad_relerr_max": worst_grad}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--out", default="profiles/r03_small_models_bench.json")
    args = ap.parse_args()
    out = {"card": card(), "unit": "us per model-step (ELBO step + Adam), median of 3 windows", "configs": {}}
    for cfg, B in (("C2_forrester_N16", 16), ("synthetic_N75", 75)):
        res = {}
        for K in (1, 3, 6):
            row = {}
            for mode, make in (("a_sequential_graphs", run_a), ("b_stream_and_graph_per_model", run_b),
                               ("c_small_step_graph", run_c)):
                x, ys, fid, ms = models(cfg, K)
                ok, why = SmallModelsELBOStep.supported([m for m, _ in ms])
                if mode.startswith("c") and not ok:
                    row[mode] = "not applicable: " + why
                    continue
                med, all_ = timed(make(ms, batches_for(x, ys, fid, K, B, seed=K)), args.steps)
                row[mode] = round(med / K, 2)
                row[mode + "_windows_us_per_step"] = [round(v, 1) for v in all_]
            res["K%d" % K] = row
            print(cfg, K, row, flush=True)
        if cfg.startswith("C2"):
            res["parity_a_vs_c_K6"] = compare(cfg, 6, B)
        out["configs"][cfg] = res
    # where one CTA per model stops paying: per (M, B, K) the existing concurrent path (b) against the small step (c)
    sweep = {}
    for M in (16, 24, 32, 40, 48, 64):
        for B in (16, 32, 64, 128, 256):
            for K in (1, 3, 6):
                row = {}
                for mode, make in (("b_stream_and_graph_per_model", run_b), ("c_small_step_graph", run_c)):
                    x, ys, fid, ms = models("rows_M%d" % M, K)
                    med, _ = timed(make(ms, batches_for(x, ys, fid, K, B, seed=B)), max(50, args.steps // 4))
                    row[mode] = round(med / K, 2)
                sweep["M%d_B%d_K%d" % (M, B, K)] = row
                print("M", M, "B", B, "K", K, row, flush=True)
    out["sweep_S1"] = sweep
    out["parity_a_vs_c_M64_B128"] = compare("rows_M64", 3, 128)

    def wins(M, B):
        return all(sweep["M%d_B%d_K%d" % (M, B, K)]["c_small_step_graph"] <
                   sweep["M%d_B%d_K%d" % (M, B, K)]["b_stream_and_graph_per_model"] for K in (1, 3, 6))
    ms_ok = [M for M in (16, 24, 32, 40, 48, 64) if wins(M, 16)]
    max_m = max(ms_ok) if ms_ok else None
    rows_ok = [B for B in (16, 32, 64, 128, 256) if max_m is not None and wins(max_m, B)]
    # the fitter's bounds: the largest M at which c beats b for every K at B = 16, and at that M the largest B
    out["selection"] = {"max_inducing": max_m, "max_rows": max(rows_ok) if rows_ok else None}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
