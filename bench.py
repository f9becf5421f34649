#!/usr/bin/env python
"""Benchmark of the MFDGP hot path on B200:  python bench.py --gpus N --steps K --warmup W [--impl reference]

Workload (BASELINE.json configs[3], SURVEY.md §8d "C4"): scaled MFDGP training, d=6, 3 fidelities, N=50 000
synthetic points, M=256 inducing inputs, minibatch B=1024 rows x S=64 MC samples, fp64.  One STEP = the body of
``_update_model`` (mobocmf/util/blackbox_mfdgp_fitter.py:161-171): zero-grad, forward, ELBO, backward, Adam.
``--scaling weak`` (default): with N GPUs every rank processes its own 1024-row minibatch and the parameter gradients
are summed over NCCL, i.e. one global step over N*1024 rows; ``value`` counts 1024 x 64 step units per second.
``--scaling strong``: ONE 1024 x 64 step whose rows are split over the ranks (``util.distributed.shard_bounds``);
``value`` counts global steps per second.

The second headline of BASELINE.json (JESMOC acquisition evals/s, configs[4] "C5": 10^6 candidates x 16 Pareto samples
x (4 objectives + 2 constraints) sharded over 8 GPUs = 125 000 candidates per GPU) is reported under ``"acq"`` in the
same JSON line with its own roofline / cpu_baseline / e2e blocks; ``"parity"`` holds the CUDA-vs-oracle errors of
one C4 step, computed outside the timed region.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C4 = dict(N=50000, d=6, L=3, M=256, B=1024, S=64, fid_sizes=(30000, 15000, 5000), lengthscale=0.3, seed=0)
C5_CANDIDATES_PER_GPU = 125000   # 10^6 candidates over 8 GPUs (BASELINE.json configs[4])


def workload_config(world, scaling, B):
    """``config`` of the JSON line, shared by both arms (the reference arm times the same workload on the host)."""
    per = "per GPU (step unit = 1024 x 64)" if scaling == "weak" else "in total, rows sharded over the GPUs"
    return {"workload": "C4 scaled MFDGP training: d=6, 3 fidelities, N=50000, M=256, B=1024 rows x S=64 MC samples "
                        "%s, lengthscale 0.3, Adam lr 1e-3" % per,
            "global_batch": world * B if scaling == "weak" else B,
            "parallelism": "dp%d rows sharded, grads all-reduced" % world,
            "cache": "per-step working set (3 x 134 MB saved tiles per upper layer) exceeds L2"}
FP64_PEAK_TFLOPS = 37.1   # measured DMMA.8x8x4 pipe peak on this pool's B200 (profiles/r01_fp64_probe.log);
#                           cuBLAS DGEMM reaches 35.4 (profiles/r01_dgemm_probe.log).  MEASURED_PEAKS.json has no fp64 entry.


def c4_data(cfg):
    """SURVEY.md §8d C4 recipe: seeded closed-form 3-fidelity targets on U[0,1]^6, rows shuffled so that the first M
    rows (the inducing inputs) are a random subset."""
    g = torch.Generator().manual_seed(cfg["seed"])
    N, d = cfg["N"], cfg["d"]
    x = torch.rand(N, d, generator=g, dtype=torch.float64)
    fid = torch.cat([torch.full((n,), float(l)) for l, n in enumerate(cfg["fid_sizes"])]).double()
    y0 = torch.sin(2 * math.pi * x).sum(1) / math.sqrt(d)
    y1 = 0.8 * y0 + 0.2 * torch.cos(math.pi * x.sum(1))
    y2 = y1 ** 2 - 0.5 * y1 + 0.1 * x[:, 0]
    y = torch.where(fid == 0, y0, torch.where(fid == 1, y1, y2)) + 1e-2 * torch.randn(N, generator=g).double()
    perm = torch.randperm(N, generator=g)
    return x[perm].contiguous(), y[perm][:, None].contiguous(), fid[perm][:, None].contiguous()


def build_model(cfg, x, y, fid, device):
    from mobocmf_b200.models.mfdgp import MFDGP
    torch.manual_seed(cfg["seed"])
    model = MFDGP(x, y, fid, cfg["L"], num_inducing=cfg["M"], init_lengthscale=cfg["lengthscale"])
    model.double()
    return model.to(device)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                self.rows.append([c.strip() for c in out.stdout.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if len(r) >= 6 and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) >= 6 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i] == "Active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def step_flops(cfg):
    """Algorithmic flops of one step (SURVEY.md §8d): per (row, layer) forward F = 2 M^2 + 2 M + 3 d_l M, rows
    R_tot = B + (L-1) B S, step ~ 3 F R_tot + 12 L M^3."""
    M, B, S, L, d = cfg["M"], cfg["B"], cfg["S"], cfg["L"], cfg["d"]
    f0 = 2 * M * M + 2 * M + 3 * d * M
    f1 = 2 * M * M + 2 * M + 3 * (d + 1) * M
    return 3 * (f0 * B + (L - 1) * f1 * B * S) + 12 * L * M ** 3, f1


def run_ours(args):
    import torch.distributed as dist
    from mobocmf_b200 import _lib
    from mobocmf_b200.gp import settings
    from mobocmf_b200.mlls.variational_elbo_mf import VariationalELBOMF
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"       # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        dist.init_process_group("nccl", device_id=dev)
    cfg = dict(C4)
    if os.environ.get("MOBO_BENCH_B"):          # development: another minibatch size (not the BASELINE workload)
        cfg["B"] = int(os.environ["MOBO_BENCH_B"])
    x, y, fid = c4_data(cfg)
    model = build_model(cfg, x, y, fid, dev)
    elbo = VariationalELBOMF(model, cfg["N"], cfg["L"])
    model.fix_variational_hypers(False)
    params = [p for p in model.parameters() if p.requires_grad]
    xd, yd, fd = x.to(dev), y.to(dev), fid.to(dev)
    S, N = cfg["S"], cfg["N"]
    strong = args.scaling == "strong"
    if strong:
        # ONE global minibatch of cfg["B"] points per step, drawn identically on every rank; rank r owns a contiguous
        # shard of its points (and their S sample rows)
        from mobocmf_b200.util.distributed import shard_bounds
        lo_b, hi_b = shard_bounds(cfg["B"], rank, world)
        B = hi_b - lo_b
    else:
        lo_b, B = 0, cfg["B"]
    Bdraw = cfg["B"]
    g = torch.Generator(device=dev).manual_seed(1234 + (0 if strong else rank))
    # pinned host staging for the end-to-end arm
    xh, yh, fh = x.pin_memory(), y.pin_memory(), fid.pin_memory()

    if args.path == "fused":
        # the product path of the fitter's hot loop: mobo_elbo_step (one enqueue, no autograd) + mobo_adam
        from mobocmf_b200.fused import Adam, FusedELBOStep
        from mobocmf_b200.util.distributed import broadcast_parameters
        broadcast_parameters(model)
        fstep = FusedELBOStep(model, elbo)
        opt = Adam([{"params": params}], lr=0.001)
        comm = torch.cuda.Stream(device=dev) if world > 1 and args.allreduce == "overlapped" else None

        def one_step(xb, yb, fb):
            loss, _ = fstep(xb, yb, fb, num_samples=S)
            if world > 1:
                if comm is not None:
                    # the three M x M blocks d L_q (1.5 of the 1.6 MB) leave as soon as their layer's operator-chain
                    # backward is done, behind the lower layers' row kernels; only the ~6 KB tail waits for the step
                    fstep.flat.all_reduce_overlapped(fstep.wait_bucket, comm)
                else:
                    fstep.flat.all_reduce()      # ONE all-reduce of the flat gradient buffer (NCCL over NVLink)
            opt.step()
            return loss
    else:
        # composable path: the same kernels under torch autograd + torch.optim.Adam (kept for comparison)
        opt = torch.optim.Adam([{"params": params}], lr=0.001)

        def one_step(xb, yb, fb):
            opt.zero_grad(set_to_none=True)
            with settings.num_likelihood_samples(1):
                out = model(xb, num_samples=S)
                res = elbo(out, yb.T, fb)
            loss = -res[0]
            loss.backward()
            if world > 1:
                flat = torch.cat([p.grad.reshape(-1) for p in params])
                dist.all_reduce(flat)
                off = 0
                for p in params:
                    n = p.numel()
                    p.grad.copy_(flat[off:off + n].view_as(p.grad))
                    off += n
            opt.step()
            return loss

    def device_step():
        idx = torch.randint(0, N, (Bdraw,), device=dev, generator=g)[lo_b:lo_b + B]
        return one_step(xd[idx], yd[idx], fd[idx])

    # two pinned staging sets: the host fills set i % 2 while the copies of step i - 1 may still be in flight; set
    # i % 2 was last used by step i - 2, whose loss has been consumed (so its copies are complete) by then
    hbs = [[torch.empty(B, cfg["d"], dtype=torch.float64).pin_memory(), torch.empty(B, 1, dtype=torch.float64).pin_memory(),
            torch.empty(B, 1, dtype=torch.float64).pin_memory()] for _ in range(2)]
    gh = torch.Generator().manual_seed(99 + (0 if strong else rank))

    # End-to-end arm: every step copies ITS minibatch from pinned host memory (H2D inside the timed region) and the
    # step's loss comes back to pinned host memory (D2H).  The loss of step i is consumed by the host while step
    # i + 1 is already enqueued (a one-deep prefetch, like any data loader), so the GPU never waits for Python;
    # the last loss is read inside the timed region too.
    loss_host = torch.zeros(2, dtype=torch.float64).pin_memory()
    pending = []
    e2e_losses = []

    def e2e_step():
        slot = len(e2e_losses) % 2
        hb = hbs[slot]
        idx = torch.randint(0, N, (Bdraw,), generator=gh)[lo_b:lo_b + B]
        torch.index_select(xh, 0, idx, out=hb[0]); torch.index_select(yh, 0, idx, out=hb[1])
        torch.index_select(fh, 0, idx, out=hb[2])
        xb, yb, fb = (t.to(dev, non_blocking=True) for t in hb)
        loss = one_step(xb, yb, fb)
        if pending:                       # consume the previous step's loss before its slot can be reused
            ev, sl = pending.pop()
            ev.synchronize()
            e2e_losses[-1] = float(loss_host[sl])
        loss_host[slot:slot + 1].copy_(loss.detach().reshape(1), non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        pending.append((ev, slot))
        e2e_losses.append(None)

    def e2e_drain():
        if pending:
            ev, sl = pending.pop()
            ev.synchronize()
            e2e_losses[-1] = float(loss_host[sl])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            last = fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms), last

    parity = None
    if rank == 0 and not args.no_parity and args.path == "fused":
        parity = parity_block(cfg, x, y, fid, model, fstep, dev)

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()                   # sampled through warm-up and the timed region (a timed region of K steps
    for _ in range(max(args.warmup, 3)):  # of 3 ms is shorter than one nvidia-smi call)
        device_step()
    for _ in range(400):                  # ~1 s more under load on EVERY rank (the step holds a collective), so
        device_step()                     # that the sampler has several readings under load before the clock starts
    l0 = _lib.launch_count()
    ms, last_loss = timed(device_step, args.steps)
    launches = _lib.launch_count() - l0
    dump = None
    if args.dump_outputs and rank == 0:
        # what a caller of the step holds after the last timed step: its loss, the gradients it wrote and the
        # parameters Adam updated (copied now: the steps below overwrite all three)
        dump = {"loss": last_loss.detach().reshape(1).cpu()}
        for n, p in model.named_parameters():
            if p.requires_grad:
                dump["grad." + n] = p.grad.detach().cpu()
                dump["param." + n] = p.detach().cpu()
    if sampler:
        sampler.stop_flag = True
    for _ in range(2):
        e2e_step()
    e2e_drain()

    barrier()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        e2e_step()
    e2e_drain()                            # the last step's loss is on the host before the clock stops
    e1.record()
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    ms_e2e = torch.tensor([max(e0.elapsed_time(e1), wall_ms)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms_e2e, op=dist.ReduceOp.MAX)
    ms_e2e = float(ms_e2e)
    e2e_finite = all(v is not None and math.isfinite(v) for v in e2e_losses[-args.steps:])

    # per-kernel CUDA-event timing of a few extra steps (launch stream = torch's current stream)
    prof = {}
    nprof = min(args.steps, 5)
    if rank == 0:
        _lib.profile_enable(True)
        _lib.load().mobo_step_side_stream(0)   # serialise the step's side stream so that per-kernel times are clean
    for _ in range(nprof):            # every rank steps (the step contains the gradient all-reduce); rank 0 records
        device_step()
    torch.cuda.synchronize()
    if rank == 0:
        for name, t in _lib.profile_collect():
            prof.setdefault(name, []).append(t)
        _lib.profile_enable(False)
        _lib.load().mobo_step_side_stream(1)

    # acquisition slice (C5-shaped): n candidates x S=25 samples through an (uncond, cond) pair at the top fidelity
    acq = None
    if not args.no_acq:
        acq = bench_acq(model, dev, cfg, world, rank, n=args.acq_candidates, with_cpu=not args.no_cpu, dump=dump)

    if rank == 0:
        flops, f1 = step_flops(cfg)
        ms_step = ms / args.steps
        units = 1 if strong else world          # 1024 x 64 step units completed per timed step
        out = {
            "metric": "mfdgp_elbo_steps_per_s", "value": units * args.steps / (ms / 1e3), "unit": "steps/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": workload_config(world, args.scaling, cfg["B"]),
            "e2e": {"value": units * args.steps / (ms_e2e / 1e3), "unit": "steps/s",
                    "h2d_bytes_per_step": B * (cfg["d"] + 2) * 8, "d2h_bytes_per_step": 8,
                    "losses_finite": e2e_finite, "last_loss": e2e_losses[-1],
                    "note": "host minibatch -> pinned H2D -> fused step + Adam -> loss D2H, every step; the loss of "
                            "step i is read while step i+1 is enqueued"},
            "gpu_launches": int(launches),
            "clocks": sampler.summary() if sampler else None,
            "step_tflops": flops / (ms_step * 1e-3) / 1e12 * (1 if not strong else 1.0 / world),
        }
        if parity is not None:
            out["parity"] = parity
        if prof:
            tot = {k: sum(v) for k, v in prof.items()}
            nst = min(args.steps, 5)
            # dominant kernel = the one of OUR kernels with the largest share of the step; its algorithmic flops are
            # summed over its launches of a step (layer 0 runs on B rows, the upper layers on B*S) and divided by the
            # summed launch durations (DESIGN.md section 2 "Roofline numerator")
            M, d, L = cfg["M"], cfg["d"], cfg["L"]
            rows = [B] + [B * S] * (L - 1)       # this rank's rows (strong scaling: its shard)
            dl = [d] + [d + 1] * (L - 1)
            fwd_l = [r * (2 * M * M + 2 * M + 3 * k * M) for r, k in zip(rows, dl)]
            ws = "row_fwd_ws_kernel" in tot      # the S-sample rows of the upper layers run in the warp-specialised kernel
            alg_per_step = {
                "row_fwd_kernel": fwd_l[0] if ws else sum(fwd_l),
                "row_fwd_ws_kernel": sum(fwd_l[1:]),
                "row_bwd_gemm_kernel": sum(r * (2 * M * M + 2 * M) for r in rows),
                "syrk_kernel": sum(r * M * M for r in rows),
            }
            top = max((k for k in tot if k in alg_per_step), key=lambda k: tot[k])
            ms_top = tot[top] / nst
            achieved = alg_per_step[top] / (ms_top * 1e-3) / 1e12
            traffic = None
            tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
            if os.path.exists(tpath):
                traffic = json.load(open(tpath)).get(top)
            out["roofline"] = {"bound": "tensor", "kernel": top, "achieved": achieved, "peak": FP64_PEAK_TFLOPS,
                               "unit": "TFLOP/s", "frac": achieved / FP64_PEAK_TFLOPS, "traffic": traffic,
                               "peak_source": "measured DMMA fp64 pipe peak (mma.sync.m8n8k4.f64), "
                                              "profiles/r01_fp64_probe.log; MEASURED_PEAKS.json has no fp64 figure "
                                              "(cuBLAS DGEMM on the same pool: 35.4)",
                               "launches_per_step": len(prof[top]) // nst, "ms_per_step": ms_top,
                               "algorithmic_gflop_per_step": alg_per_step[top] / 1e9,
                               "share_of_step": ms_top / ms_step}
            out["roofline_by_kernel"] = {k: round(alg_per_step[k] / (tot[k] / nst * 1e-3) / 1e12 / FP64_PEAK_TFLOPS, 4)
                                         for k in alg_per_step if k in tot and tot[k] > 0}
            out["kernel_ms_per_step"] = {k: round(v / nst, 4) for k, v in sorted(tot.items(), key=lambda kv: -kv[1])}
            out["kernel_ms_note"] = ("CUDA-event time per kernel over %d extra steps run with the step's side stream "
                                     "serialised (mobo_step_side_stream(0)); in the timed region the operator-chain "
                                     "backward overlaps the row kernels, so ms_per_step is below the sum" % nst)
        if acq:
            out["acq"] = acq
        if not args.no_acq and world == 1:
            out["pareto_sampling"] = bench_pareto(dev, with_cpu=not args.no_cpu)
        if not args.no_acq and world == 1:
            out["small_configs"] = bench_small_configs(dev)
        if not args.no_cpu and world == 1:      # reported on rank 0 at N = 1 only
            out["cpu_baseline"] = cpu_baseline(cfg, x, y, fid, model, steps=8, warmup=2)
        if dump is not None:
            write_outputs(args.dump_outputs, dump)
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


DUMP_SAMPLE = 1 << 20          # entries kept of a larger output array
DUMP_MAX_BYTES = 64 << 20


def write_outputs(directory, arrays):
    """``--dump-outputs``: every array as ``directory/<name>.npy`` in float64.  An array of more than DUMP_SAMPLE
    entries is flattened and reduced to the entries at DUMP_SAMPLE positions drawn with a fixed seed, so that runs with
    the same arguments write the same positions and two builds can be compared entry for entry."""
    import numpy as np
    out = {}
    for name, t in arrays.items():
        a = t.double().numpy()
        if a.size > DUMP_SAMPLE:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))]
        out[name] = a
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_MAX_BYTES))
    os.makedirs(directory, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def bench_small_configs(dev, steps=200):
    """The reference's own (launch-latency-bound) configurations: full-batch ELBO step + Adam, one MC sample, through
    the fitter's hot loop body, eager fused enqueue vs one CUDA-graph launch per step (SURVEY.md section 8d C1-C3).
    C2 = Forrester (d=1, 2 fidelities, N=M=B=16, examples/example_acquisition_mfdgp_forrester); C1/C3-sized = d=2,
    2 fidelities, N=M=B=75 (the toy / synthetic-2D runs at their largest)."""
    from mobocmf_b200.fused import Adam, FusedELBOStep, GraphedELBOStep
    from mobocmf_b200.mlls.variational_elbo_mf import VariationalELBOMF
    from mobocmf_b200.models.mfdgp import MFDGP
    import numpy as np

    def forrester_data():
        """Deterministic data of examples/example_acquisition_mfdgp_forrester/...py:51-104 (config C2)."""
        mf1 = lambda t: ((6 * t - 2) ** 2) * np.sin(12 * t - 4)
        mf0 = lambda t: 0.5 * mf1(t) + 10 * (t - 0.5) + 5
        x0, x1 = np.linspace(0, 1.0, 12).reshape(12, 1), np.array([0.1, 0.3, 0.5, 0.7]).reshape(4, 1)
        y0, y1 = mf0(x0), mf1(x1)
        mean, std = np.mean(np.vstack((y1, y0))), np.std(np.vstack((y1, y0)))
        yy = torch.cat((torch.from_numpy((y1 - mean) / std), torch.from_numpy((y0 - mean) / std)), 0).double()
        xx = torch.cat((torch.from_numpy(x1), torch.from_numpy(x0)), 0).double()
        ff = torch.cat((torch.ones(4).double(), torch.zeros(12).double()))[:, None]
        return xx, yy, ff

    def synthetic_data(n_per_fid, d, seed=0):
        gg = torch.Generator().manual_seed(seed)
        xs, ys, fs = [], [], []
        for l, n in enumerate(n_per_fid):
            xx = torch.rand(n, d, generator=gg, dtype=torch.float64)
            y0 = torch.sin(2 * math.pi * xx).sum(1) / math.sqrt(d)
            yl = y0 if l == 0 else 0.8 * y0 + 0.2 * torch.cos(math.pi * xx.sum(1))
            xs.append(xx); ys.append(yl[:, None]); fs.append(torch.full((n, 1), float(l), dtype=torch.float64))
        return torch.cat(xs), torch.cat(ys), torch.cat(fs)
    out = {}
    for name in ("C2_forrester_N16", "C1C3_sized_N75"):
        if name.startswith("C2"):
            x, y, fid = forrester_data()
        else:
            x, y, fid = synthetic_data([50, 25], 2, seed=4)
        N = x.shape[0]
        res = {}
        for mode in ("eager", "graph"):
            torch.manual_seed(0)
            model = MFDGP(x, y, fid, 2)
            model.double().to(dev)
            elbo = VariationalELBOMF(model, N, 2)
            model.fix_variational_hypers(False)
            opt = Adam([{"params": model.parameters()}], lr=0.001, capturable=(mode == "graph"))
            fstep = FusedELBOStep(model, elbo)
            xd, yd, fd = x.to(dev), y.to(dev), fid.to(dev)
            perm = torch.randperm(N)
            xb, yb, fb = xd[perm.to(dev)], yd[perm.to(dev)], fd[perm.to(dev)]
            xb._mobo_host = x[perm]          # what the fitter's loader attaches: the Q4 test runs on the host
            if mode == "graph":
                gstep = GraphedELBOStep(fstep, opt, N)
                fn = lambda: gstep(xb, yb, fb)
            else:
                def fn():
                    fstep(xb, yb, fb, check_shortcut=False)
                    opt.step()
            for _ in range(10):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            res[mode + "_us_per_step"] = round(e0.elapsed_time(e1) / steps * 1e3, 1)
            if mode == "eager":
                res["kernels_per_step"] = _lib_launches_per_step(fn)
        res["steps_per_s"] = round(1e6 / res["graph_us_per_step"], 1)
        res["launch_floor"] = launch_floor(dev, res["kernels_per_step"])
        # K = 6 independent black-box models (4 objectives + 2 constraints, BASELINE.json configs[4]) trained round-robin,
        # one CUDA stream and one graph each (BlackBoxMFDGPFitter(concurrent_models=True)): their latency-bound chains
        # overlap on the GPU.  Wall clock between two device synchronisations.
        K = 6
        gsteps, streams = [], []
        for k in range(K):
            torch.manual_seed(k)
            model = MFDGP(x, y, fid, 2)
            model.double().to(dev)
            elbo = VariationalELBOMF(model, N, 2)
            model.fix_variational_hypers(False)
            opt = Adam([{"params": model.parameters()}], lr=0.001, capturable=True)
            gsteps.append(GraphedELBOStep(FusedELBOStep(model, elbo), opt, N))
            streams.append(torch.cuda.Stream(device=dev))
        for it in range(10 + steps):
            if it == 10:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
            for gs, st in zip(gsteps, streams):
                with torch.cuda.stream(st):
                    gs(xb, yb, fb)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        res["six_models_concurrent_us_per_model_step"] = round(dt / (steps * K) * 1e6, 1)
        res["six_models_concurrent_steps_per_s"] = round(steps * K / dt, 1)
        if name.startswith("C2"):
            res["conditioned_iteration_ms"] = bench_conditioned(dev, x, y, fid)
        res["get_nextpoint_coupled"] = bench_optimize(dev, x, y, fid)
        out[name] = res
    return out


def _lib_launches_per_step(fn):
    from mobocmf_b200 import _lib
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    fn()
    torch.cuda.synchronize()
    return int(_lib.launch_count() - n0)


def launch_floor(dev, nodes, reps=200):
    """SURVEY.md section 8d: what a step of `nodes` kernels costs when the kernels do nothing - a CUDA graph of `nodes`
    one-element kernels in ONE dependent chain (the upper bound of the step's critical path: its side-stream branches
    shorten it) and the same number in two parallel chains."""
    t = torch.zeros(2, device=dev)
    out = {"nodes": nodes}
    for name, chains in (("one_chain_us", 1), ("two_chains_us", 2)):
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(device=dev)
        with torch.cuda.graph(g):
            if chains == 2:
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    for _ in range(nodes // 2):
                        t[1:2].add_(0.0)
            for _ in range(nodes - (nodes // 2 if chains == 2 else 0)):
                t[0:1].add_(0.0)
            if chains == 2:
                torch.cuda.current_stream().wait_stream(side)
        for _ in range(5):
            g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        out[name] = round(e0.elapsed_time(e1) / reps * 1e3, 1)
    return out


def bench_optimize(dev, x, y, fid):
    """JESMOC_MFDGP.get_nextpoint_coupled (mobocmf/acquisition_functions/JESMOC_MFDGP.py:151-168: optimize_acqf per
    fidelity, 200 raw samples, 5 restarts, L-BFGS-B) with 2 objectives + 1 constraint: all fidelities' restarts in one
    batch whose value + gradient is replayed from a CUDA graph, vs the same optimiser enqueued eagerly, vs the oracle's
    coupled acquisition on the host (torch autograd, same optimiser, same seeds).  Wall clock."""
    from mobocmf_b200.acquisition_functions.JESMOC_MFDGP import JESMOC_MFDGP
    from mobocmf_b200.util.blackbox_mfdgp_fitter import BlackBoxMFDGPFitter
    from mobocmf_b200.util.optimize import optimize_acqf_multi
    torch.manual_seed(0)
    d = x.shape[1]
    fitter = BlackBoxMFDGPFitter(2, x.shape[0], num_epochs_1=3, num_epochs_2=3, device=dev, use_cuda_graph=True)
    fitter.verbose = False
    fitter.initialize_mfdgp(x, y, fid, "obj1")
    fitter.initialize_mfdgp(x, -y, fid, "obj2")
    fitter.initialize_mfdgp(x, torch.sin(7.85 * x.sum(1, keepdim=True)), fid, "con1", threshold_constraint=0.0,
                            is_constraint=True)
    fitter.train_mfdgps()
    g = torch.Generator().manual_seed(1)
    fitter.pareto_set = torch.rand(50, d, generator=g, dtype=torch.float64)
    fitter.pareto_front = torch.randn(50, 2, generator=g, dtype=torch.float64) * 0.3
    cond = fitter.copy_uncond()
    cond.pareto_set, cond.pareto_front = fitter.pareto_set, fitter.pareto_front
    with torch.no_grad():       # stand-in for the conditioned training: timing does not depend on the values
        for h in list(cond.mfdgp_handlers_objs.values()) + list(cond.mfdgp_handlers_cons.values()):
            for n, p in h.mfdgp.named_parameters():
                if "chol_variational_covar" in n:
                    p.mul_(0.7)
    bounds = torch.tensor([[0.0] * d, [1.0] * d], dtype=torch.float64, device=dev)
    acq = JESMOC_MFDGP(model=fitter, num_fidelities=2, model_cond=cond, standard_bounds=bounds)
    for f in range(2):
        acq.add_blackbox(f, "obj1", cost_evaluation=1.0 + 9.0 * f)
        acq.add_blackbox(f, "obj2", cost_evaluation=1.0 + 9.0 * f)
        acq.add_blackbox(f, "con1", cost_evaluation=1.0 + 9.0 * f, is_constraint=True)
    fns = [(lambda X, f=f: acq.coupled_acq(X, fidelity=f)) for f in range(2)]
    out = {}
    for mode, graph in (("graph", True), ("eager", False)):
        best = None
        for rep in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res, info = optimize_acqf_multi(fns, bounds, num_restarts=5, raw_samples=200, options={"maxiter": 200}, seed=0,
                                            use_cuda_graph=graph, return_info=True)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        out[mode + "_ms"] = round(best * 1e3, 2)
        out[mode + "_lbfgs_evaluations"] = info["evaluations"]
        out[mode + "_ms_per_evaluation"] = round(best * 1e3 / max(1, info["evaluations"]), 3)
        out[mode + "_values"] = [float(v) for _, v in res]
    try:
        from oracle import mfdgp_oracle as O
        from tests.helpers import oracle_view
        torch.set_num_threads(os.cpu_count() or 1)
        names = [("obj1", False), ("obj2", False), ("con1", True)]

        def mod(fit, name, is_con):
            sd, lo, up, smp = oracle_view(fit.get_model(name, is_constraint=is_con))
            return dict(sd=sd, num_layers=2, noise_upper=up, noise_lower=lo, samples=smp)
        mu = [mod(acq.blackbox_mfdgp_fitter_uncond, n, c) for n, c in names]
        mc = [mod(acq.blackbox_mfdgp_fitter_cond, n, c) for n, c in names]
        cfns = [(lambda X, f=f: O.coupled_acq(mu, mc, X, f, float32_accumulator=True)) for f in range(2)]
        t0 = time.perf_counter()
        res_c, info_c = optimize_acqf_multi(cfns, bounds.cpu(), num_restarts=5, raw_samples=200, options={"maxiter": 200},
                                            seed=0, use_cuda_graph=False, return_info=True)
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"ms": round(dt * 1e3, 1), "kind": "port", "cores": torch.get_num_threads(),
                               "lbfgs_evaluations": info_c["evaluations"],
                               "ms_per_evaluation": round(dt * 1e3 / max(1, info_c["evaluations"]), 3),
                               "values": [float(v) for _, v in res_c]}
    except Exception as e:       # the timing above stands without the host arm
        out["cpu_baseline"] = {"error": repr(e)[:200]}
    return out


def bench_conditioned(dev, x, y, fid, iters=100):
    """One conditioned iteration (_update_conditioned_models, mobocmf/util/blackbox_mfdgp_fitter.py:272-354) at the
    Forrester size with 2 objectives + 1 constraint and a 50-point Pareto set: enqueued eagerly vs replayed as one CUDA
    graph.  Wall clock between device synchronisations."""
    from mobocmf_b200.fused import Adam
    from mobocmf_b200.util.blackbox_mfdgp_fitter import BlackBoxMFDGPFitter
    out = {}
    for mode, use_graph in (("eager", False), ("graph", True)):
        torch.manual_seed(0)
        fitter = BlackBoxMFDGPFitter(2, x.shape[0], num_epochs_1=3, num_epochs_2=3, device=dev, use_cuda_graph=use_graph)
        fitter.verbose = False
        fitter.initialize_mfdgp(x, y, fid, "obj1")
        fitter.initialize_mfdgp(x, -y, fid, "obj2")
        fitter.initialize_mfdgp(x, torch.sin(7.85 * x), fid, "con1", threshold_constraint=0.0, is_constraint=True)
        fitter.train_mfdgps()
        g = torch.Generator().manual_seed(1)
        fitter.pareto_set = torch.rand(50, x.shape[1], generator=g, dtype=torch.float64)
        fitter.pareto_front = torch.randn(50, 2, generator=g, dtype=torch.float64) * 0.3
        cond = fitter.copy_uncond()
        cond.pareto_set, cond.pareto_front = fitter.pareto_set, fitter.pareto_front
        cond.verbose = False
        hs = (cond.mfdgp_handlers_objs.values(), cond.mfdgp_handlers_cons.values())
        params = [p for h in list(hs[0]) + list(hs[1]) for p in h.mfdgp.parameters()]
        for h in list(hs[0]) + list(hs[1]):
            h.mfdgp.fix_variational_hypers_cond(True)
        opt = Adam([{"params": params}], lr=1e-3, capturable=use_graph)
        for _ in range(5):
            cond._update_conditioned_models(hs[0], hs[1], opt)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(iters):
            cond._update_conditioned_models(hs[0], hs[1], opt)
        torch.cuda.synchronize()
        out[mode] = round((time.perf_counter() - t0) / iters * 1e3, 3)
    return out


def acq_models(model, dev, K=6, P=16):
    """K black boxes x (1 unconditioned + P Pareto-conditioned) MFDGPs: seeded perturbations of the bench model (cond
    params = uncond + perturbation of m and L_q, SURVEY.md section 8d C5; timing does not depend on the values)."""
    import copy
    g = torch.Generator(device=dev).manual_seed(7)
    boxes = []
    for k in range(K):
        u = copy.deepcopy(model)
        with torch.no_grad():
            for nme, p in u.named_parameters():
                if "variational_mean" in nme:
                    p.add_(0.05 * torch.randn(p.shape, generator=g, device=dev, dtype=p.dtype))
        conds = []
        for pp in range(P):
            c = copy.deepcopy(u)
            with torch.no_grad():
                for nme, p in c.named_parameters():
                    if "chol_variational_covar" in nme:
                        p.mul_(0.6 + 0.3 * (pp + 1) / P)
            conds.append(c)
        boxes.append((u, conds))
    return boxes


def acq_flop_per_candidate(cfg, K, P, S=25):
    """SURVEY.md section 8d: per candidate and model chain 1 layer-0 row + S rows in each of the L - 1 upper layers,
    F = 2 M^2 + 2 M + 3 d_l M flop per row; K (1 + P) chains -> 7.1e8 flop per candidate at C5."""
    M, d, L = cfg["M"], cfg["d"], cfg["L"]
    f0 = 2 * M * M + 2 * M + 3 * d * M
    f1 = 2 * M * M + 2 * M + 3 * (d + 1) * M
    return K * (1 + P) * (f0 + (L - 1) * S * f1)


def bench_acq(model, dev, cfg, world, rank, n=C5_CANDIDATES_PER_GPU, K=6, P=16, iters=1, with_cpu=True, n_grad=1024,
              dump=None):
    """JESMOC acquisition sweep, BASELINE.json configs[4] (SURVEY.md section 8d "C5"): every rank evaluates ITS n
    candidates (10^6 over 8 GPUs = 125 000 per GPU; candidates shard, no data-path collective) through the full coupled
    acquisition: K = 6 black boxes (4 objectives + 2 constraints) x (1 unconditioned + P = 16 Pareto-conditioned) MFDGPs
    = 102 model chains per candidate, each S = 25 samples through 3 layers (1 + 25 + 25 rows, M = 256), evaluated at
    the top fidelity:
        acq(x) = 1/P sum_p sum_k 1/2 max(0, log v_u,k(x) - log v_c,k,p(x))
    (mobocmf/acquisition_functions/JESMOC_MFDGP.py:38-52,125-135; mobocmf_b200...JESMOC_MFDGP.jes_sweep).  One 'eval'
    = one candidate through all 102 chains.  Legs: device-resident forward (value), end to end from pinned host
    memory (e2e), forward + d/dX on n_grad candidates (what optimize_acqf consumes), the CPU oracle on a bounded slice
    (rank 0, N = 1).  ``dump``: a dict that receives the values of the timed sweep."""
    import torch.distributed as dist
    from mobocmf_b200.acquisition_functions.JESMOC_MFDGP import jes_sweep
    fidelity = cfg["L"] - 1
    boxes = acq_models(model, dev, K, P)
    g = torch.Generator().manual_seed(1 + rank)
    Xh = torch.rand(n, cfg["d"], dtype=torch.float64, generator=g).pin_memory()
    X = Xh.to(dev)

    def sync_max(ms):
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    jes_sweep(X[:4096], fidelity, boxes)          # warm-up: operator buffers of the 102 models, allocator, kernels
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        out = jes_sweep(X, fidelity, boxes)
    e1.record()
    barrier()
    ms = sync_max(e0.elapsed_time(e1) / iters)
    if dump is not None:
        dump["acq_values"] = out.cpu()

    # end to end: candidates from pinned host memory, values back to pinned host memory, host waits for them
    vals_h = torch.empty(n, dtype=torch.float64).pin_memory()
    barrier()
    t0 = time.perf_counter()
    Xd = Xh.to(dev, non_blocking=True)
    vals_h.copy_(jes_sweep(Xd, fidelity, boxes), non_blocking=True)
    torch.cuda.synchronize()
    ms_e2e = sync_max((time.perf_counter() - t0) * 1e3)
    same = bool(torch.equal(vals_h, out.cpu()))

    # forward + d acq / dX (autograd over the composable kernels; saved whitened rows of all chains stay alive until
    # the backward, which bounds the candidate count of this leg)
    Xg = X[:n_grad].clone().requires_grad_(True)
    jes_sweep(Xg, fidelity, boxes).sum().backward()
    Xg.grad = None
    barrier()
    e0.record()
    v = jes_sweep(Xg, fidelity, boxes)
    v.sum().backward()
    e1.record()
    barrier()
    ms_g = sync_max(e0.elapsed_time(e1))
    grad_ok = bool(torch.isfinite(Xg.grad).all()) and float(Xg.grad.abs().max()) > 0.0
    fwd_vs_grad = float((v.detach() - out[:n_grad]).abs().max())

    chains = K * (1 + P)
    flop = acq_flop_per_candidate(cfg, K, P)
    tf = n * flop / (ms * 1e-3) / 1e12
    res = {"metric": "jesmoc_acq_evals_per_s", "value": world * n / (ms * 1e-3),
           "unit": "candidates/s through the full coupled acquisition (6 black boxes x (1 + 16) MFDGPs, S=25, "
                   "fidelity 2, forward)",
           "workload": "C5: %d candidates per GPU x 16 Pareto samples x (4 objectives + 2 constraints), d=6, L=3, "
                       "M=256, S=25 (10^6 candidates on 8 GPUs)" % n,
           "candidates_per_gpu": n, "candidates_total": world * n, "n_gpus": world, "ms_per_sweep": ms,
           "scaling": "weak", "model_chains_per_candidate": chains,
           "model_chain_evals_per_s": world * n * chains / (ms * 1e-3),
           "rows_per_s": world * n * chains * 51 / (ms * 1e-3), "acq_mean": float(out.mean()),
           "roofline": {"bound": "tensor", "kernel": "row_fwd_kernel (eval branch)", "achieved": tf,
                        "peak": FP64_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": tf / FP64_PEAK_TFLOPS, "traffic": None,
                        "algorithmic_flop_per_candidate": flop, "per_gpu": True,
                        "peak_source": "measured DMMA fp64 pipe peak, profiles/r01_fp64_probe.log"},
           "e2e": {"value": world * n / (ms_e2e * 1e-3), "unit": "candidates/s", "h2d_bytes_per_step": n * cfg["d"] * 8,
                   "d2h_bytes_per_step": n * 8, "ms_per_sweep": ms_e2e, "values_equal_device_run": same,
                   "note": "pinned host candidates -> H2D -> jes_sweep (102 chains) -> values D2H -> host sync"},
           "fwd_plus_dX": {"value": world * n_grad / (ms_g * 1e-3), "unit": "candidates/s (forward + d acq / dX)",
                           "candidates_per_gpu": n_grad, "ms": ms_g, "grad_finite_nonzero": grad_ok,
                           "max_abs_diff_vs_forward_only": fwd_vs_grad,
                           "note": "_JES-style autograd through the composable kernels (mobo_layer_rows_fwd/_bwd), "
                                   "the call optimize_acqf makes (acquisition_functions/JESMOC_MFDGP.py:142-143)"}}
    if with_cpu and world == 1 and rank == 0:
        res["cpu_baseline"] = acq_cpu_baseline(boxes, cfg, Xh, out, fidelity, K, P)
    return res


def acq_cpu_baseline(boxes, cfg, Xh, gpu_vals, fidelity, K, P, budget_s=20.0, chunk=200):
    """SURVEY.md section 8d: the oracle's coupled acquisition on a bounded slice of the SAME candidates in chunks of 200
    (= raw_samples of optimize_acqf), diagonal-only predictive variance, all host threads; plus ONE literal R x R
    eval-branch timing (what upstream's eval mode materialises) at the C3 grid size, 625 points x 25 samples."""
    from oracle import mfdgp_oracle as O
    from tests.helpers import oracle_view, random_state
    torch.set_num_threads(os.cpu_count() or 1)
    L = cfg["L"]
    mods = []
    for u, conds in boxes:
        vu = oracle_view(u)
        mods.append((vu, [oracle_view(c) for c in conds]))
    done, t_start, worst = 0, time.time(), 0.0
    with torch.no_grad():
        while done < Xh.shape[0]:
            Xc = Xh[done:done + chunk].clone()
            acc = torch.zeros(Xc.shape[0], dtype=torch.float64)
            for (sd, lo, up, smp), conds in mods:
                _, vu = O.predict_for_acquisition(sd, L, up, smp, Xc, fidelity, noise_lower=lo)
                for (sdc, loc, upc, smpc) in conds:
                    _, vc = O.predict_for_acquisition(sdc, L, upc, smpc, Xc, fidelity, noise_lower=loc)
                    acc += O.jes(vu, vc)
            acc /= P
            worst = max(worst, float((acc - gpu_vals[done:done + chunk].cpu()).abs().max()))
            done += Xc.shape[0]
            if time.time() - t_start > budget_s:
                break
    t = time.time() - t_start
    out = {"value": done / t, "unit": "candidates/s", "cores": torch.get_num_threads(), "kind": "port",
           "sample": "oracle coupled acquisition (102 chains, diagonal variance) on the first %d of the candidates in "
                     "chunks of %d: %.1f s" % (done, chunk, t),
           "max_abs_diff_vs_gpu": worst}
    try:    # literal R x R eval branch at the C3 size (d=2, L=2, M=15, 625 grid points x 25 samples = 15 625 rows)
        sd, up = random_state(15, 2, 2, seed=0, ls=0.3)
        g = torch.Generator().manual_seed(0)
        xt = torch.rand(625, 2, generator=g, dtype=torch.float64).repeat_interleave(25, 0)
        smp = torch.randn(25, generator=g).double()
        t0 = time.time()
        with torch.no_grad():
            m0, v0 = O.layer_q(sd, 0, xt, training=False, literal_eval_cov=True)
            f = (m0 + torch.sqrt(O.read_variance(v0)) * smp.repeat(625)).reshape(-1, 1)
            O.layer_q(sd, 1, torch.cat([xt, f], 1), training=False, literal_eval_cov=True)
        out["literal_RxR_eval_branch_C3"] = {"seconds_per_model_chain": time.time() - t0, "rows": 15625,
                                             "note": "upstream eval mode builds the R x R predictive covariance and "
                                                     "reads its diagonal; 2 layers, M = 15"}
    except (MemoryError, RuntimeError) as e:
        out["literal_RxR_eval_branch_C3"] = {"error": str(e)[:120]}
    return out


def bench_pareto(dev, d=6, L=3, F=500, K=6, iters=5, with_cpu=True):
    """Pareto-sample generation (SURVEY.md section 8f-3) at the C5 shape: K = 6 black boxes, each one RFF function
    sample of a 3-layer chain (F = 500 features per kernel), evaluated on MOOP's grid of 1000 d^2 = 36 000 points
    (mobocmf/util/moop.py:231), then the non-dominated cull of the 4 objectives.  Random draws as in
    _sample_from_prior (no model needed: the evaluation cost does not depend on theta)."""
    import numpy as np
    from mobocmf_b200.rff import RFFSample
    from mobocmf_b200.util.moop import pareto_mask
    rng = np.random.RandomState(0)
    n = 1000 * d * d

    def chain():
        t = lambda a: torch.as_tensor(a, dtype=torch.float64, device=dev)
        c = [dict(kind=0, nF=F, W=t(rng.normal(size=(F, d)) / (0.25 * d)), b=t(rng.uniform(0, 2 * np.pi, size=(F, 1))),
                  theta=t(rng.normal(size=F)), alpha=1.0)]
        for _ in range(L - 1):
            c.append(dict(kind=1, nF=F, W_x1=t(rng.normal(size=(F, d)) / (2.5 * d)), W_f=t(rng.normal(size=F)),
                          W_x2=t(rng.normal(size=(F, d)) / (0.25 * d)), b_x1=t(rng.uniform(0, 2 * np.pi, size=(F, 1))),
                          b_x2=t(rng.uniform(0, 2 * np.pi, size=(F, 1))), theta=t(rng.normal(size=3 * F)), alpha_x1=1.0,
                          alpha_x1f=1.0, alpha_x2=0.01, nu_lin=1.0))
        return c
    chains = [chain() for _ in range(K)]
    samples = [RFFSample(c, d, F, dev) for c in chains]
    grid = torch.as_tensor(rng.uniform(size=(n, d)), device=dev)
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    vals = None
    for it in range(iters + 2):
        if it == 2:
            e0.record()
        vals = torch.stack([s(grid) for s in samples[:4]] + [s(grid) for s in samples[4:]], dim=1)
    e1.record()
    for it in range(iters):
        mask = pareto_mask(vals[:, :4].contiguous())
    e2.record()
    torch.cuda.synchronize()
    ms_eval, ms_cull = e0.elapsed_time(e1) / iters, e1.elapsed_time(e2) / iters
    cos_per_point = F + (L - 1) * 3 * F        # one fp64 cos per (point, feature): 3500 per point and sample here
    out = {"metric": "rff_grid_evals_per_s", "value": K * n / (ms_eval * 1e-3), "unit": "grid points x function samples / s",
           "config": "C5 shape: d=6, 3-layer chains, F=500, %d-point grid, %d samples per pass" % (n, K),
           "ms_per_pass": ms_eval, "fp64_cos_per_s": K * n * cos_per_point / (ms_eval * 1e-3),
           "roofline_note": "FP64-pipe bound (DFMA + cos polynomial): ncu sm__inst_executed_pipe_fp64 35% of peak, "
                            "issue slots 60% (profiles/r01z_ncu_full_summary_rff_pareto.txt)",
           "pareto_cull_ms": ms_cull, "pareto_points": int(mask.sum()), "cull_pairs_per_s": n * n / (ms_cull * 1e-3)}
    if with_cpu:
        from oracle import rff_moop_oracle as R
        cpu_chain = [{k: (v.cpu().numpy() if torch.is_tensor(v) else v) for k, v in s.items()} for s in chains[0]]
        xs = grid[:4096].cpu().numpy()
        t0 = time.time()
        ref = R.eval_chain(cpu_chain, xs)[-1]
        t_cpu = time.time() - t0
        out["cpu_baseline"] = {"value": 4096 / t_cpu, "unit": out["unit"], "cores": os.cpu_count(), "kind": "port",
                               "sample": "numpy oracle, one sample on 4096 of the grid points (%.2f s)" % t_cpu,
                               "max_abs_diff_vs_gpu": float(np.abs(ref - vals[:4096, 0].cpu().numpy()).max())}
    return out


def cpu_baseline(cfg, x, y, fid, model, steps=8, warmup=2):
    """The oracle's tiled S-sample ELBO step (forward + autograd backward + Adam) on the host cores at the FULL C4
    configuration (B = 1024, M = 256, S = 64, L = 3), every step measured, nothing extrapolated.  This leg (and
    ``--impl reference``) is the only place where bench.py TIMES ``oracle/``."""
    from oracle import mfdgp_oracle as O
    from tests.helpers import oracle_view
    torch.set_num_threads(os.cpu_count() or 1)      # torchrun exports OMP_NUM_THREADS=1: use every host core anyway
    sd, lo, up, _ = oracle_view(model)
    names = [n for n, p in model.named_parameters() if p.requires_grad]
    for n in names:
        sd[n].requires_grad_(True)
    B, S, N, L = cfg["B"], cfg["S"], cfg["N"], cfg["L"]
    g = torch.Generator().manual_seed(5)
    opt = torch.optim.Adam([sd[n] for n in names], lr=0.001)
    times = []
    for it in range(warmup + steps):
        idx = torch.randint(0, N, (B,), generator=g)
        eps = [None] + [torch.randn(B * S, generator=g).double() for _ in range(1, L)]
        t0 = time.time()
        opt.zero_grad()
        loss, _ = O.elbo_step_loss_tiled(sd, L, up, x[idx], y[idx], fid[idx], eps, N, S, noise_lower=lo)
        loss.backward()
        opt.step()
        if it >= warmup:
            times.append(time.time() - t0)
    t = sum(times) / len(times)
    return {"value": 1.0 / t, "unit": "steps/s", "cores": torch.get_num_threads(), "kind": "port",
            "seconds_timed": sum(times), "steps_timed": len(times),
            "sample": "oracle tiled ELBO step (fwd + autograd bwd + torch Adam) at the full C4 step, B=1024, M=256, "
                      "S=64: mean %.3f s over %d steps after %d warm-up steps, nothing scaled" % (t, len(times), warmup)}


def parity_block(cfg, x, y, fid, model, fstep, dev):
    """CUDA vs CPU oracle on ONE C4 step (same parameters, minibatch and normals), outside the timed region: relative
    errors of the loss, the KL term and the worst gradient, with cond(K_zz + jitter I) and the bar they are held to
    (1e-10 on well-conditioned inputs, 20 * eps * cond otherwise; gradients 1e3 x that: SURVEY.md section 7)."""
    from oracle import mfdgp_oracle as O
    from tests.helpers import oracle_view, parity_tol, relerr
    torch.set_num_threads(os.cpu_count() or 1)
    B, S, N, L = cfg["B"], cfg["S"], cfg["N"], cfg["L"]
    g = torch.Generator().manual_seed(31)
    idx = torch.randint(0, N, (B,), generator=g)
    eps = [None] + [torch.randn(B * S, generator=g).double() for _ in range(1, L)]
    loss, kl = fstep(x[idx].to(dev), y[idx].to(dev), fid[idx].to(dev),
                     eps=[None if e is None else e.to(dev) for e in eps], num_samples=S)
    fstep.check()
    loss, kl = loss.clone(), kl.clone()
    grads = {n: p.grad.clone() for n, p in model.named_parameters() if p.requires_grad}
    sd, lo, up, _ = oracle_view(model)
    for n in grads:
        sd[n].requires_grad_(True)
    t0 = time.time()
    loss_o, kl_o = O.elbo_step_loss_tiled(sd, L, up, x[idx], y[idx], fid[idx], eps, N, S, noise_lower=lo)
    loss_o.backward()
    t_oracle = time.time() - t0
    worst, where = 0.0, None
    for n, gc in grads.items():
        go = sd[n].grad
        if "chol_variational_covar" in n:
            gc, go = torch.tril(gc), torch.tril(go)
        e = relerr(gc, go)
        if e > worst:
            worst, where = e, n
    tol, cond = parity_tol(model)
    return {"loss_relerr": relerr(loss, loss_o), "kl_relerr": relerr(kl, kl_o), "max_grad_relerr": worst,
            "max_grad_relerr_param": where, "cond": cond, "tol_values": tol, "tol_grads": 1e3 * tol,
            "ok": bool(relerr(loss, loss_o) < tol and relerr(kl, kl_o) < tol and worst < 1e3 * tol),
            "oracle_seconds": t_oracle, "retries": fstep.retries(),
            "what": "one C4 step (B=1024 x S=64, all parameters trainable) vs oracle/mfdgp_oracle.py on the host"}


def run_reference(args):
    """Reference arm: the reference's CPU implementation of the path.  GPyTorch/BoTorch are not installable here
    (SURVEY.md §8c), so this times the oracle port with all host threads on the SAME configuration: every one of the
    K steps is a full C4 step (B = 1024 x S = 64), W warm-up steps before them."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = dict(C4)
    x, y, fid = c4_data(cfg)
    from mobocmf_b200.models.mfdgp import MFDGP
    torch.manual_seed(cfg["seed"])
    model = MFDGP(x, y, fid, cfg["L"], num_inducing=cfg["M"], init_lengthscale=cfg["lengthscale"])
    model.double()
    model.fix_variational_hypers(False)
    cb = cpu_baseline(cfg, x, y, fid, model, steps=max(1, args.steps), warmup=max(1, args.warmup))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    out = {"impl": "reference", "metric": "mfdgp_elbo_steps_per_s", "value": cb["value"], "unit": "steps/s",
           "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 / cb["value"],
           "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": workload_config(world, args.scaling, cfg["B"]),
           "reference_note": "CPU oracle port of the reference path (GPyTorch is not installable here); one process, "
                             "one 1024 x 64 step unit at a time whatever --gpus says",
           "cpu_baseline": cb,
           "e2e": {"value": cb["value"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--path", default="fused", choices=["fused", "composable"],
                    help="fused: mobo_elbo_step + mobo_adam (product hot loop); composable: autograd over the same kernels")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: one 1024 x 64 step unit per GPU; strong: one 1024 x 64 step split over the GPUs")
    ap.add_argument("--allreduce", default="single", choices=["overlapped", "single"],
                    help="multi-GPU gradient exchange: per-layer buckets behind the row kernels, or one all-reduce")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--no-acq", action="store_true", help="skip the acquisition sweep and the small-config legs")
    ap.add_argument("--no-parity", action="store_true", help="skip the CUDA-vs-oracle parity block")
    ap.add_argument("--acq-candidates", type=int, default=C5_CANDIDATES_PER_GPU,
                    help="candidates per GPU of the C5 acquisition sweep (10^6 / 8 by default)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (loss, gradients, updated parameters) and the values "
                         "of the timed acquisition sweep as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
