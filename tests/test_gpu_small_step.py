"""The single-kernel ELBO step of small MFDGPs (mobo_elbo_step_small, fused.SmallModelsELBOStep): parity with the
fused step (mobo_elbo_step) and the oracle, independence of the models of one launch, failure flags, accumulation,
rejected shapes, a graphed training loop and the fitter's routing."""
import copy

import pytest
import torch

from oracle import mfdgp_oracle as O
from tests.helpers import adjudicate_step, forrester_data, oracle_view, parity_tol, relerr, synthetic_data

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def make_model(L=2, M=16, d=2, ls=0.3, seed=1, n_per=None):
    """A perturbed L-fidelity MFDGP on seeded synthetic data with its first M inputs as inducing inputs."""
    from mobocmf_b200.models.mfdgp import MFDGP
    n_per = n_per or [max(M, 24)] + [12] * (L - 1)
    x, y, fid = synthetic_data(list(n_per[:L]), d, seed=3 + seed)
    N = x.shape[0]
    g = torch.Generator().manual_seed(seed)
    perm = torch.randperm(N, generator=g)
    x, y, fid = x[perm], y[perm], fid[perm]
    model = MFDGP(x, y, fid, L, num_inducing=M, init_lengthscale=ls)
    model.double()
    with torch.no_grad():     # move off the initial point so that every term matters
        for n, p in model.named_parameters():
            if "chol_variational_covar" in n:
                p.add_(torch.tril(torch.randn(p.shape, generator=g, dtype=p.dtype)) * 0.02 / p.shape[0] ** 0.5)
                p.diagonal().abs_().add_(0.05)
            else:
                p.add_(0.1 * torch.randn(p.shape, generator=g, dtype=p.dtype))
    return model.to(DEV), x, y, fid, N


def freeze(model, how):
    if how == "phase1":
        model.fix_variational_hypers(True)
    elif how == "cond":
        model.fix_variational_hypers_cond(True)


def draw_batch(x, y, fid, B, S, L, seed):
    g = torch.Generator().manual_seed(seed)
    idx = torch.randint(0, x.shape[0], (B,), generator=g)
    eps = [None] + [torch.randn(B * S, generator=g).double() for _ in range(1, L)]
    return idx, eps


def grads(model):
    return {n: (None if p.grad is None else p.grad.detach().clone()) for n, p in model.named_parameters()}


def small_step(models, elbos):
    from mobocmf_b200.fused import SmallModelsELBOStep
    return SmallModelsELBOStep(models, elbos)


# (L, S, B, M, d, freeze): together M in {1, 16, 31, 32, 33, 64}, L in {1, 2, 3}, S in {1, 4}, B in {1, 16, 75},
# d in {1, 2, 8} and every freeze set
CASES = [(1, 1, 16, 16, 1, None), (2, 4, 16, 31, 2, "phase1"), (3, 1, 75, 32, 8, "cond"), (2, 1, 1, 33, 2, None),
         (3, 4, 16, 64, 2, None), (2, 1, 75, 64, 1, "cond"), (2, 4, 75, 1, 2, "phase1"), (3, 4, 1, 16, 8, None)]


def test_cases_cover_the_edges():
    col = list(zip(*CASES))
    assert set(col[0]) == {1, 2, 3} and set(col[1]) == {1, 4} and {1, 16, 75} <= set(col[2])
    assert {1, 16, 31, 32, 33, 64} <= set(col[3]) and {1, 2, 8} <= set(col[4]) and set(col[5]) == {None, "phase1", "cond"}


def _check_parity(model, elbo, x, y, fid, idx, eps, N, L, S):
    from mobocmf_b200.fused import FusedELBOStep
    xb, yb, fb = x[idx].to(DEV), y[idx].to(DEV), fid[idx].to(DEV)
    eps_d = [None if e is None else e.to(DEV) for e in eps]
    tol, cond = parity_tol(model)
    ref = FusedELBOStep(model, elbo)
    loss_f, kl_f = [t.clone() for t in ref(xb, yb, fb, eps=eps_d, num_samples=S)]
    ref.check()
    g_f = grads(model)
    for p in model.parameters():
        if p.grad is not None:
            p.grad.fill_(float("nan"))     # every gradient must be written by the small step
    small = small_step([model], [elbo])
    (loss, kl), = small([(xb, yb, fb)], eps=[eps_d], num_samples=S)
    small.steps[0].check()
    g_s = grads(model)
    print("cond %.2e: loss relerr vs fused step %.2e" % (cond, relerr(loss, loss_f)))
    # Both steps are fp64 programs of the same formulation that differ in the order of their sums (DMMA products and
    # a blocked factorisation there, FMA loops here).  On well-conditioned inputs that leaves the loss equal to 1e-12;
    # at cond(K_zz) >= 1e5 both are ~eps * cond from the exact loss, so neither is the judge of the other: the bar is
    # the parity tolerance, and the longdouble truth below decides which is right
    bar = 1e-12 if cond < 1e5 else tol
    assert relerr(loss, loss_f) < bar and relerr(kl, kl_f) < bar, (relerr(loss, loss_f), relerr(kl, kl_f), cond)
    for n, p in model.named_parameters():
        if not p.requires_grad:
            assert g_s[n] is None, n
            continue
        a, b = g_s[n], g_f[n]
        if "chol_variational_covar" in n:
            assert torch.equal(torch.triu(a, 1), torch.zeros_like(a)), n
        assert relerr(a, b) < max(1e-9, 30 * tol), (n, relerr(a, b), cond)
    # oracle
    sd, lo, up, _ = oracle_view(model)
    names = [n for n, p in model.named_parameters() if p.requires_grad]
    for n in names:
        sd[n].requires_grad_(True)
    loss_o, kl_o = O.elbo_step_loss_tiled(sd, L, up, x[idx], y[idx], fid[idx], eps, N, S, noise_lower=lo)
    loss_o.backward()
    if cond >= 1e5:
        adjudicate_step(model, loss, g_s, loss_o.detach(), {n: sd[n].grad for n in names}, L, x[idx], y[idx],
                        fid[idx], eps, N, S)
        return
    assert relerr(loss, loss_o) < tol and relerr(kl, kl_o) < tol
    for n in names:
        a = g_s[n]
        b = sd[n].grad if sd[n].grad is not None else torch.zeros_like(sd[n])   # no row of the minibatch reaches it
        if "chol_variational_covar" in n:
            a, b = torch.tril(a), torch.tril(b)
        assert relerr(a, b) < 1e3 * tol, (n, relerr(a, b))


@pytest.mark.parametrize("L,S,B,M,d,how", CASES)
def test_small_step_matches_fused_step_and_oracle(L, S, B, M, d, how):
    from mobocmf_b200.mlls.variational_elbo_mf import VariationalELBOMF
    model, x, y, fid, N = make_model(L=L, M=M, d=d, ls=0.3 if d < 8 else 0.9)
    freeze(model, how)
    elbo = VariationalELBOMF(model, N, L)
    idx, eps = draw_batch(x, y, fid, B, S, L, seed=2)
    _check_parity(model, elbo, x, y, fid, idx, eps, N, L, S)


def test_small_step_forrester_reference_defaults():
    """The reference's own Forrester model (TL.MEDIAN lengthscale, M = N = 16, cond(K_zz) ~ 1e7): judged by the
    longdouble truth."""
    from mobocmf_b200.mlls.variational_elbo_mf import VariationalELBOMF
    from mobocmf_b200.models.mfdgp import MFDGP
    x, ys, fid = forrester_data()
    torch.manual_seed(0)
    model = MFDGP(x, ys["obj1"], fid, 2)
    model.double().to(DEV)
    elbo = VariationalELBOMF(model, 16, 2)
    idx, eps = draw_batch(x, ys["obj1"], fid, 16, 1, 2, seed=5)
    _check_parity(model, elbo, x, ys["obj1"], fid, idx, eps, 16, 2, 1)


def _hetero():
    """Models of different L, d, M, B, S and frozen sets with their minibatches and normals."""
    from mobocmf_b200.mlls.variational_elbo_mf import VariationalELBOMF
    out = []
    for k, (L, S, B, M, d, how) in enumerate([(2, 1, 16, 16, 1, None), (3, 4, 20, 33, 2, "phase1"),
                                               (1, 1, 75, 64, 3, None), (2, 2, 5, 8, 8, "cond")]):
        model, x, y, fid, N = make_model(L=L, M=M, d=d, seed=10 + k, ls=0.3 if d < 8 else 0.9)
        freeze(model, how)
        elbo = VariationalELBOMF(model, N, L)
        idx, eps = draw_batch(x, y, fid, B, S, L, seed=20 + k)
        out.append(dict(model=model, elbo=elbo, S=S, batch=(x[idx].to(DEV), y[idx].to(DEV), fid[idx].to(DEV)),
                        eps=[None if e is None else e.to(DEV) for e in eps]))
    return out


def test_models_of_one_launch_are_independent():
    """Heterogeneous models (L, d, M, B, S, frozen sets) in one launch: each result is bit-identical to launching the
    model alone, and two launches are bit-identical."""
    from mobocmf_b200 import _lib
    ms = _hetero()
    alone = []
    for m in ms:
        st = small_step([m["model"]], [m["elbo"]])
        st([m["batch"]], eps=[m["eps"]], num_samples=m["S"])
        alone.append((st.steps[0].out.clone(), grads(m["model"])))
    st = small_step([m["model"] for m in ms], [m["elbo"] for m in ms])
    for rep in range(2):
        n0 = _lib.launch_count()
        st([m["batch"] for m in ms], eps=[m["eps"] for m in ms], num_samples=[m["S"] for m in ms])
        assert _lib.launch_count() - n0 == 1
        for m, s, (a_out, a_g) in zip(ms, st.steps, alone):
            assert torch.equal(s.out, a_out), rep
            for n, g in grads(m["model"]).items():
                assert (g is None and a_g[n] is None) or torch.equal(g, a_g[n]), (rep, n)


def _retry_model(extra, seed):
    """A one-layer model whose K_zz + jitter I needs the retries that add `extra` to the diagonal: jitter =
    -lambda_min(K_zz) - extra / 2 (psd_safe_cholesky adds 1e-8, then 1e-7, then 1e-6 in total)."""
    from mobocmf_b200.mlls.variational_elbo_mf import VariationalELBOMF
    model, x, y, fid, N = make_model(L=1, M=16, d=2, seed=seed)
    sd, _, _, _ = oracle_view(model)
    Z = O.layer_inducing_points(sd, 0)
    lam = float(torch.linalg.eigvalsh(O.layer_kernel(sd, 0, Z, Z)).min())
    model.hidden_layer_0.variational_strategy.jitter_val = -lam - extra / 2
    return model, VariationalELBOMF(model, N, 1), x, y, fid


def test_retries_and_failures_in_one_launch():
    from mobocmf_b200.errors import NanError, NotPSDError
    from mobocmf_b200.fused import Adam, FusedELBOStep, GraphedSmallModelsELBOStep, SmallModelsELBOStep
    from mobocmf_b200.mlls.variational_elbo_mf import VariationalELBOMF
    specs = [("ok", None), ("r1", 1e-8), ("r2", 1e-7), ("r3", 1e-6), ("fail", 4e-6), ("nan", None)]
    models, elbos, batches = [], [], []
    for k, (tag, extra) in enumerate(specs):
        if extra is None:
            model, x, y, fid, N = make_model(L=1, M=16, d=2, seed=30 + k)
            elbo = VariationalELBOMF(model, N, 1)
        else:
            model, elbo, x, y, fid = _retry_model(extra, seed=30 + k)
        idx = torch.arange(20)
        yb = y[idx].clone()
        if tag == "nan":
            yb[3] = float("nan")
        models.append(model); elbos.append(elbo)
        batches.append((x[idx].to(DEV), yb.to(DEV), fid[idx].to(DEV)))
    # the composable reference: mobo_elbo_step per model
    ref = []
    for m, e, b in zip(models, elbos, batches):
        f = FusedELBOStep(m, e)
        f(*b)
        ref.append(f.out.clone())
    small = SmallModelsELBOStep(models, elbos)
    small(batches)
    for (tag, _), s, r in zip(specs, small.steps, ref):
        assert torch.equal(s.out[3:8], r[3:8]), (tag, s.out.tolist(), r.tolist())
    assert [int(s.out[7]) for s in small.steps] == [0, 1, 2, 3, 3, 0]
    assert [int(s.out[3]) for s in small.steps] == [0, 0, 0, 0, 1, 0]
    assert float(small.steps[5].out[5]) == 1.0 and float(small.steps[5].out[6]) == 1.0
    # graphed step + Adam: only the failed models' parameters stay where they were
    opts = [Adam([{"params": m.parameters()}], lr=0.01, capturable=True) for m in models]
    before = [[p.detach().clone() for p in m.parameters()] for m in models]
    gs = GraphedSmallModelsELBOStep(small, opts)
    gs(batches)
    for (tag, _), m, b in zip(specs, models, before):
        same = all(torch.equal(a, p.detach()) for a, p in zip(b, m.parameters()))
        assert same == (tag in ("fail", "nan")), tag
    for (tag, _), s in zip(specs, small.steps):
        if tag == "fail":
            with pytest.raises(NotPSDError):
                s.check()
        elif tag == "nan":
            with pytest.raises(NanError):
                s.check()
        else:
            s.check()


def test_accumulate_adds_to_existing_gradients():
    ms = _hetero()
    st = small_step([m["model"] for m in ms], [m["elbo"] for m in ms])
    kw = dict(eps=[m["eps"] for m in ms], num_samples=[m["S"] for m in ms])
    st([m["batch"] for m in ms], **kw)
    g1 = [grads(m["model"]) for m in ms]
    st([m["batch"] for m in ms], accumulate=True, **kw)
    for m, g in zip(ms, g1):
        for n, p in m["model"].named_parameters():
            if p.requires_grad:
                assert torch.equal(p.grad, 2 * g[n]), n


def test_unsupported_shapes_are_rejected_before_any_launch():
    from mobocmf_b200 import _lib
    from mobocmf_b200.fused import StepDesc
    lib = _lib.load()
    assert lib.mobo_elbo_step_small_workspace_doubles(2, 1, 16, 1, 16) > 0
    good = dict(L=2, d=1, M=16, B=16)
    for bad in (dict(M=65), dict(d=9), dict(L=0), dict(L=9), dict(B=0), dict(M=0), dict(d=0)):
        arr = (StepDesc * 2)()
        for i in range(2):
            for k, v in good.items():
                setattr(arr[i], k, v)
        for k, v in bad.items():
            setattr(arr[1], k, v)
        n0 = _lib.launch_count()
        assert lib.mobo_elbo_step_small(arr, 2, _lib.stream_ptr()) == -2, bad
        assert _lib.launch_count() == n0, bad
        s = dict(good, **bad)
        assert lib.mobo_elbo_step_small_workspace_doubles(s["L"], s["d"], s["M"], 1, s["B"]) == 0, bad
    n0 = _lib.launch_count()
    assert lib.mobo_elbo_step_small((StepDesc * 1)(), 0, _lib.stream_ptr()) == -2
    assert _lib.launch_count() == n0


def _forrester_models(k):
    """k Forrester-sized models (d = 1, 2 fidelities, N = M = B = 16) on evenly spaced inputs with lengthscale 0.06,
    cond(K_zz + jitter I) ~ 1e4, and likelihood noise 1e-2.  An implementation-parity bar over 20 Adam steps needs a
    well-conditioned problem: the Forrester example's own inputs hold pairs 0.009 apart (cond ~ 1e7 at any usable
    lengthscale), and the initial layer-0 noise of 1e-6 scales rounding in the means by 1 / noise in the loss and its
    gradients; two fp64 programs differ there by far more than 1e-9 after one step, which Adam carries into the
    parameters.  The ill-conditioned regime is judged step by step against the longdouble truth above."""
    from mobocmf_b200.mlls.variational_elbo_mf import VariationalELBOMF
    from mobocmf_b200.models.mfdgp import MFDGP
    x = torch.linspace(0, 1, 16, dtype=torch.float64)[:, None]
    fid = torch.zeros(16, 1, dtype=torch.float64)
    fid[::4] = 1.0
    f1 = ((6 * x - 2) ** 2) * torch.sin(12 * x - 4)
    f0 = 0.5 * f1 + 10 * (x - 0.5) + 5
    out = []
    for i, sign in enumerate((1.0, -1.0, 0.5)[:k]):
        y = sign * torch.where(fid > 0, f1, f0)
        y = (y - y.mean()) / y.std()
        torch.manual_seed(i)
        model = MFDGP(x, y, fid, 2, init_lengthscale=0.06)
        model.double()
        for l in range(2):
            getattr(model, "hidden_layer_likelihood_%d" % l).noise = 1e-2
        model.to(DEV)
        out.append((model, VariationalELBOMF(model, 16, 2), y))
    return x, fid, out


def test_graphed_training_loop_matches_graphed_fused_steps_and_eager():
    from mobocmf_b200.fused import (Adam, FusedELBOStep, GraphedELBOStep, GraphedSmallModelsELBOStep,
                                    SmallModelsELBOStep)
    x, fid, ms = _forrester_models(3)
    copies = [copy.deepcopy(m) for m, _, _ in ms]
    eager = [copy.deepcopy(m) for m, _, _ in ms]
    from mobocmf_b200.mlls.variational_elbo_mf import VariationalELBOMF
    e2 = [VariationalELBOMF(m, 16, 2) for m in copies]
    e3 = [VariationalELBOMF(m, 16, 2) for m in eager]
    o1 = [Adam([{"params": m.parameters()}], lr=0.01, capturable=True) for m, _, _ in ms]
    o2 = [Adam([{"params": m.parameters()}], lr=0.01, capturable=True) for m in copies]
    o3 = [Adam([{"params": m.parameters()}], lr=0.01, capturable=True) for m in eager]
    gsmall = GraphedSmallModelsELBOStep(SmallModelsELBOStep([m for m, _, _ in ms], [e for _, e, _ in ms]), o1,
                                        static_eps=True)
    gfused = [GraphedELBOStep(FusedELBOStep(m, e), o, 16, static_eps=True) for m, e, o in zip(copies, e2, o2)]
    esmall = SmallModelsELBOStep(eager, e3)
    for o, s in zip(o3, esmall.steps):
        o.skip_flag = s.skip_flag
    g = torch.Generator().manual_seed(7)
    first, last = None, None
    for it in range(20):
        batches, eps = [], []
        for _, _, y in ms:
            perm = torch.randperm(16, generator=g)
            perm = torch.roll(perm, 1) if torch.equal(perm, torch.arange(16)) else perm
            batches.append((x[perm].to(DEV), y[perm].to(DEV), fid[perm].to(DEV)))
            eps.append([None, torch.randn(16, generator=g).double().to(DEV)])
        res = gsmall(batches, eps=eps)
        ref = [gf(*b, eps=e) for gf, b, e in zip(gfused, batches, eps)]
        res_e = esmall(batches, eps=eps)
        for o in o3:
            o.step()
        for (l1, _), (l2, _), (l3, _) in zip(res, ref, res_e):
            assert relerr(l1, l2) < 1e-9, (it, relerr(l1, l2))
            assert torch.equal(l1, l3), it
        tot = sum(float(r[0]) for r in res)
        first = tot if first is None else first
        last = tot
    assert last < first
    for (m, _, _), c, e in zip(ms, copies, eager):
        for (n, a), (_, b), (_, c_) in zip(m.named_parameters(), c.named_parameters(), e.named_parameters()):
            assert relerr(a, b) < 1e-8, (n, relerr(a, b))
            assert torch.equal(a, c_), n


def test_fitter_routes_small_models_to_one_launch_per_batch():
    from mobocmf_b200.errors import NotPSDError
    from mobocmf_b200.util.blackbox_mfdgp_fitter import BlackBoxMFDGPFitter
    x, ys, fid = forrester_data()

    def fitter_for():
        torch.manual_seed(0)
        f = BlackBoxMFDGPFitter(2, 16, num_epochs_1=4, num_epochs_2=4, device=torch.device(DEV),
                                use_cuda_graph=True, concurrent_models=True)
        f.verbose = False
        for name in ("obj1", "obj2", "con1"):
            f.initialize_mfdgp(x, ys[name], fid, name, is_constraint=name.startswith("con"))
        return f

    f = fitter_for()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        f._train_mfdgp(f._update_model, fix_variational_hypers=True, num_epochs=4, lr=0.003)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    # B = N = 16: one batch index per epoch.  Per group (2 objectives, 1 constraint) the graph is built at the first
    # batch index (3 eager warm-up steps, then the capture, which runs nothing) and replayed at every batch index: 3 + 4
    # executions of small_step_kernel, each ONE launch for all models of the group; nothing of mobo_elbo_step's
    # sequence runs
    assert sum("small_step_kernel" in n for n in names) == 2 * (3 + 4), [n for n in names if "step" in n]
    assert not any(k in n for n in names for k in ("opchain_kernel", "row_fwd_kernel", "ell_kernel",
                                                   "step_finish_kernel"))
    small = f._small_steps
    assert sorted(len(s.steps) for s in small.values()) == [1, 2]
    for h in list(f.mfdgp_handlers_objs.values()) + list(f.mfdgp_handlers_cons.values()):
        assert all(bool(torch.isfinite(p).all()) for p in h.mfdgp.parameters())
    # a model whose factorisation fails surfaces at the reporting boundary
    f = fitter_for()
    bad = f.mfdgp_handlers_objs["obj2"].mfdgp
    for l in range(2):
        getattr(bad, "hidden_layer_%d" % l).variational_strategy.jitter_val = -1e-2
    with pytest.raises(NotPSDError):
        f._train_mfdgp(f._update_model, fix_variational_hypers=True, num_epochs=2, lr=0.003)
