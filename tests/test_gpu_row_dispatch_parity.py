"""The acquisition chain and the training rows against the fp64 oracle at every input dimension d = 1 .. 8 and in
every sample-tiling regime of the row kernels.

The row kernels are instantiated per d (`build_k_tile<KIND, D, SHX>`, `kgrad_tile<KIND, D, PARAM, XGRAD, SHX>`), and
above layer 0 the forward takes one of three shapes, chosen from xrep = S (the acquisition samples per candidate):
  * S = 1 .. 3:   the generic kernel, no warp of which shares one x over its 4 rows;
  * S = 4 .. 10:  the generic kernel with SHX warps (all warps at S = 4 and 8, some at the other S);
  * S >= 11:      `row_fwd_ws_kernel`, which evaluates the x-kernels once per distinct x of a 32-row tile (at most 4).
A case of those switches dispatched to the wrong instantiation, or an x-kernel loop that drops dimensions, changes the
numbers only at the d and S it concerns, so every case below is compared with an independent fp64 reference (the
oracle's formulas under CPU autograd), not with another path through the same kernels.  The GPU tests are marked one by
one; the table's coverage test runs on the CPU."""
import numpy as np
import pytest
import torch

from mobocmf_b200 import _lib
from oracle import mfdgp_oracle as O
from tests.helpers import adjudicate, model_from_state, oracle_view, parity_tol, random_state, relerr, state_cond

DEV = "cuda:0"
EPS64 = 2.220446049250313e-16
COND_MAX = 1e5        # every table case stays below this cond(K_zz + jitter I), so that it is judged by the tight bar
XSHARE_MIN_REP = 11   # row_pass.cu: rows with xrep >= this go to row_fwd_ws_kernel
TR = 32               # rows per tile of the row kernels

# ---- 1. the case table ------------------------------------------------------------------------------------------
# One M per d, and two acquisition shapes (S, n): one on the generic forward (S <= 10), one on row_fwd_ws_kernel (S >= 11).
# S = 11 puts 4 distinct x in some tiles (the most the ws kernel holds), S = 40 gives tiles with fewer rows than S.
# M = 20, 33, 65, 96, 200 leave 12, 31, 31, 0, 24 padded columns of MP.  n is small (the oracle runs on the CPU) and
# n * S is mostly not a multiple of 4 or 32, so that last tiles and last warp groups are ragged.  The lengthscale keeps
# cond(K_zz + jitter I) <= COND_MAX on every layer of both the model and its conditioned copy (asserted).
# `rows_S` is the S of the training-rows case on the generic kernel; it has SHX warps (4 <= S <= 10).
#       d    M    ls     (S, n) generic  (S, n) ws   rows_S
TABLE = [
    (1,  20, 0.035, (7, 13),   (25, 13),  7),
    (2,  33, 0.18,  (3, 37),   (11, 1),   8),
    (3,  48, 0.3,   (4, 29),   (40, 9),   4),
    (4,  96, 0.35,  (7, 23),   (11, 31),  7),
    (5, 200, 0.3,   (10, 17),  (25, 11),  10),
    (6, 256, 0.4,   (1, 19),   (12, 27),  5),
    (7,  65, 0.8,   (4, 35),   (25, 7),   4),
    (8, 256, 0.5,   (7, 39),   (11, 21),  7),
]
L3 = 3
# A four-layer chain: a third upper layer (prep = 1 above layer 1) and a four-layer dX fold.
L4_CASE = (3, 48, 0.3, 4, 7, 15)            # d, M, ls, L, S, n

ACQ_CASES = [(d, M, ls, L3, S, n) for d, M, ls, gen, ws, _ in TABLE for S, n in (gen, ws)] + [L4_CASE]
ROWS_CASES = [(d, M, ls, S, n) for d, M, ls, gen, ws, rows_S in TABLE for S, n in ((rows_S, gen[1]), ws)]


def case_id(c):
    return "d%d-M%d-L%d-S%d-n%d" % (c[0], c[1], c[3], c[4], c[5])


def seed_of(d, L):
    return 100 + d + 10 * (L - 3)


def distinct_x_per_tile(S, n):
    """Most distinct candidates any 32-row tile of the n * S rows (row r reads candidate r // S) holds."""
    R = n * S
    return max((min(R, t + TR) - 1) // S - t // S + 1 for t in range(0, R, TR))


def test_case_table_covers_every_dimension_and_regime():
    assert sorted(c[0] for c in TABLE) == list(range(1, 9))
    for d, M, ls, (sg, ng), (sw, nw), rows_S in TABLE:
        assert 1 <= sg < XSHARE_MIN_REP <= sw, d
        assert 4 <= rows_S < XSHARE_MIN_REP, d                  # generic kernel with SHX warps
        assert distinct_x_per_tile(sw, nw) <= 4, d              # the ws kernel's XMAX
        assert max(ng, nw) <= 40, d                             # the oracle's n stays small
    S_all = {S for c in TABLE for S, _ in (c[3], c[4])}
    assert {1, 3, 4, 7, 11, 12, 25, 40} <= S_all
    assert any(distinct_x_per_tile(sw, nw) == 4 for _, _, _, _, (sw, nw), _ in TABLE)
    assert any(sw > TR for _, _, _, _, (sw, _), _ in TABLE)
    Ms = {c[1] for c in TABLE}
    assert {20, 33, 65, 96, 200, 256} <= Ms and any(M % 32 == 1 for M in Ms)
    shapes = [(S, n) for c in TABLE for S, n in (c[3], c[4])]
    assert any(n == 1 for _, n in shapes)
    assert sum((n * S) % 4 != 0 for S, n in shapes) > len(shapes) // 2
    assert L4_CASE[3] == 4 and 4 <= L4_CASE[4] < XSHARE_MIN_REP
    for d in range(1, 9):
        rows_S = sorted(S for dd, _, _, S, _ in ROWS_CASES if dd == d)
        assert len(rows_S) == 2 and 4 <= rows_S[0] < XSHARE_MIN_REP <= rows_S[1], d


# ---- fixtures ---------------------------------------------------------------------------------------------------
_MODELS = {}


def conditioned_state(sd, seed):
    """A conditioned copy's state: shifted variational means, a more certain q(u)."""
    g = torch.Generator().manual_seed(seed + 7)
    out = {k: v.clone() for k, v in sd.items()}
    for k in out:
        if "variational_mean" in k:
            out[k] = out[k] + 0.05 * torch.randn(out[k].shape, generator=g, dtype=torch.float64)
        if "chol_variational_covar" in k:
            out[k] = out[k] * 0.6
    return out


def models(d, M, ls, L, S):
    """(model, conditioned copy) with the same S eval samples per layer (quirk Q7), in eval mode; cached per shape."""
    key = (d, M, ls, L, S)
    if key not in _MODELS:
        seed = seed_of(d, L)
        sd, up = random_state(M, d, L, seed=seed, ls=ls)
        g = torch.Generator().manual_seed(seed + S)
        samples = [torch.randn(S, 1, generator=g) for _ in range(L)]
        pair = (model_from_state(sd, up, L, samples=samples),
                model_from_state(conditioned_state(sd, seed), up, L, samples=samples))
        for m in pair:
            m.eval()
        _MODELS[key] = pair
    return _MODELS[key]


def candidates(n, d, seed):
    g = torch.Generator().manual_seed(1000 + seed)
    return torch.rand(n, 1, d, generator=g, dtype=torch.float64)


def weights(n):
    return torch.linspace(-1.0, 2.0, n, dtype=torch.float64)


def noise_key(fidelity):
    return "hidden_layer_likelihood_%d.noise_covar.raw_noise" % fidelity


def kernels_run(fn):
    """fn's result and the names of the library's kernels it launched."""
    _lib.profile_enable(True)
    try:
        out = fn()
        return out, {name for name, _ in _lib.profile_collect()}
    finally:
        _lib.profile_enable(False)


def cuda_grads(model, cond, X, fidelity, upstream):
    """(dX, d raw_noise of `model`) of one scalar of the fused chain: w . mu, w . var or the JES sum."""
    from mobocmf_b200.acquisition_functions.JESMOC_MFDGP import _JES_MFDGP
    Xg = X.to(DEV).requires_grad_(True)
    if upstream == "jes":
        loss = _JES_MFDGP(fidelity, model, cond)(Xg).sum()
        model.eval(); cond.eval()           # _JES_MFDGP leaves the models in training mode
    else:
        mu, var = model.predict_for_acquisition(Xg, fidelity)
        loss = (weights(X.shape[0]).to(DEV) * (mu if upstream == "mu" else var)).sum()
    rn = getattr(model, "hidden_layer_likelihood_%d" % fidelity).noise_covar.raw_noise
    gx, gn = torch.autograd.grad(loss, [Xg, rn], allow_unused=True)
    return gx.cpu(), (torch.zeros(1, dtype=torch.float64) if gn is None else gn.cpu())


def oracle_module(model):
    sd, lo, up, samples = oracle_view(model)
    return dict(sd=sd, num_layers=model.num_fidelities, noise_upper=up, noise_lower=lo, samples=samples)


def oracle_chain(mod, X, fidelity):
    """fp64 oracle: mu, var, d(w . mu)/dX, d(w . var)/dX and d(w . var)/d raw_noise."""
    sd = dict(mod["sd"])
    rn = sd[noise_key(fidelity)] = sd[noise_key(fidelity)].clone().requires_grad_(True)
    Xo = X.clone().requires_grad_(True)
    mu, var = O.predict_for_acquisition(sd, mod["num_layers"], mod["noise_upper"], mod["samples"], Xo, fidelity,
                                        noise_lower=mod["noise_lower"])
    w = weights(X.shape[0])
    gmu, = torch.autograd.grad((w * mu).sum(), Xo, retain_graph=True)
    gvar, gn = torch.autograd.grad((w * var).sum(), [Xo, rn])
    return dict(mu=mu.detach(), var=var.detach(), dx_mu=gmu, dx_var=gvar, dn=gn)


def oracle_jes(mods, X, fidelity):
    """JES's dX and the scale of the two terms whose difference it is: max |d sum 1/2 log v / dX| over the models."""
    Xo = X.clone().requires_grad_(True)
    O.jes_mfdgp(mods[0], mods[1], Xo, fidelity).sum().backward()
    scale = 0.0
    for mod in mods:
        Xt = X.clone().requires_grad_(True)
        _, v = O.predict_for_acquisition(mod["sd"], mod["num_layers"], mod["noise_upper"], mod["samples"], Xt,
                                         fidelity, noise_lower=mod["noise_lower"])
        g, = torch.autograd.grad((0.5 * torch.log(v)).sum(), Xt)
        scale = max(scale, float(g.abs().max()))
    return Xo.grad, scale


def cuda_chain(model, cond, X, fidelity, S):
    """Everything the fused chain computes for the comparisons, with the dispatch it claims asserted."""
    with torch.no_grad():
        (mu, var), names = kernels_run(lambda: model.predict_for_acquisition(X.to(DEV), fidelity))
    ws = S >= XSHARE_MIN_REP and fidelity >= 1
    assert ("row_fwd_ws_kernel" in names) == ws, (S, fidelity, sorted(names))
    (gx_mu, gn_mu), names = kernels_run(lambda: cuda_grads(model, cond, X, fidelity, "mu"))
    assert "acq_moment_bwd_kernel" in names and ("row_fwd_ws_kernel" in names) == ws, sorted(names)
    gx_var, gn_var = cuda_grads(model, cond, X, fidelity, "var")
    gx_jes, _ = cuda_grads(model, cond, X, fidelity, "jes")
    assert float(gn_mu.abs().max()) == 0.0                     # the mean does not depend on the likelihood's noise
    return dict(mu=mu.cpu(), var=var.cpu(), dx_mu=gx_mu, dx_var=gx_var, dn=gn_var, dx_jes=gx_jes)


# ---- 2. the acquisition chain against the fp64 oracle ----------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", ACQ_CASES, ids=case_id)
def test_acquisition_chain_matches_oracle(case):
    d, M, ls, L, S, n = case
    model, cond = models(d, M, ls, L, S)
    tol, kzz = parity_tol(model)
    tol_c, kzz_c = parity_tol(cond)
    assert max(kzz, kzz_c) <= COND_MAX, (case, kzz, kzz_c)
    tol = max(tol, tol_c)
    X = candidates(n, d, seed=d + S)
    mods = (oracle_module(model), oracle_module(cond))
    for fidelity in range(L):
        c = cuda_chain(model, cond, X, fidelity, S)
        o = oracle_chain(mods[0], X, fidelity)
        jes_o, term = oracle_jes(mods, X, fidelity)
        # no comparison is vacuous
        for k in ("dx_mu", "dx_var", "dn"):
            assert float(o[k].abs().max()) > 1e-3, (case, fidelity, k)
        assert float(jes_o.abs().max()) > 1e-3, (case, fidelity)
        assert relerr(c["dx_mu"], c["dx_var"]) > 1e-2, (case, fidelity)
        err = {k: relerr(c[k], o[k]) for k in ("mu", "var", "dx_mu", "dx_var", "dn")}
        err["dx_jes"] = float((c["dx_jes"] - jes_o).abs().max()) / max(float(jes_o.abs().max()), term)
        print("%s fidelity %d cond %.1e tol %.1e | mu %.1e var %.1e dX(d_mu) %.1e dX(d_var) %.1e dX(jes) %.1e "
              "d raw_noise %.1e" % (case_id(case), fidelity, max(kzz, kzz_c), tol, err["mu"], err["var"],
                                    err["dx_mu"], err["dx_var"], err["dx_jes"], err["dn"]))
        bars = dict(mu=tol, var=10 * tol, dx_mu=tol, dx_var=tol, dn=tol, dx_jes=tol)
        for k, e in err.items():
            assert e <= bars[k], (case, fidelity, k, e, bars[k])


# ---- 3. layer rows in training and composable mode ----------------------------------------------------------------
def theta_upper(sd, l):
    """Constrained hyper-parameters of an upper layer in the kernels' layout (include/mobocmf_b200.h)."""
    sp = torch.nn.functional.softplus
    c = "hidden_layer_%d.covar_module." % l
    return torch.cat([sp(sd[c + "kernels.0.kernels.0.raw_outputscale"]).reshape(1),
                      sp(sd[c + "kernels.0.kernels.1.kernels.0.raw_variance"]).reshape(1),
                      sp(sd[c + "kernels.0.kernels.1.kernels.1.raw_outputscale"]).reshape(1),
                      sp(sd[c + "kernels.0.kernels.1.kernels.1.base_kernel.raw_lengthscale"]).reshape(1),
                      sp(sd[c + "kernels.1.raw_outputscale"]).reshape(1),
                      sp(sd[c + "kernels.0.kernels.0.base_kernel.raw_lengthscale"]).reshape(-1),
                      sp(sd[c + "kernels.1.base_kernel.raw_lengthscale"]).reshape(-1)])


@pytest.mark.gpu
@pytest.mark.parametrize("d,M,ls,S,n", ROWS_CASES, ids=lambda v: str(v))
def test_layer_rows_training_matches_oracle(d, M, ls, S, n):
    """Layer 1's rows f = mu_prev + sqrt(var_prev) eps, S per point, in training mode: the forward of the S class
    (generic with SHX warps, or row_fwd_ws_kernel) and kgrad_kernel with and without the x gradient, against the
    oracle's layer_q on the explicitly tiled rows."""
    from mobocmf_b200 import functional as F
    l = 1
    sd, _ = random_state(M, d, L3, seed=seed_of(d, L3), ls=ls)
    Z = O.layer_inducing_points(sd, l)
    kzz = float(torch.linalg.cond(O.layer_kernel(sd, l, Z, Z) + O.JITTER * torch.eye(M, dtype=torch.float64)))
    assert kzz <= COND_MAX, kzz
    tol = max(1e-10, 20 * EPS64 * kzz)
    g = torch.Generator().manual_seed(17 * d + S)
    x = torch.rand(n, d, generator=g, dtype=torch.float64)
    mu0 = torch.randn(n, generator=g, dtype=torch.float64)
    var0 = 0.05 + torch.rand(n, generator=g, dtype=torch.float64)
    eps = torch.randn(n * S, generator=g, dtype=torch.float64)
    wmu, wvar = torch.randn(n * S, generator=g, dtype=torch.float64), torch.randn(n * S, generator=g, dtype=torch.float64)
    q = "hidden_layer_%d.variational_strategy._variational_distribution."
    keys = [k for k in sd if k.startswith("hidden_layer_1.covar_module.")] + \
        [(q % 0) + "variational_mean", (q % 1) + "variational_mean", (q % 1) + "chol_variational_covar"]

    def tril_if_chol(k, v):
        return torch.tril(v) if "chol_variational_covar" in k else v

    # oracle: the tiled rows through layer_q (training branch)
    sdo = {k: (v.clone().requires_grad_(True) if k in keys else v) for k, v in sd.items()}
    xo, mo, vo = (t.clone().requires_grad_(True) for t in (x, mu0, var0))
    f = mo.repeat_interleave(S) + torch.sqrt(vo.clamp_min(O.MIN_VARIANCE)).repeat_interleave(S) * eps
    mu_o, var_o = O.layer_q(sdo, l, torch.cat([xo.repeat_interleave(S, 0), f[:, None]], 1), training=True)
    grads_o = torch.autograd.grad((wmu * mu_o).sum() + (wvar * var_o).sum(), [xo, mo, vo] + [sdo[k] for k in keys])

    Zx = sd["hidden_layer_0.variational_strategy.inducing_points"].to(DEV).contiguous()
    fwd = "row_fwd_ws_kernel" if S >= XSHARE_MIN_REP else "row_fwd_kernel"
    for want_x in (True, False):
        sdc = {k: sd[k].to(DEV).requires_grad_(True) for k in keys}
        xc = x.to(DEV).requires_grad_(want_x)
        mc, vc = (t.to(DEV).requires_grad_(True) for t in (mu0, var0))

        def run():
            theta = theta_upper(sdc, l)
            ops = F.layer_operators(theta, sdc[(q % 0) + "variational_mean"], sdc[(q % 1) + "variational_mean"],
                                    sdc[(q % 1) + "chol_variational_covar"], Zx, 1)
            mu, var = F.layer_rows(ops, theta, sdc[(q % 0) + "variational_mean"], Zx, xc, mu_prev=mc, var_prev=vc,
                                   eps=eps.to(DEV), kind=1, xrep=S, prep=S, eps_mod=n * S, R=n * S, training=True)
            loss = (wmu.to(DEV) * mu).sum() + (wvar.to(DEV) * var).sum()
            leaves = ([xc] if want_x else []) + [mc, vc] + [sdc[k] for k in keys]
            return mu.detach(), var.detach(), torch.autograd.grad(loss, leaves)
        (mu, var, grads), names = kernels_run(run)
        assert fwd in names and ("row_fwd_ws_kernel" in names) == (S >= XSHARE_MIN_REP), sorted(names)
        assert ("kgrad_kernel<param,x>" if want_x else "kgrad_kernel<param>") in names, sorted(names)
        em, ev = relerr(mu, mu_o), relerr(var, var_o)
        assert em <= tol and ev <= tol, (want_x, em, ev, tol)
        names_g = (["x"] if want_x else []) + ["mu_prev", "var_prev"] + keys
        ref = list(grads_o) if want_x else list(grads_o[1:])
        worst = 0.0
        for name, gc, go in zip(names_g, grads, ref):
            assert float(go.abs().max()) > 0.0, name
            e = relerr(tril_if_chol(name, gc), tril_if_chol(name, go))
            worst = max(worst, e)
            assert e <= 100 * tol, (want_x, name, e, tol)
        print("rows d%d M%d S%d n%d x-grad %s cond %.1e | mean %.1e var %.1e worst gradient %.1e (bar %.1e)"
              % (d, M, S, n, want_x, kzz, em, ev, worst, 100 * tol))


# ---- 4. one ill-conditioned case, judged by the longdouble truth ---------------------------------------------------
def truth_chain(mod, X, fidelity):
    """The truth's mu, var, d(w . mu)/dX, d(w . var)/dX and d(w . var)/d raw_noise (numpy longdouble)."""
    from oracle import ld_autodiff as A
    from oracle import mfdgp_truth as T
    sd = T.leaves(mod["sd"], {noise_key(fidelity)})
    Xn = A.leaf(X.reshape(X.shape[0], -1))
    mu, var = T.predict_for_acquisition(sd, mod["num_layers"], mod["noise_upper"], mod["samples"], Xn, fidelity,
                                        noise_lower=mod["noise_lower"])
    w = weights(X.shape[0]).numpy().astype(A.LD)
    A.backward(A.sum_(mu * w))
    dx_mu = Xn.g.copy()
    A.backward(A.sum_(var * w))
    return dict(mu=mu.v, var=var.v, dx_mu=dx_mu, dx_var=Xn.g.copy(), dn=sd[noise_key(fidelity)].g.copy())


def truth_jes(mods, X, fidelity):
    from oracle import mfdgp_truth as T
    return T.jes_truth(mods[0], mods[1], X, fidelity)[1]


@pytest.mark.gpu
def test_ill_conditioned_chain_against_truth():
    """d = 1 at a median-heuristic-sized lengthscale (cond 1e7 - 1e8, the Forrester example's regime): there two
    correct fp64 programs differ by ~cond * eps, so the CUDA path must be as close to the longdouble truth as the fp64
    oracle is, or within the effect of rounding the covariance entries (helpers.adjudicate)."""
    from oracle import mfdgp_truth as T
    d, M, ls, L, S, n = 1, 20, 0.3, L3, 25, 12
    model, cond = models(d, M, ls, L, S)
    kzz = state_cond(oracle_view(model)[0], L)
    assert kzz >= 1e6, kzz
    X = candidates(n, d, seed=99)
    mods = (oracle_module(model), oracle_module(cond))
    for fidelity in range(L):
        c = cuda_chain(model, cond, X, fidelity, S)
        o = oracle_chain(mods[0], X, fidelity)
        Xo = X.clone().requires_grad_(True)
        O.jes_mfdgp(mods[0], mods[1], Xo, fidelity).sum().backward()
        o["dx_jes"] = Xo.grad
        t = truth_chain(mods[0], X, fidelity)
        t["dx_jes"] = truth_jes(mods, X, fidelity).reshape(X.shape)
        sens = {k: 0.0 for k in t}
        for k in range(4):
            with T.covariance_rounding(2000 + k):
                p = truth_chain(mods[0], X, fidelity)
                p["dx_jes"] = truth_jes(mods, X, fidelity).reshape(X.shape)
            for q in t:
                den = np.max(np.abs(t[q]))
                sens[q] = max(sens[q], float(np.max(np.abs(p[q] - t[q])) / den))
        rep = []
        for q in ("mu", "var", "dx_mu", "dx_var", "dx_jes", "dn"):
            assert q in ("mu", "var") or float(np.max(np.abs(t[q]))) > 1e-3, (fidelity, q)
            adjudicate("fidelity %d %s" % (fidelity, q), c[q], o[q], t[q], sens[q], report=rep)
        print("ill-conditioned d1 M20 S25 fidelity %d cond %.1e | " % (fidelity, kzz) +
              " ".join("%s cuda %.1e oracle %.1e sens %.1e" % r for r in rep))


# ---- 5. forward chunking ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("S", [7, 25])
def test_chunked_forward_is_bit_identical(S, monkeypatch):
    """MFDGP.ACQ_CHUNK candidates per mobo_acq_moments enqueue: every row's arithmetic is independent of its tile and of
    whether its warp shares x, so the chunked moments equal one unchunked call bit for bit."""
    from mobocmf_b200.models.mfdgp import MFDGP
    d, M, ls = 5, 200, 0.3
    model, _ = models(d, M, ls, L3, S)
    X = candidates(3 * 64 + 5, d, seed=S).to(DEV)
    with torch.no_grad():
        ref = [model.predict_for_acquisition(X, f) for f in range(L3)]
        for chunk in (64, 7):
            monkeypatch.setattr(MFDGP, "ACQ_CHUNK", chunk)
            for f in range(L3):
                mu, var = model.predict_for_acquisition(X, f)
                assert torch.equal(mu, ref[f][0]) and torch.equal(var, ref[f][1]), (chunk, f)
