"""GPU edge cases of the row / operator kernels against the oracle: ragged row counts (1 row, tile size +- 1), M not a
multiple of 32 and below one block, d from 1 to 8 (the ARD limit), a single-fidelity model, empty candidate batches,
shape limits returning errors instead of wrong numbers."""
import pytest
import torch

from oracle import mfdgp_oracle as O
from tests.helpers import random_state, clone_state, param_keys, relerr, model_from_state

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _cond(sd, L):
    worst = 1.0
    for l in range(L):
        Z = O.layer_inducing_points(sd, l)
        P = O.layer_kernel(sd, l, Z, Z) + 1e-6 * torch.eye(Z.shape[0], dtype=torch.float64)
        worst = max(worst, float(torch.linalg.cond(P)))
    return worst


@pytest.mark.parametrize("M,d,L,B,S", [(5, 1, 2, 1, 1), (33, 8, 2, 31, 1), (32, 3, 1, 33, 1), (17, 2, 3, 65, 2),
                                       (96, 4, 2, 16, 4), (2, 1, 2, 3, 1)])
def test_ragged_shapes_fused_step(M, d, L, B, S):
    from mobocmf_b200.fused import FusedELBOStep
    from mobocmf_b200.mlls.variational_elbo_mf import VariationalELBOMF
    sd, noise_upper = random_state(M, d, L, seed=M + d + B, ls=0.35 if d < 6 else 0.8)
    g = torch.Generator().manual_seed(B)
    x = torch.rand(B, d, generator=g, dtype=torch.float64)
    y = torch.randn(B, 1, generator=g, dtype=torch.float64)
    fid = torch.randint(0, L, (B, 1), generator=g).double()
    eps = [None] + [torch.randn(B * S, generator=g).double() for _ in range(1, L)]
    sdo = clone_state(sd, requires_grad=True)
    loss_o, kl_o = O.elbo_step_loss_tiled(sdo, L, noise_upper, x, y, fid, eps, 5 * B, S)
    loss_o.backward()
    model = model_from_state(sd, noise_upper, L)
    step = FusedELBOStep(model, VariationalELBOMF(model, 5 * B, L))
    loss, kl = step(x.to(DEV), y.to(DEV), fid.to(DEV), eps=[None if e is None else e.to(DEV) for e in eps],
                    num_samples=S)
    step.check()
    cond = _cond(sd, L)
    tol = max(1e-10, 20 * 2.2e-16 * cond)
    assert relerr(loss, loss_o) < tol and relerr(kl, kl_o) < tol, (relerr(loss, loss_o), tol)
    grads = {n: p.grad for n, p in model.named_parameters()}
    if cond >= 1e5:       # ill-conditioned: adjudicated by the longdouble truth (tests/helpers.adjudicate)
        from tests.helpers import adjudicate_state
        keys = param_keys(sd)
        zero = lambda k: torch.zeros_like(sd[k])
        adjudicate_state(sd, O.NOISE_LOWER, noise_upper, loss, {k: grads[k] for k in keys}, loss_o.detach(),
                         {k: (sdo[k].grad if sdo[k].grad is not None else zero(k)) for k in keys}, L, x, y, fid, eps,
                         5 * B, S)
        return
    for k in param_keys(sd):
        gp, go = grads[k], sdo[k].grad
        if "chol_variational_covar" in k:
            gp, go = torch.tril(gp), torch.tril(go)
        if go is None or float(go.abs().max()) == 0.0:     # parameter not reached by this minibatch (e.g. one fidelity only)
            assert float(gp.abs().max()) < 1e-12, k
            continue
        assert relerr(gp.reshape(-1), go.reshape(-1)) < 1e3 * tol, (k, relerr(gp.reshape(-1), go.reshape(-1)))


@pytest.mark.parametrize("n", [1, 31, 32, 33, 257])
def test_acquisition_ragged_candidate_counts(n):
    M, d, L = 20, 2, 3
    sd, noise_upper = random_state(M, d, L, seed=3, ls=0.4)
    g = torch.Generator().manual_seed(n)
    samples = [torch.randn(25, 1, generator=g) for _ in range(L)]
    model = model_from_state(sd, noise_upper, L, samples=samples)
    model.eval()
    X = torch.rand(n, 1, d, generator=g, dtype=torch.float64)
    tol = max(1e-10, 20 * 2.2e-16 * _cond(sd, L))
    for f in range(L):
        with torch.no_grad():
            mu, var = model.predict_for_acquisition(X.to(DEV), f)
        model.eval()
        mu_o, var_o = O.predict_for_acquisition(sd, L, noise_upper, samples, X, f)
        assert mu.shape == (n,) and relerr(mu, mu_o) < tol and relerr(var, var_o) < 10 * tol


def test_shape_limits_are_errors_not_wrong_numbers():
    from mobocmf_b200 import _lib
    lib = _lib.load()
    t = torch.zeros(16, dtype=torch.float64, device=DEV)
    p = _lib.ptr(t)
    # M > 256 and d > 8 are outside the kernels' limits
    rc = lib.mobo_layer_precompute(0, 2, 300, p, None, p, p, p, 1e-6, p, _lib.stream_ptr())
    assert rc == -2
    rc = lib.mobo_layer_precompute_bwd(0, 2, 300, p, None, p, p, p, p, p, p, p, None, p, p, _lib.stream_ptr())
    assert rc == -2
    rc = lib.mobo_layer_rows_fwd(0, 9, 16, p, None, p, p, p, 1, None, None, 1, None, 1, None, 4, 1, p, p, None, None,
                                 None, None, _lib.stream_ptr())
    assert rc == -2
    # zero rows: nothing is launched, success
    rc = lib.mobo_layer_rows_fwd(0, 2, 16, p, None, p, p, p, 1, None, None, 1, None, 1, None, 0, 1, p, p, None, None,
                                 None, None, _lib.stream_ptr())
    assert rc == 0
    torch.cuda.synchronize()


def test_cpu_tensors_are_refused():
    from mobocmf_b200 import functional as F
    sd, _ = random_state(8, 2, 1, seed=1)
    Zx = sd["hidden_layer_0.variational_strategy.inducing_points"]
    with pytest.raises(RuntimeError):
        F.layer_operators(torch.ones(3, dtype=torch.float64), None, torch.zeros(8, dtype=torch.float64),
                          torch.eye(8, dtype=torch.float64), Zx, 0)


def test_not_positive_definite_is_reported():
    """Upstream raises NotPSDError from psd_safe_cholesky; the fused step reports it through its status word."""
    from mobocmf_b200.fused import FusedELBOStep
    from mobocmf_b200.mlls.variational_elbo_mf import VariationalELBOMF
    M, d, L, B = 24, 2, 2, 8
    sd, noise_upper = random_state(M, d, L, seed=2, ls=0.4)
    Zk = "hidden_layer_0.variational_strategy.inducing_points"
    sd[Zk][1] = sd[Zk][0]                      # duplicated inducing input ...
    sd["hidden_layer_1.variational_strategy.inducing_points"][:, :d] = sd[Zk]
    model = model_from_state(sd, noise_upper, L)
    for l in range(L):
        getattr(model, "hidden_layer_%d" % l).variational_strategy.jitter_val = -1e-3   # ... and a negative jitter
    step = FusedELBOStep(model, VariationalELBOMF(model, 40, L))
    g = torch.Generator().manual_seed(0)
    x = torch.rand(B, d, generator=g, dtype=torch.float64).to(DEV)
    step(x, torch.zeros(B, 1, dtype=torch.float64, device=DEV), torch.zeros(B, 1, dtype=torch.float64, device=DEV))
    with pytest.raises(RuntimeError, match="NotPSDError|NanError"):
        step.check()


@pytest.mark.parametrize("jitter,retries", [(1e-6, 0), (-5e-9, 1), (-5e-8, 2), (-5e-7, 3)])
def test_psd_safe_cholesky_retries_on_device(jitter, retries):
    """Upstream factors K(Z, Z) + jitter I with psd_safe_cholesky: on a non-positive pivot it retries with 1e-8, 1e-7,
    1e-6 more on the diagonal (SURVEY.md quirk Q5).  The operator-chain kernel does the same inside the launch.
    A duplicated inducing input gives K an exactly-zero eigenvalue, so P's smallest eigenvalue IS the jitter: a barely
    negative one needs exactly 1, 2 or 3 retries.  The factor, the KL and the predictive moments then equal the
    oracle's, which calls its restatement of psd_safe_cholesky on the same matrix."""
    from mobocmf_b200 import functional as F
    M, d = 40, 2
    sd, noise_upper = random_state(M, d, 1, seed=6, ls=0.4)
    Zk = "hidden_layer_0.variational_strategy.inducing_points"
    sd[Zk][7] = sd[Zk][3]
    Z = sd[Zk]
    P = O.layer_kernel(sd, 0, Z, Z) + jitter * torch.eye(M, dtype=torch.float64)
    L_o = O.psd_safe_cholesky(P)
    if retries:
        assert bool(torch.linalg.cholesky_ex(P)[1] != 0)                       # the first attempt does fail
    h = O.layer_hypers(sd, 0)
    theta = torch.cat([h["a"].reshape(1), h["ls"].reshape(-1)]).to(DEV)
    m, Lq = O.variational_q(sd, 0)
    ops = F.layer_operators(theta, None, m.to(DEV), sd["hidden_layer_0.variational_strategy._variational_distribution."
                                                       "chol_variational_covar"].to(DEV), Z.to(DEV), 0, jitter)
    lay = F.ops_layout(M)
    MP = lay["MP"]
    scal = ops[lay["scal"]:lay["scal"] + 16].cpu()
    assert scal[F.SC_STATUS] == 0.0 and int(scal[7]) == retries, scal
    L_c = ops[lay["L"]:lay["L"] + MP * MP].reshape(MP, MP)[:M, :M].cpu()
    # the smallest eigenvalue is ~5e-8 .. 5e-7 after the rescue: cond ~ 1e9, so the factor agrees to ~cond * eps
    assert relerr(L_c, L_o) < 1e-6, relerr(L_c, L_o)
    kl_o = O.kl_layer(sd, 0, jitter)
    assert abs(float(scal[F.SC_KL]) - float(kl_o)) < 1e-6 * abs(float(kl_o))
    F.check_status()                                                           # nothing sticky was recorded


def test_psd_failure_after_all_retries_is_sticky_in_the_composable_path():
    from mobocmf_b200 import functional as F
    from mobocmf_b200.errors import NotPSDError
    M, d = 16, 2
    sd, _ = random_state(M, d, 1, seed=6, ls=0.4)
    Z = sd["hidden_layer_0.variational_strategy.inducing_points"]
    Z[5] = Z[2]
    h = O.layer_hypers(sd, 0)
    theta = torch.cat([h["a"].reshape(1), h["ls"].reshape(-1)]).to(DEV)
    m, Lq = O.variational_q(sd, 0)
    F.check_status()
    ops = F.layer_operators(theta, None, m.to(DEV), Lq.to(DEV), Z.to(DEV), 0, -1e-3)
    lay = F.ops_layout(M)
    assert float(ops[lay["scal"] + F.SC_STATUS]) == 1.0 and int(ops[lay["scal"] + 7]) == 3
    with pytest.raises(NotPSDError):
        F.check_status()
    F.check_status()          # cleared by the raise
