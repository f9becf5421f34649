"""d acquisition / dX through the fused acquisition chain (mobo_acq_moments_bwd, functional.acq_moments): parity with
the composable autograd path and the oracle, the C ABI's contract (accumulate, determinism, shape errors before any
launch), chunking, bounded memory and routing.  The GPU tests are marked one by one; the layout test runs on the CPU."""
import copy

import pytest
import torch

from mobocmf_b200 import _lib
from tests.helpers import oracle_view, parity_tol, relerr, synthetic_data

DEV = "cuda:0"
_MODELS = {}


def make_model(M, d, S, L=3, only_hf=False, seed=0):
    """An L-fidelity MFDGP with M shared inducing inputs and S acquisition samples, moved away from its initial point
    so that every term of the chain matters; cached per shape."""
    key = (M, d, S, L, only_hf, seed)
    if key not in _MODELS:
        from mobocmf_b200.models.mfdgp import MFDGP
        sizes = [M + 40, 80, 40][:L]
        x, y, fid = synthetic_data(sizes, d, seed=seed)
        torch.manual_seed(seed)
        model = MFDGP(x, y, fid, L, num_samples_for_acquisition=S, num_inducing=M, init_lengthscale=0.3,
                      use_only_highest_fidelity=only_hf)
        model.double()
        g = torch.Generator().manual_seed(seed + 11)
        with torch.no_grad():
            for n, p in model.named_parameters():
                if "chol_variational_covar" in n:
                    p.add_(torch.tril(torch.randn(p.shape, generator=g, dtype=p.dtype)) * 0.02 / p.shape[0] ** 0.5)
                    p.diagonal().abs_().add_(0.05)
                else:
                    p.add_(0.1 * torch.randn(p.shape, generator=g, dtype=p.dtype))
        _MODELS[key] = model.to(DEV)
    return _MODELS[key]


def cond_copy(model, seed=9):
    """A conditioned copy: same eval samples (quirk Q7), shifted means, a more certain q(u)."""
    c = copy.deepcopy(model)
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n, p in c.named_parameters():
            if "variational_mean" in n:
                p.add_(0.05 * torch.randn(p.shape, generator=g, dtype=p.dtype).to(DEV))
            if "chol_variational_covar" in n:
                p.mul_(0.6)
    return c


def raw_noise(model, fidelity):
    return getattr(model, "hidden_layer_likelihood_%d" % fidelity).noise_covar.raw_noise


def candidates(n, d, seed=3):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(n, 1, d, generator=g, dtype=torch.float64).to(DEV)


def grads(model, cond, X, fidelity, upstream):
    """(dX, d raw_noise of `model`) of one scalar built from the acquisition moments."""
    from mobocmf_b200.acquisition_functions.JESMOC_MFDGP import _JES_MFDGP
    Xg = X.clone().requires_grad_(True)
    n = X.shape[0]
    w = torch.linspace(-1.0, 2.0, n, dtype=torch.float64, device=DEV)
    if upstream == "jes":
        loss = _JES_MFDGP(fidelity, model, cond)(Xg).sum()
    else:
        model.eval()
        mu, var = model.predict_for_acquisition(Xg, fidelity)
        model.train()
        loss = {"mu": lambda: (w * mu).sum(), "var": lambda: (w * var).sum(),
                "both": lambda: (w * mu).sum() + (w.flip(0) * var).sum()}[upstream]()
    rn = raw_noise(model, fidelity)
    gx, gn = torch.autograd.grad(loss, [Xg, rn], allow_unused=True)
    return gx, (torch.zeros_like(rn) if gn is None else gn)


def kzz_condition(model, fidelity):
    """Largest condition number of K(Z, Z) + jitter I over the layers 0 .. fidelity (from the eval operator buffers)."""
    from mobocmf_b200.functional import ops_layout
    worst = 1.0
    for i in range(fidelity + 1):
        lay = getattr(model, "hidden_layer_%d" % i)
        ops = lay.operators()[0].detach()
        M = lay.num_inducing
        lo = ops_layout(M)
        P = ops[lo["P"]:lo["P"] + lo["MP"] ** 2].view(lo["MP"], lo["MP"])[:M, :M].cpu()
        worst = max(worst, float(torch.linalg.cond(P)))
    return worst


def term_scale(models, X, fidelity):
    """max |d sum 1/2 log v / dX| over the models: the size of the two terms whose difference is JES's dX."""
    out = 0.0
    for m in models:
        Xg = X.clone().requires_grad_(True)
        m.eval()
        _, var = m.predict_for_acquisition(Xg, fidelity)
        m.train()
        gx, = torch.autograd.grad((0.5 * torch.log(var)).sum(), Xg)
        out = max(out, float(gx.abs().max()))
    return out


def composable(monkeypatch):
    from mobocmf_b200.models.mfdgp import MFDGP
    monkeypatch.setattr(MFDGP, "_fused_acquisition_applies", lambda self, x: False)


def kernels_run(fn):
    """fn's result and the names of the library's kernels it launched."""
    _lib.profile_enable(True)
    try:
        out = fn()
        return out, {name for name, _ in _lib.profile_collect()}
    finally:
        _lib.profile_enable(False)


# ---- 1. against the composable autograd path ------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("M", [48, 256])
@pytest.mark.parametrize("d", [1, 6])
@pytest.mark.parametrize("S", [1, 7, 25])
def test_fused_dX_matches_composable_path(M, d, S, monkeypatch):
    model = make_model(M, d, S)
    cond = cond_copy(model)
    X = candidates(45, d)
    for fidelity in range(3):
        for upstream in ("mu", "var", "both", "jes"):
            (gx, gn), names = kernels_run(lambda: grads(model, cond, X, fidelity, upstream))
            assert "acq_moment_bwd_kernel" in names
            with monkeypatch.context() as mp:
                composable(mp)
                gx_r, gn_r = grads(model, cond, X, fidelity, upstream)
            # The two paths feed the same row kernels with d mu, d var that differ in the last bits (the composable
            # path's torch glue sums S equal shares and subtracts 2 mu g - 2 mean g, the fused kernel uses the closed
            # form).  The row backward goes through W = L^-1 twice, so such differences grow with cond(K_zz), which the
            # random inducing inputs of the d = 1 and M = 256 models make large.  Bar: 1e-12, or the
            # unit round-off times cond(K_zz) with a factor 10 when that is larger.  JES's dX is the difference of
            # two models' terms, which can cancel: it is measured against the larger term.
            models = (model, cond) if upstream == "jes" else (model,)
            bar = max(1e-12, 1e-15 * max(kzz_condition(m, fidelity) for m in models))
            scale = float(gx_r.abs().max())
            assert scale > 0.0, (fidelity, upstream)
            if upstream == "jes":
                scale = max(scale, term_scale(models, X, fidelity))
            err = float((gx - gx_r).abs().max())
            assert err <= bar * scale, (fidelity, upstream, err, scale, bar)
            nerr = float((gn - gn_r).abs().max())
            assert nerr <= bar * max(float(gn_r.abs().max()), 1e-300) or nerr == 0.0, (fidelity, upstream, nerr,
                                                                                         float(gn_r.abs().max()), bar)


# ---- 2. against the oracle --------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_fused_jes_dX_matches_oracle():
    from mobocmf_b200.acquisition_functions.JESMOC_MFDGP import _JES_MFDGP
    from oracle import mfdgp_oracle as O
    L = 3
    model = make_model(256, 6, 25, L=L)
    cond = cond_copy(model)
    X = candidates(16, 6, seed=5)
    tol = max(parity_tol(model)[0], parity_tol(cond)[0])
    for fidelity in range(L):
        Xc = X.clone().requires_grad_(True)
        _, names = kernels_run(lambda: _JES_MFDGP(fidelity, model, cond)(Xc).sum().backward())
        assert "acq_moment_bwd_kernel" in names
        Xo = X.cpu().clone().requires_grad_(True)
        mods = []
        for m in (model, cond):
            sd, lo, up, samples = oracle_view(m)
            mods.append(dict(sd=sd, num_layers=L, noise_upper=up, noise_lower=lo, samples=samples))
        O.jes_mfdgp(mods[0], mods[1], Xo, fidelity).sum().backward()
        assert float(Xc.grad.abs().max()) > 1e-3
        assert relerr(Xc.grad, Xo.grad) < 1e3 * tol, (fidelity, relerr(Xc.grad, Xo.grad), tol)


# ---- 3. the C ABI through ctypes ----------------------------------------------------------------------------------
def captured_chain(model, X, fidelity, monkeypatch):
    """The AcqChain the model hands to functional.acq_moments."""
    from mobocmf_b200 import functional as F
    seen = {}
    orig = F.acq_moments

    def spy(chain, x, rn, chunk, grad_chunk):
        seen["chain"], seen["rn"] = chain, rn
        return orig(chain, x, rn, chunk, grad_chunk)
    monkeypatch.setattr(F, "acq_moments", spy)
    model.eval()
    with torch.no_grad():
        model.predict_for_acquisition(X, fidelity)
    model.train()
    return seen["chain"], seen["rn"]


def call_bwd(c, n, d, rn, X, d_mu, d_var, accumulate, dX, dn, work, fidelity=None, M=None, S=None):
    lib = _lib.load()
    return lib.mobo_acq_moments_bwd(
        c.fidelity if fidelity is None else fidelity, d, c.M if M is None else M, c.S if S is None else S, n,
        _lib.ptr(c.Zx), _lib.ptr_array(c.zf), _lib.ptr_array(c.theta), _lib.ptr_array(c.ops),
        _lib.ptr_array(c.samples), _lib.ptr(rn), c.noise_lower, c.noise_upper, _lib.ptr(X), _lib.ptr(d_mu),
        _lib.ptr(d_var), accumulate, _lib.ptr(dX), _lib.ptr(dn), _lib.ptr(work), _lib.stream_ptr())


@pytest.mark.gpu
def test_abi_accumulate_determinism_and_shape_errors(monkeypatch):
    lib = _lib.load()
    M, d, S, fidelity, n = 48, 6, 7, 2, 77
    model = make_model(M, d, S)
    X = candidates(n, d)[:, 0, :].contiguous()
    c, rn = captured_chain(model, X, fidelity, monkeypatch)
    g = torch.Generator().manual_seed(2)
    d_mu = torch.randn(n, generator=g, dtype=torch.float64).to(DEV)
    d_var = torch.randn(n, generator=g, dtype=torch.float64).to(DEV)
    work = torch.empty(lib.mobo_acq_bwd_work_doubles(fidelity, d, M, S, n), dtype=torch.float64, device=DEV)
    outs = []
    for _ in range(2):
        dX = torch.full((n, d), float("nan"), dtype=torch.float64, device=DEV)
        dn = torch.full((1,), float("nan"), dtype=torch.float64, device=DEV)
        assert call_bwd(c, n, d, rn, X, d_mu, d_var, 0, dX, dn, work) == 0
        outs.append((dX, dn))
    torch.cuda.synchronize()
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    assert bool(torch.isfinite(outs[0][0]).all()) and float(outs[0][0].abs().max()) > 0.0
    pre_x = torch.randn(n, d, generator=g, dtype=torch.float64).to(DEV)
    pre_n = torch.randn(1, generator=g, dtype=torch.float64).to(DEV)
    dX, dn = pre_x.clone(), pre_n.clone()
    assert call_bwd(c, n, d, rn, X, d_mu, d_var, 1, dX, dn, work) == 0
    assert torch.equal(dX, pre_x + outs[0][0]) and torch.equal(dn, pre_n + outs[0][1])
    # NULL upstream gradients are zero
    dX0 = torch.empty(n, d, dtype=torch.float64, device=DEV)
    assert call_bwd(c, n, d, rn, X, None, None, 0, dX0, None, work) == 0
    assert float(dX0.abs().max()) == 0.0

    # unsupported shapes: -2 before any launch, with buffers far too small for the shape
    tiny = torch.zeros(16, dtype=torch.float64, device=DEV)
    bad = [dict(fidelity=-1), dict(fidelity=8), dict(n=0), dict(S=0), dict(M=300), dict(d=9),
           dict(n=1 << 27, S=16)]
    before = _lib.launch_count()
    for b in bad:
        kw = dict(fidelity=fidelity, d=d, M=M, S=S, n=n)
        kw.update(b)
        assert lib.mobo_acq_bwd_work_doubles(kw["fidelity"], kw["d"], kw["M"], kw["S"], kw["n"]) == 0, b
        assert call_bwd(c, kw["n"], kw["d"], rn, tiny, tiny, tiny, 0, tiny, tiny, tiny, fidelity=kw["fidelity"],
                        M=kw["M"], S=kw["S"]) == -2, b
    assert _lib.launch_count() == before


# ---- 4. chunking --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("S", [7, 25])
def test_chunked_backward_is_bit_identical(S, monkeypatch):
    from mobocmf_b200.models.mfdgp import MFDGP
    model = make_model(256, 6, S)
    cond = cond_copy(model)
    chunk = 64
    X = candidates(3 * chunk + 5, 6, seed=7)
    gx, gn = grads(model, cond, X, 2, "jes")
    monkeypatch.setattr(MFDGP, "ACQ_GRAD_CHUNK", chunk)
    gx_c, gn_c = grads(model, cond, X, 2, "jes")
    assert torch.equal(gx, gx_c)
    # d raw_noise folds the chunks' partials in another order
    assert float((gn - gn_c).abs().max()) <= 1e-14 * float(gn.abs().max())


# ---- 5. bounded memory ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_jes_sweep_gradient_memory_is_bounded():
    from mobocmf_b200.acquisition_functions.JESMOC_MFDGP import jes_sweep
    model = make_model(256, 6, 25)
    boxes = [(model, [cond_copy(model)])]
    X = torch.rand(20000, 6, generator=torch.Generator().manual_seed(4), dtype=torch.float64).to(DEV)
    ref = jes_sweep(X, 2, boxes)              # also builds and caches the eval-mode operators
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    Xg = X.clone().requires_grad_(True)
    v = jes_sweep(Xg, 2, boxes)
    v.sum().backward()
    torch.cuda.synchronize()
    grown = torch.cuda.max_memory_allocated() - base
    print("peak growth %.3f GiB" % (grown / 2 ** 30))
    assert grown < 2 * 2 ** 30
    assert torch.equal(v.detach(), ref)
    assert bool(torch.isfinite(Xg.grad).all()) and float(Xg.grad.abs().max()) > 0.0


# ---- 6. routing ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_only_shared_z_models_take_the_fused_backward():
    from mobocmf_b200.acquisition_functions.JESMOC_MFDGP import _JES_MFDGP
    X = candidates(20, 2)
    shared = make_model(48, 2, 7)
    _, names = kernels_run(lambda: _JES_MFDGP(2, shared, cond_copy(shared))(X.clone().requires_grad_(True)).sum()
                           .backward())
    assert {"acq_moment_bwd_kernel", "acq_prop_bwd_kernel", "acq_dx_fold_kernel"} <= names
    only_hf = make_model(48, 2, 7, L=2, only_hf=True)     # non-shared Z above layer 1 is unsupported (F3)
    Xg = X.clone().requires_grad_(True)
    _, names = kernels_run(lambda: _JES_MFDGP(1, only_hf, cond_copy(only_hf))(Xg).sum().backward())
    assert "acq_moment_bwd_kernel" not in names and "row_bwd_gemm_kernel" in names
    assert bool(torch.isfinite(Xg.grad).all()) and float(Xg.grad.abs().max()) > 0.0


# ---- 7. work size and layout (CPU) ----------------------------------------------------------------------------------
def documented_layout(fidelity, d, M, S, n):
    """Offsets (doubles) of the work regions in the order include/mobocmf_b200.h documents, and the total."""
    lib = _lib.load()
    off, regions = 0, []

    def take(name, k, rows_mp=False):
        nonlocal off
        regions.append((name, off, rows_mp))
        off += (k + 15) // 16 * 16
    RF = n if fidelity == 0 else n * S
    for l in range(fidelity + 1):
        R = n if l == 0 else n * S
        take("mu%d" % l, R)
        take("var%d" % l, R)
        take("T%d" % l, lib.mobo_rows_save_doubles(M, R), True)
        take("U%d" % l, lib.mobo_rows_save_doubles(M, R), True)
        take("dxrow%d" % l, R * d)
    take("dmu", RF)
    take("dvar", RF)
    take("df", RF)
    take("dk", lib.mobo_rows_save_doubles(M, RF), True)
    take("noise", (n + 255) // 256)
    return regions, off


def test_acq_bwd_work_size_and_layout():
    lib = _lib.load()
    for bad in [(-1, 6, 256, 25, 10), (8, 6, 256, 25, 10), (2, 0, 256, 25, 10), (2, 9, 256, 25, 10),
                (2, 6, 0, 25, 10), (2, 6, 257, 25, 10), (2, 6, 256, 0, 10), (2, 6, 256, 25, 0),
                (2, 6, 256, 16, 1 << 27), (0, 6, 256, 1, (1 << 31) - 32)]:
        assert lib.mobo_acq_bwd_work_doubles(*bad) == 0, bad
    for fidelity, d, M, S in [(0, 1, 48, 1), (1, 6, 48, 7), (2, 6, 256, 25), (2, 3, 75, 25), (7, 8, 256, 3)]:
        prev = first = 0
        for n in (1, 5, 33, 256, 257, 1000, 4096):
            w = lib.mobo_acq_bwd_work_doubles(fidelity, d, M, S, n)
            regions, total = documented_layout(fidelity, d, M, S, n)
            assert w == total, (fidelity, d, M, S, n, w, total)
            assert w >= prev            # rows are rounded up to 32-row tiles: equal for n = 1 and 5 at S = 1
            prev, first = w, first or w
            for name, off, rows_mp in regions:
                assert (off * 8) % 16 == 0, name
                if rows_mp:     # every row of a [R][MP] block starts 16-byte aligned too
                    assert (lib.mobo_padded_m(M) * 8) % 16 == 0
        assert prev > first
    # C5's chunk (MFDGP.ACQ_GRAD_CHUNK = 4096 at M = 256, S = 25, fidelity 2) stays near 1 GiB
    assert lib.mobo_acq_bwd_work_doubles(2, 6, 256, 25, 4096) * 8 < 1.1e9

