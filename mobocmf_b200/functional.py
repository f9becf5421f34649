"""torch.autograd wrappers over the C-ABI kernels: one Function for the per-step M x M operator chain of a layer
(``layer_operators``) and one for the fused row pass (``layer_rows``).  They compose under torch autograd, so the
ELBO step, the conditioned step and the acquisition of the models the fused chain does not serve all run through the
same kernels.  ``acq_moments`` is the fused acquisition chain of one model, whose backward (d / dX for
``optimize_acqf``) is one C-ABI call per chunk of candidates.

Reference code replaced: UnwhitenedVariationalStrategy.forward / kl_mvn_mvn [upstream gpytorch] as reached from
``mobocmf/layers/mfdgp_hidden_layer.py:232-286,542-559`` and ``mobocmf/mlls/variational_elbo_mf.py:40``.
"""
import torch

from . import _lib

JITTER = 1e-6          # gpytorch settings.variational_cholesky_jitter (fp64), SURVEY.md quirk Q5
MIN_VARIANCE = 1e-10   # gpytorch settings.min_variance (fp64), quirk Q9
SC_KL = 0
SC_STATUS = 5


def padded_m(M):
    return ((M + 31) // 32) * 32


def ops_layout(M):
    """Offsets (in doubles) inside an operator buffer; mirrors csrc/common.cuh."""
    MP = padded_m(M)
    MP2 = MP * MP
    return {"MP": MP, "L": 0, "W": MP2, "WT": 2 * MP2, "H": 3 * MP2, "HT": 4 * MP2, "P": 5 * MP2, "LQ": 6 * MP2,
            "WF": 7 * MP2, "HTF": 8 * MP2, "HF": 9 * MP2, "WTF": 10 * MP2,
            "beta": 11 * MP2, "alpha": 11 * MP2 + MP, "scal": 11 * MP2 + 2 * MP, "rowstat": 11 * MP2 + 2 * MP + 16,
            "flags": 11 * MP2 + 6 * MP + 16, "size": 11 * MP2 + 6 * MP + 16 + 128}


def _c(t):
    return None if t is None else t.detach().contiguous()


# ---- Cholesky status of the composable path -------------------------------------------------------------------
# The operator-chain kernel retries a failed factorisation like upstream's psd_safe_cholesky (+1e-8, +1e-7, +1e-6) and
# records a final failure in the operator buffer.  Reading it would cost a device synchronisation per layer and step,
# so every precompute ADDS its status into one sticky device counter per GPU (an asynchronous 1-element add, also
# capturable in a CUDA graph) and the callers that already synchronise - the fitter at its reporting boundaries, the
# acquisition optimiser when it returns - call ``check_status()``.
_STICKY = {}


def _record_status(ops, M):
    dev = ops.device.index
    sticky = _STICKY.get(dev)
    if sticky is None:
        sticky = _STICKY[dev] = torch.zeros(1, dtype=torch.float64, device=ops.device)
    i = ops_layout(M)["scal"] + SC_STATUS
    sticky.add_(ops.detach()[i:i + 1])


def check_status(device=None):
    """Raises ``NotPSDError`` if any operator chain since the last call failed on this device (synchronises)."""
    from .errors import NotPSDError
    for dev, sticky in list(_STICKY.items()):
        if device is not None and torch.device(device).index not in (None, dev):
            continue
        if float(sticky) != 0.0:
            sticky.zero_()
            raise NotPSDError("NotPSDError: K(Z, Z) + jitter I is not positive definite (after the 1e-8, 1e-7, 1e-6 "
                              "jitter retries)")


class _LayerOperators(torch.autograd.Function):
    @staticmethod
    def forward(ctx, theta, zf, m, Lq, Zx, kind, jitter):
        lib = _lib.load()
        M, d = Zx.shape
        theta_, zf_, m_, Lq_, Zx_ = _c(theta), _c(zf), _c(m), _c(Lq), _c(Zx)
        ops = torch.zeros(lib.mobo_ops_doubles(M), dtype=torch.float64, device=Zx.device)
        _lib.check(lib.mobo_layer_precompute(kind, d, M, _lib.ptr(Zx_), _lib.ptr(zf_), _lib.ptr(theta_),
                                             _lib.ptr(m_), _lib.ptr(Lq_), float(jitter), _lib.ptr(ops),
                                             _lib.stream_ptr()), "mobo_layer_precompute")
        _record_status(ops, M)
        ctx.save_for_backward(theta_, zf_, m_, Lq_, Zx_, ops)
        ctx.kind = kind
        return ops

    @staticmethod
    def backward(ctx, gops):
        lib = _lib.load()
        theta, zf, m, Lq, Zx, ops = ctx.saved_tensors
        M, d = Zx.shape
        gops = gops.contiguous()
        dev = Zx.device
        work = torch.empty(lib.mobo_precompute_bwd_work_doubles(M), dtype=torch.float64, device=dev)
        dtheta = torch.zeros_like(theta)
        dzf = torch.zeros(M, dtype=torch.float64, device=dev) if ctx.kind == 1 else None
        dm = torch.zeros_like(m)
        dLq = torch.zeros_like(Lq)
        _lib.check(lib.mobo_layer_precompute_bwd(ctx.kind, d, M, _lib.ptr(Zx), _lib.ptr(zf), _lib.ptr(theta),
                                                 _lib.ptr(m), _lib.ptr(Lq), _lib.ptr(ops), _lib.ptr(gops),
                                                 _lib.ptr(work), _lib.ptr(dtheta), _lib.ptr(dzf), _lib.ptr(dm),
                                                 _lib.ptr(dLq), _lib.stream_ptr()), "mobo_layer_precompute_bwd")
        return dtheta, dzf, dm, dLq, None, None, None


def layer_operators(theta, zf, m, Lq, Zx, kind, jitter=JITTER):
    """Operator buffer [L | W | WT | H | HT | P | LQ | beta | alpha | scal] of one layer (differentiable)."""
    return _LayerOperators.apply(theta, zf, m, Lq, Zx, kind, jitter)


def ops_kl(ops, M):
    """KL(q(u) || p(u)) of the layer, read from the operator buffer (differentiable)."""
    return ops[ops_layout(M)["scal"] + SC_KL]


class _LayerRows(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ops, theta, zf, Zx, x, mu_prev, var_prev, eps, f_direct, kind, xrep, prep, eps_mod, R,
                training):
        lib = _lib.load()
        M, d = Zx.shape
        dev = Zx.device
        ops_, theta_, zf_, Zx_, x_ = _c(ops), _c(theta), _c(zf), _c(Zx), _c(x)
        mu_prev_, var_prev_, eps_, f_direct_ = _c(mu_prev), _c(var_prev), _c(eps), _c(f_direct)
        mu = torch.empty(R, dtype=torch.float64, device=dev)
        var = torch.empty(R, dtype=torch.float64, device=dev)
        need_bwd = any(ctx.needs_input_grad)
        craw = torch.empty(R, dtype=torch.float64, device=dev) if (need_bwd and training) else None
        cnt = torch.zeros(1, dtype=torch.int32, device=dev) if (need_bwd and training) else None
        Ts = Us = None
        if need_bwd:
            nsave = lib.mobo_rows_save_doubles(M, R)
            Ts = torch.empty(nsave, dtype=torch.float64, device=dev)
            Us = torch.empty(nsave, dtype=torch.float64, device=dev)
        _lib.check(lib.mobo_layer_rows_fwd(kind, d, M, _lib.ptr(Zx_), _lib.ptr(zf_), _lib.ptr(theta_),
                                           _lib.ptr(ops_), _lib.ptr(x_), xrep, _lib.ptr(mu_prev_),
                                           _lib.ptr(var_prev_), prep, _lib.ptr(eps_), eps_mod, _lib.ptr(f_direct_),
                                           R, int(training), _lib.ptr(mu), _lib.ptr(var), _lib.ptr(craw),
                                           _lib.ptr(cnt), _lib.ptr(Ts), _lib.ptr(Us),
                                           _lib.stream_ptr()), "mobo_layer_rows_fwd")
        if need_bwd:
            ctx.save_for_backward(ops_, theta_, zf_, Zx_, x_, mu_prev_, var_prev_, eps_, f_direct_, craw, cnt, Ts, Us)
            ctx.cfg = (kind, xrep, prep, eps_mod, R, int(training))
        return mu, var

    @staticmethod
    def backward(ctx, dmu, dvar):
        lib = _lib.load()
        ops, theta, zf, Zx, x, mu_prev, var_prev, eps, f_direct, craw, cnt, Ts, Us = ctx.saved_tensors
        kind, xrep, prep, eps_mod, R, training = ctx.cfg
        M, d = Zx.shape
        dev = Zx.device
        need = ctx.needs_input_grad
        want_x = need[4]
        want_param = need[0] or need[1] or need[2]
        dmu = dmu.contiguous()
        dvar = dvar.contiguous()
        gops = torch.zeros_like(ops) if need[0] else None
        dtheta = torch.zeros_like(theta) if want_param else None
        dzf = torch.zeros(M, dtype=torch.float64, device=dev) if (want_param and kind == 1) else None
        df = torch.zeros(R, dtype=torch.float64, device=dev) if kind == 1 else None
        dxrow = torch.empty(R, d, dtype=torch.float64, device=dev) if want_x else None
        work = torch.empty(lib.mobo_rows_bwd_work_doubles(M, R), dtype=torch.float64, device=dev)
        _lib.check(lib.mobo_layer_rows_bwd(kind, d, M, _lib.ptr(Zx), _lib.ptr(zf), _lib.ptr(theta), _lib.ptr(ops),
                                           _lib.ptr(x), xrep, _lib.ptr(mu_prev), _lib.ptr(var_prev), prep,
                                           _lib.ptr(eps), eps_mod, _lib.ptr(f_direct), R, training, _lib.ptr(dmu),
                                           _lib.ptr(dvar), _lib.ptr(craw), _lib.ptr(cnt),
                                           _lib.ptr(Ts), _lib.ptr(Us), int(want_param), _lib.ptr(df),
                                           _lib.ptr(dxrow), _lib.ptr(dtheta), _lib.ptr(dzf), _lib.ptr(gops),
                                           _lib.ptr(work), _lib.stream_ptr()), "mobo_layer_rows_bwd")
        dx = dmu_prev = dvar_prev = df_direct = None
        if want_x:
            dx = dxrow.view(-1, xrep, d).sum(1) if xrep > 1 else dxrow
        if kind == 1:
            if f_direct is not None:
                df_direct = df if need[8] else None
            elif need[5] or need[6]:
                # f = mu_prev + sqrt(max(var_prev, 1e-10)) * eps   (layers/mfdgp_hidden_layer.py:263-274)
                idx = torch.arange(R, device=dev)
                e = eps[idx % eps_mod] if eps_mod != R else eps
                dmu_prev = df.view(-1, prep).sum(1)
                vc = var_prev.clamp_min(MIN_VARIANCE)
                dvar_prev = (df * e).view(-1, prep).sum(1) / (2.0 * vc.sqrt()) * (var_prev >= MIN_VARIANCE)
        return (gops, dtheta if need[1] else None, dzf if need[2] else None, None, dx, dmu_prev, dvar_prev, None,
                df_direct, None, None, None, None, None, None)


def layer_rows(ops, theta, zf, Zx, x, mu_prev=None, var_prev=None, eps=None, f_direct=None, kind=0, xrep=1, prep=1,
               eps_mod=None, R=None, training=True):
    """mean / raw variance of q(f_l) for R rows.  Row r reads x[r // xrep]; for kind 1 its propagated input is
    f_direct[r] or mu_prev[r // prep] + sqrt(max(var_prev[r // prep], 1e-10)) * eps[r % eps_mod]."""
    if R is None:
        R = x.shape[0] * xrep
    if eps_mod is None:
        eps_mod = eps.numel() if eps is not None else 1
    return _LayerRows.apply(ops, theta, zf, Zx, x, mu_prev, var_prev, eps, f_direct, kind, xrep, prep, eps_mod, R,
                            training)


class AcqChain(object):
    """The constants of one model's eval-mode acquisition chain up to layer ``fidelity``: per layer the operator
    buffer, constrained theta, propagated inducing column zf and S fixed normals (None at layer 0), the shared
    inducing inputs Zx and the likelihood's noise bounds."""

    def __init__(self, fidelity, M, S, Zx, zf, theta, ops, samples, noise_lower, noise_upper):
        self.fidelity, self.M, self.S, self.Zx = fidelity, M, S, Zx
        self.zf, self.theta, self.ops, self.samples = zf, theta, ops, samples
        self.noise_lower, self.noise_upper = noise_lower, noise_upper


def _acq_forward(chain, X, raw_noise, chunk):
    lib = _lib.load()
    c = chain
    n, d = X.shape
    out_mu = torch.empty(n, dtype=torch.float64, device=X.device)
    out_var = torch.empty(n, dtype=torch.float64, device=X.device)
    chunk = min(n, chunk)
    scratch = torch.empty(4 * chunk * c.S, dtype=torch.float64, device=X.device)
    for a in range(0, n, chunk):
        b = min(n, a + chunk)
        _lib.check(lib.mobo_acq_moments(c.fidelity, d, c.M, c.S, b - a, _lib.ptr(c.Zx), _lib.ptr_array(c.zf),
                                        _lib.ptr_array(c.theta), _lib.ptr_array(c.ops), _lib.ptr_array(c.samples),
                                        _lib.ptr(raw_noise), c.noise_lower, c.noise_upper, _lib.ptr(X[a:b]),
                                        _lib.ptr(out_mu[a:b]), _lib.ptr(out_var[a:b]), _lib.ptr(scratch),
                                        _lib.stream_ptr()), "mobo_acq_moments")
    return out_mu, out_var


class _AcqMoments(torch.autograd.Function):
    """(out_mu, out_var) of the acquisition chain, differentiable with respect to X and raw_noise.  The forward keeps
    no rows: the backward recomputes each chunk's forward (mobo_acq_moments_bwd), so the memory of d / dX is bounded
    by the chunk, not by the number of candidates."""

    @staticmethod
    def forward(ctx, X, raw_noise, chain, chunk, grad_chunk):
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(X, raw_noise)
        ctx.chain, ctx.grad_chunk = chain, grad_chunk
        return _acq_forward(chain, _c(X), _c(raw_noise), chunk)

    @staticmethod
    def backward(ctx, d_mu, d_var):
        lib = _lib.load()
        X, raw_noise = ctx.saved_tensors
        c = ctx.chain
        X, rn = _c(X), _c(raw_noise)
        d_mu, d_var = _c(d_mu), _c(d_var)
        n, d = X.shape
        dX = torch.zeros(n, d, dtype=torch.float64, device=X.device)
        dn = torch.zeros(1, dtype=torch.float64, device=X.device) if ctx.needs_input_grad[1] else None
        chunk = min(n, ctx.grad_chunk)
        work = torch.empty(lib.mobo_acq_bwd_work_doubles(c.fidelity, d, c.M, c.S, chunk), dtype=torch.float64,
                           device=X.device)
        # chunks write disjoint rows of dX; d raw_noise sums over all of them
        for a in range(0, n, chunk):
            b = min(n, a + chunk)
            _lib.check(lib.mobo_acq_moments_bwd(
                c.fidelity, d, c.M, c.S, b - a, _lib.ptr(c.Zx), _lib.ptr_array(c.zf), _lib.ptr_array(c.theta),
                _lib.ptr_array(c.ops), _lib.ptr_array(c.samples), _lib.ptr(rn), c.noise_lower, c.noise_upper,
                _lib.ptr(X[a:b]), None if d_mu is None else _lib.ptr(d_mu[a:b]),
                None if d_var is None else _lib.ptr(d_var[a:b]), 1, _lib.ptr(dX[a:b]), _lib.ptr(dn), _lib.ptr(work),
                _lib.stream_ptr()), "mobo_acq_moments_bwd")
        return (dX if ctx.needs_input_grad[0] else None, None if dn is None else dn.reshape(raw_noise.shape),
                None, None, None)


def acq_moments(chain, X, raw_noise, chunk, grad_chunk):
    """Moment-matched (mean, variance) over the S samples of the acquisition chain for the n candidates X (n, d):
    MFDGP.predict_for_acquisition (models/mfdgp.py:237-262) in enqueues of ``chunk`` candidates.  When X requires a
    gradient, the result is differentiable with respect to X and raw_noise, and the backward runs in chunks of
    ``grad_chunk`` candidates."""
    if torch.is_grad_enabled() and X.requires_grad:
        return _AcqMoments.apply(X, raw_noise, chain, chunk, grad_chunk)
    with torch.no_grad():
        return _acq_forward(chain, X, raw_noise, chunk)
