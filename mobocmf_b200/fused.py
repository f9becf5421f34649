"""Fused ELBO step and Adam update: host mirror of ``mobo_elbo_step`` / ``mobo_adam`` (include/mobocmf_b200.h).

``FusedELBOStep(model, elbo)(x_batch, y_batch, fidelities)`` is the body of ``_update_model``
(``mobocmf/util/blackbox_mfdgp_fitter.py:161-168``) up to ``loss.backward()``: it returns ``(loss, kl_scaled)`` as device
scalars and leaves d loss / d parameter in every trainable parameter's ``.grad`` (slices of one flat buffer, see
``util.distributed.FlatGrads``) — one ctypes call, ~50 kernel launches, no host synchronisation, no torch autograd.
``Adam`` is ``torch.optim.Adam`` (same defaults, same state names) on one multi-tensor kernel launch.

The composable autograd path (``functional.py``) computes the same numbers through the same kernels; the fused path is
used whenever its preconditions hold (``FusedELBOStep.supported``), there is no CPU fallback in either.
"""
import ctypes

import torch

from . import _lib
from .errors import NanError, NotPSDError
from .util.distributed import FlatGrads

MAX_LAYERS = 8
MAX_THETA = 21
_dp = ctypes.c_void_p


class LayerDesc(ctypes.Structure):
    _fields_ = [("Zx", _dp), ("raw_theta", _dp * MAX_THETA), ("g_raw_theta", _dp * MAX_THETA), ("m", _dp),
                ("Lq", _dp), ("g_m", _dp), ("g_Lq", _dp), ("raw_noise", _dp), ("g_raw_noise", _dp),
                ("noise_lower", ctypes.c_double), ("noise_upper", ctypes.c_double), ("eps", _dp)]


class StepDesc(ctypes.Structure):
    _fields_ = [("L", ctypes.c_int), ("d", ctypes.c_int), ("M", ctypes.c_int), ("S", ctypes.c_int),
                ("B", ctypes.c_longlong), ("num_data", ctypes.c_longlong), ("jitter", ctypes.c_double),
                ("x", _dp), ("y", _dp), ("fid", _dp), ("layer", LayerDesc * MAX_LAYERS), ("out", _dp),
                ("workspace", _dp), ("accumulate", ctypes.c_int), ("ctx", _dp)]


class AdamTensor(ctypes.Structure):
    _fields_ = [("p", _dp), ("g", _dp), ("exp_avg", _dp), ("exp_avg_sq", _dp), ("n", ctypes.c_longlong)]


def _bind():
    return _lib.load()


def _addr(t, index=0):
    return t.data_ptr() + index * t.element_size()


def _layer_raw_slots(layer):
    """[(parameter, flat index)] of the RAW hyper-parameters in the kernels' theta order (include/mobocmf_b200.h):
    layer 0 [a, l_0..]; layer >= 1 [a1, v_lin, a_f, l_f, a2, l1_0.., l2_0..]."""
    cm = layer.covar_module
    d = layer.x_dims
    if layer.num_layer == 0:
        return [(cm.raw_outputscale, 0)] + [(cm.base_kernel.raw_lengthscale, c) for c in range(d)]
    k_x1, k_sum = cm.kernels[0].kernels
    k_lin, k_f = k_sum.kernels
    k_x2 = cm.kernels[1]
    return ([(k_x1.raw_outputscale, 0), (k_lin.raw_variance, 0), (k_f.raw_outputscale, 0),
             (k_f.base_kernel.raw_lengthscale, 0), (k_x2.raw_outputscale, 0)] +
            [(k_x1.base_kernel.raw_lengthscale, c) for c in range(d)] +
            [(k_x2.base_kernel.raw_lengthscale, c) for c in range(d)])


class FusedELBOStep(object):
    """One MFDGP's ELBO step on the fused kernel sequence."""

    def __init__(self, model, elbo):
        ok, why = self.supported(model)
        if not ok:
            raise RuntimeError("fused ELBO step not applicable: " + why)
        self.model = model
        self.elbo = elbo
        self.lib = _bind()
        self.L = model.num_hidden_layers
        self.layers = [getattr(model, model.name_hidden_layer + str(i)) for i in range(self.L)]
        self.liks = [getattr(model, model.name_hidden_layer_likelihood + str(i)) for i in range(self.L)]
        self.M = self.layers[0].num_inducing
        self.d = model.input_dims
        self.device = self.layers[0]._Zx().device
        # [0] loss, [1] KL B/N, [2] data term, [3] status, [4] sticky status, [5] sticky non-finite loss,
        # [6] "this step failed" (the Adam kernel's skip flag), [7] psd_safe_cholesky retries (include/mobocmf_b200.h)
        self.out = torch.zeros(8, dtype=torch.float64, device=self.device)
        self.skip_flag = self.out[6:7]
        self.flat = None
        self._ws = {}             # (B, S) -> workspace; entries referenced by a captured CUDA graph are pinned
        self._ws_pinned = set()
        self._desc = StepDesc()
        self._sig = None
        # this step's own side stream + events (include/mobocmf_b200.h: mobo_step_ctx_create): concurrently trained
        # models must not share one, their operator-chain backwards would serialise on it
        with torch.cuda.device(self.device):
            self._ctx = self.lib.mobo_step_ctx_create()
        if not self._ctx:
            raise RuntimeError("mobocmf_b200: mobo_step_ctx_create failed")

    def wait_bucket(self, k, stream):
        """Makes ``stream`` wait until leading gradient block k of ``self.flat`` (d L_q of a layer) is final in the step
        enqueued last (include/mobocmf_b200.h: mobo_step_ctx_wait_layer)."""
        _lib.check(self.lib.mobo_step_ctx_wait_layer(self._ctx, self._bucket_layer[k],
                                                     ctypes.c_void_p(stream.cuda_stream)), "mobo_step_ctx_wait_layer")

    def __del__(self):
        ctx, self._ctx = getattr(self, "_ctx", None), None
        if ctx:
            try:
                torch.cuda.synchronize(self.device)     # no step that uses the context may still be in flight
                self.lib.mobo_step_ctx_destroy(ctx)
            except Exception:
                pass

    @staticmethod
    def supported(model):
        layers = [getattr(model, model.name_hidden_layer + str(i)) for i in range(model.num_hidden_layers)]
        p = layers[0].variational_strategy._variational_distribution.variational_mean
        if not p.is_cuda or p.dtype != torch.float64:
            return False, "the model must hold fp64 CUDA parameters"
        if model.use_only_highest_fidelity is True:
            return False, "only-highest-fidelity models use per-layer inducing inputs"
        if model.num_hidden_layers > MAX_LAYERS or model.input_dims > 8 or layers[0].num_inducing > 256:
            return False, "shape outside the kernels' limits (L <= 8, d <= 8, M <= 256)"
        z0 = layers[0]._Zx()
        for lay in layers[1:]:
            z = lay._Zx()
            if z.shape != z0.shape or not bool(torch.equal(z, z0)):
                return False, "layers do not share their inducing inputs"
        return True, ""

    # ---- descriptor -------------------------------------------------------------------------------------------
    def _signature(self):
        sig = []
        for p in self.model.parameters():
            sig.append((p.data_ptr(), p.requires_grad, None if p.grad is None else p.grad.data_ptr()))
        return tuple(sig)

    def _ensure_grads(self):
        for p in self.model.parameters():
            if not p.requires_grad and p.grad is not None:
                p.grad = None      # frozen since an earlier phase: torch's zero_grad would have dropped it too
        params = [p for p in self.model.parameters() if p.requires_grad]
        # the M x M blocks d L_q lead the flat buffer, highest layer first: the order in which the step completes them
        # (FlatGrads.all_reduce_overlapped sends each behind the lower layers' row kernels)
        first = [lay.variational_strategy._variational_distribution.chol_variational_covar for lay in self.layers[::-1]]
        first = [p for p in first if p.requires_grad]
        want = [id(p) for p in first] + [id(p) for p in params if not any(p is q for q in first)]
        if self.flat is None or [id(p) for p in self.flat.params] != want:
            self.flat = FlatGrads(params, first=first)
            self._bucket_layer = [self.layers.index(lay) for lay in self.layers[::-1]
                                  if lay.variational_strategy._variational_distribution.chol_variational_covar.requires_grad]
        elif not self.flat.attached():
            self.flat.reattach()

    def _build_desc(self):
        D = self._desc
        D.L, D.d, D.M = self.L, self.d, self.M
        D.out = self.out.data_ptr()
        D.accumulate = 0
        D.ctx = self._ctx
        D.jitter = float(self.layers[0].variational_strategy.jitter_val)
        self._keep = []
        for l, (layer, lik) in enumerate(zip(self.layers, self.liks)):
            ld = D.layer[l]
            zx = layer._Zx()
            self._keep.append(zx)
            ld.Zx = zx.data_ptr()
            slots = _layer_raw_slots(layer)
            for i in range(MAX_THETA):
                if i < len(slots):
                    p, idx = slots[i]
                    ld.raw_theta[i] = _addr(p, idx)
                    ld.g_raw_theta[i] = _addr(p.grad, idx) if p.requires_grad else None
                else:
                    ld.raw_theta[i] = None
                    ld.g_raw_theta[i] = None
            vd = layer.variational_strategy._variational_distribution
            ld.m, ld.Lq = vd.variational_mean.data_ptr(), vd.chol_variational_covar.data_ptr()
            ld.g_m = vd.variational_mean.grad.data_ptr() if vd.variational_mean.requires_grad else None
            ld.g_Lq = vd.chol_variational_covar.grad.data_ptr() if vd.chol_variational_covar.requires_grad else None
            rn = lik.noise_covar.raw_noise
            ld.raw_noise = rn.data_ptr()
            ld.g_raw_noise = rn.grad.data_ptr() if rn.requires_grad else None
            c = lik.noise_covar.raw_noise_constraint
            ld.noise_lower, ld.noise_upper = float(c.lower_bound), float(c.upper_bound)

    def _prepare(self):
        self._ensure_grads()
        sig = self._signature()
        if sig != self._sig:
            for p in self.model.parameters():
                if not p.is_contiguous():
                    raise RuntimeError("mobocmf_b200: parameters must be contiguous")
            self._build_desc()
            self._sig = sig

    MAX_UNPINNED_WORKSPACES = 2

    def _workspace(self, B, S, pin=False, small=False):
        """Scratch of the step for a (B, S) shape.  A captured CUDA graph bakes the workspace's address in, so a
        workspace that a graph references (``pin=True``) lives as long as this object; the others are kept for the
        last few shapes only (full batch + ragged last batch of an epoch).  ``small``: the scratch of
        ``mobo_elbo_step_small`` (its own size query) instead of ``mobo_elbo_step``'s."""
        key = (B, S, "small") if small else (B, S)
        ws = self._ws.get(key)
        if ws is None:
            loose = [k for k in self._ws if k not in self._ws_pinned]
            while len(loose) >= self.MAX_UNPINNED_WORKSPACES:
                del self._ws[loose.pop(0)]
            query = self.lib.mobo_elbo_step_small_workspace_doubles if small else \
                self.lib.mobo_elbo_step_workspace_doubles
            n = query(self.L, self.d, self.M, S, B)
            ws = torch.empty(n, dtype=torch.float64, device=self.device)
            self._ws[key] = ws
        else:
            self._ws[key] = self._ws.pop(key)      # most recently used last
        if pin:
            self._ws_pinned.add(key)
        return ws

    def applies(self, x_batch):
        """False when the minibatch equals the inducing inputs row for row: upstream then short-cuts layer 0 to
        N(m, S) (quirk Q4), which only the composable path reproduces.  Costs a device sync only when B == M."""
        if x_batch.shape[0] != self.M:
            return True
        Z = self.layers[0]._Zx()
        host = getattr(x_batch, "_mobo_host", None)       # host copy attached by the fitter's loader: no sync
        if host is not None:
            key = (Z.data_ptr(), Z._version)
            if getattr(self, "_z_host_key", None) != key:
                self._z_host, self._z_host_key = Z.detach().cpu(), key
            return not bool(torch.equal(host, self._z_host))
        return not bool(torch.equal(x_batch, Z))

    # ---- the step ---------------------------------------------------------------------------------------------
    def __call__(self, x_batch, y_batch, fidelities, eps=None, num_samples=1, accumulate=False, check_shortcut=True,
                 pin_workspace=False):
        """Returns (loss = -ELBO, KL * B / N) as 0-d device tensors (views of one result buffer, overwritten by the
        next call) and writes the gradients.  ``eps``: optional list indexed by layer of the training normals
        (B*S values for layers >= 1; reference: float32 ``torch.normal`` of shape (1, B), quirk Q6)."""
        keep = self._stage(x_batch, y_batch, fidelities, eps, num_samples, accumulate, check_shortcut,
                           pin_workspace, small=False)
        _lib.check(self.lib.mobo_elbo_step(ctypes.byref(self._desc), _lib.stream_ptr()), "mobo_elbo_step")
        return self._launched(keep)

    def _stage(self, x_batch, y_batch, fidelities, eps, num_samples, accumulate, check_shortcut, pin_workspace,
               small):
        """Fills ``self._desc`` for one step on this minibatch (the launch is the caller's); returns the tensors the
        enqueued step reads, which must stay alive until the next call."""
        B = x_batch.shape[0]
        S = int(num_samples)
        if x_batch.shape[1] != self.d or y_batch.numel() != B or fidelities.numel() != B:
            raise ValueError("x (B, d), y (B, 1), fidelities (B, 1) expected")
        if check_shortcut and not self.applies(x_batch):
            raise RuntimeError("x_batch equals the inducing inputs (quirk Q4 shortcut): use the composable path")
        self._prepare()
        D = self._desc
        x = x_batch.contiguous()
        y = y_batch.contiguous()
        f = fidelities.contiguous()
        if not (x.is_cuda and x.dtype == torch.float64 and y.dtype == torch.float64 and f.dtype == torch.float64):
            raise RuntimeError("mobocmf_b200 kernels need fp64 CUDA tensors (no CPU fallback)")
        keep = [x, y, f]
        for l in range(1, self.L):
            e = None if eps is None else eps[l]
            if e is None:
                e = torch.randn(B * S, device=self.device, dtype=torch.float32)
            e = e.to(device=self.device, dtype=torch.float64).reshape(-1).contiguous()
            if e.numel() != B * S:
                raise ValueError("eps[%d] must hold B * num_samples normals" % l)
            keep.append(e)
            D.layer[l].eps = e.data_ptr()
        D.layer[0].eps = None
        D.S, D.B, D.num_data = S, B, int(self.elbo.num_data)
        D.x, D.y, D.fid = x.data_ptr(), y.data_ptr(), f.data_ptr()
        D.workspace = self._workspace(B, S, pin=pin_workspace, small=small).data_ptr()
        D.accumulate = 1 if accumulate else 0
        return keep

    def _launched(self, keep):
        self._last_inputs = keep          # keep the step's inputs alive until the next call (async kernels)
        for layer in self.layers:         # parameters are about to change: drop the composable path's cache
            layer._ops_cache = None
        return self.out[0], self.out[1]

    def check(self):
        """Synchronises and raises like upstream's NotPSDError / NanError when ANY step since the last check failed:
        a Cholesky factorisation that psd_safe_cholesky's three jitter retries could not rescue, or a non-finite ELBO.
        The failing step's Adam update was skipped on the device (``skip_flag``), so the parameters are still the
        ones that failed.  Called by the fitter at its reporting boundaries instead of once per step."""
        o = self.out.tolist()
        st = o[4] if o[4] != 0.0 else o[3]
        if st != 0.0:
            self.out[4:6].zero_()
            raise NotPSDError("NotPSDError: K(Z, Z) + jitter I of layer %d is not positive definite (after the "
                              "1e-8, 1e-7, 1e-6 jitter retries)" % (int(st) - 1))
        if o[5] != 0.0 or o[0] != o[0] or o[0] in (float("inf"), float("-inf")):
            self.out[4:6].zero_()
            raise NanError("NanError: the ELBO is not finite")

    def retries(self):
        """psd_safe_cholesky retries the last step needed (0 .. 3); synchronises."""
        return int(self.out[7])


class Adam(torch.optim.Optimizer):
    """``torch.optim.Adam`` (defaults of ``mobocmf/util/blackbox_mfdgp_fitter.py:126,132,259``) with the update of all
    parameters in ONE kernel launch (``mobo_adam``).  State keys match torch's (``step``, ``exp_avg``,
    ``exp_avg_sq``) so ``state_dict`` round-trips with ``torch.optim.Adam``.  ``capturable=True`` keeps the step count
    in a device tensor (like torch's flag of the same name) so that ``step()`` can be captured in a CUDA graph."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, capturable=False):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps))
        self.capturable = capturable
        self._step_dev = None       # device-resident step count of the FIRST cohort of parameters (capturable)
        self._cohorts = []          # one device count per set of parameters that joined in the same step() call
        self._tables = {}
        # optional 1-element device tensor: != 0 -> the update is skipped on the device (FusedELBOStep.skip_flag:
        # the step that produced the gradients hit NotPSDError / NanError, where upstream never reaches step())
        self.skip_flag = None

    def zero_grad(self, set_to_none=False):
        # gradients live in a persistent flat buffer that the fused step overwrites: keep the tensors
        return super().zero_grad(set_to_none=set_to_none)

    def _table(self, key, chunk):
        """ctypes table of (param, grad, exp_avg, exp_avg_sq, n) for a chunk of <= 64 parameters, rebuilt only when a
        pointer changes."""
        sig = tuple((p.data_ptr(), p.grad.data_ptr()) for p in chunk)
        hit = self._tables.get(key)
        if hit is not None and hit[0] == sig:
            return hit[1]
        arr = (AdamTensor * len(chunk))()
        for j, p in enumerate(chunk):
            st = self.state[p]
            arr[j].p, arr[j].g = p.data_ptr(), p.grad.data_ptr()
            arr[j].exp_avg, arr[j].exp_avg_sq = st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr()
            arr[j].n = p.numel()
        self._tables[key] = (sig, arr)
        return arr

    # ---- CUDA-graph capture support: warm-up and capture run real updates that must not count as training ----
    @torch.no_grad()
    def snapshot(self):
        """Copies of the parameters and of every piece of optimiser state (moments, device step counts)."""
        params = [p for g in self.param_groups for p in g["params"]]
        snap = {"params": [(p, p.detach().clone()) for p in params], "state": [], "cohorts": len(self._cohorts),
                "counts": [c.clone() for c in self._cohorts]}
        for p in params:
            st = self.state.get(p)
            if st:
                snap["state"].append((p, st["exp_avg"].clone(), st["exp_avg_sq"].clone(),
                                      st["step"] if not torch.is_tensor(st["step"]) else None))
        return snap

    @torch.no_grad()
    def restore(self, snap):
        """Undo every update since ``snapshot`` in place (addresses baked into captured graphs stay valid): state
        that existed is restored, state created since is zeroed."""
        for p, v in snap["params"]:
            p.copy_(v)
        had = {id(p) for p, _, _, _ in snap["state"]}
        for p, m, v, step in snap["state"]:
            st = self.state[p]
            st["exp_avg"].copy_(m); st["exp_avg_sq"].copy_(v)
            if step is not None:
                st["step"] = step
        for p, _ in snap["params"]:
            st = self.state.get(p)
            if st and id(p) not in had:
                st["exp_avg"].zero_(); st["exp_avg_sq"].zero_()
                if not torch.is_tensor(st["step"]):
                    st["step"] = 0
        for i, c in enumerate(self._cohorts):
            if i < snap["cohorts"]:
                c.copy_(snap["counts"][i])
            else:
                c.zero_()

    @torch.no_grad()
    def step(self, closure=None):
        if closure is not None:
            raise NotImplementedError("closures are not used by the reference's training loops")
        lib = _bind()
        skip = None if self.skip_flag is None else _lib.ptr(self.skip_flag)
        ticked = set()
        new_cohort = None
        for gi, group in enumerate(self.param_groups):
            # frozen parameters are skipped even if a stale .grad survives from an earlier phase (torch's
            # zero_grad(set_to_none=True) would have dropped it)
            ps = [p for p in group["params"] if p.requires_grad and p.grad is not None]
            if not ps:
                continue
            for p in ps:
                st = self.state[p]
                if not st:
                    if not (p.is_cuda and p.dtype == torch.float64 and p.is_contiguous() and p.grad.is_contiguous()):
                        raise RuntimeError("mobocmf_b200.Adam needs contiguous fp64 CUDA parameters (no CPU fallback)")
                    if self.capturable:
                        # parameters that join in the same call share one device-resident count; a parameter that
                        # joins later starts its own (its bias correction must count ITS steps, like torch's
                        # per-parameter `step`)
                        if new_cohort is None:
                            new_cohort = torch.zeros((), dtype=torch.int64, device=p.device)
                            self._cohorts.append(new_cohort)
                            if self._step_dev is None:
                                self._step_dev = new_cohort
                        st["step"] = new_cohort
                    else:
                        st["step"] = 0
                    st["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                    st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
            b1, b2 = group["betas"]
            if self.capturable:
                for ci, cnt in enumerate(self._cohorts):
                    sel = [p for p in ps if self.state[p]["step"] is cnt]
                    if not sel:
                        continue
                    if ci not in ticked:
                        _lib.check(lib.mobo_adam_tick(_lib.ptr(cnt), skip, _lib.stream_ptr()), "mobo_adam_tick")
                        ticked.add(ci)
                    for i in range(0, len(sel), 64):
                        chunk = sel[i:i + 64]
                        _lib.check(lib.mobo_adam(len(chunk), self._table((gi, ci, i), chunk), float(group["lr"]),
                                                 float(b1), float(b2), float(group["eps"]), 0, _lib.ptr(cnt), skip,
                                                 _lib.stream_ptr()), "mobo_adam")
                continue
            steps = {int(self.state[p]["step"]) for p in ps}
            for step0 in sorted(steps):
                sel = [p for p in ps if int(self.state[p]["step"]) == step0]
                for i in range(0, len(sel), 64):
                    chunk = sel[i:i + 64]
                    _lib.check(lib.mobo_adam(len(chunk), self._table((gi, "host", step0 - min(steps), i), chunk),
                                             float(group["lr"]), float(b1), float(b2), float(group["eps"]),
                                             step0 + 1, None, skip, _lib.stream_ptr()), "mobo_adam")
                for p in sel:
                    # a skipped (failed) step still counts here: the host cannot know without a synchronisation, and
                    # the failure is raised at the next FusedELBOStep.check() anyway
                    self.state[p]["step"] = step0 + 1
        return None


class GraphedELBOStep(object):
    """The fused step + Adam update of one minibatch shape captured ONCE in a CUDA graph and replayed per step: one
    graph launch instead of ~55 kernel launches.  This is the path for the reference's own configurations (full batch,
    M = N of a few tens, ``examples/*``), where a step is a few hundred microseconds of launch latency.

    ``optimizer`` must be ``Adam(..., capturable=True)`` over the model's parameters.  The training normals are drawn
    inside the graph by torch's graph-safe generator, so every replay uses fresh ones."""

    def __init__(self, step, optimizer, batch_size, num_samples=1, warmup=3, static_eps=False):
        if not isinstance(optimizer, Adam) or not optimizer.capturable:
            raise ValueError("GraphedELBOStep needs mobocmf_b200.fused.Adam(capturable=True)")
        self.step, self.optimizer, self.S = step, optimizer, int(num_samples)
        optimizer.skip_flag = step.skip_flag
        dev, d = step.device, step.d
        # static_eps: the caller supplies the training normals on every call (parity tests); otherwise they are drawn
        # inside the graph
        self.eps = None
        if static_eps:
            self.eps = [None] + [torch.zeros(batch_size * self.S, dtype=torch.float64, device=dev)
                                 for _ in range(1, step.L)]
        self.x = torch.zeros(batch_size, d, dtype=torch.float64, device=dev)
        self.y = torch.zeros(batch_size, 1, dtype=torch.float64, device=dev)
        self.f = torch.zeros(batch_size, 1, dtype=torch.float64, device=dev)
        self.graph = None
        self._warmup = warmup

    def _capture(self):
        # parameters are NOT stepped during warm-up / capture side effects: snapshot and restore them and the
        # optimiser state, so that capturing does not count as training steps
        snap = self.optimizer.snapshot()
        out_keep = self.step.out.clone()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(self._warmup):
                self.step(self.x, self.y, self.f, eps=self.eps, num_samples=self.S, check_shortcut=False,
                          pin_workspace=True)
                self.optimizer.step()
        torch.cuda.current_stream().wait_stream(s)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss, self.kl = self.step(self.x, self.y, self.f, eps=self.eps, num_samples=self.S,
                                           check_shortcut=False, pin_workspace=True)
            self.optimizer.step()
        self.optimizer.restore(snap)
        with torch.no_grad():
            self.step.out.copy_(out_keep)      # sticky status flags: staging data of the warm-up steps does not count

    def _stage(self, x_batch, y_batch, fidelities, eps):
        self.x.copy_(x_batch); self.y.copy_(y_batch.reshape(-1, 1)); self.f.copy_(fidelities.reshape(-1, 1))
        if self.eps is not None:
            if eps is None:
                raise ValueError("this graph was built with static_eps=True: pass eps")
            for l in range(1, self.step.L):
                self.eps[l].copy_(eps[l].reshape(-1))

    def __call__(self, x_batch, y_batch, fidelities, eps=None, check_shortcut=True):
        if check_shortcut and not self.step.applies(x_batch):
            raise RuntimeError("x_batch equals the inducing inputs (quirk Q4 shortcut): use the composable path")
        if self.graph is None:
            self._stage(x_batch, y_batch, fidelities, eps)
            self._capture()
        self._stage(x_batch, y_batch, fidelities, eps)
        self.graph.replay()
        for layer in self.step.layers:
            layer._ops_cache = None
        return self.loss, self.kl


class SmallModelsELBOStep(object):
    """The ELBO steps of several independent small MFDGPs (M <= 64: the reference's own problems) in ONE launch of
    ``mobo_elbo_step_small``, one CTA per model: what ``BlackBoxMFDGPFitter._train_mfdgp`` does for the K black boxes
    of a BO iteration (``mobocmf/util/blackbox_mfdgp_fitter.py:156-173`` per model), without the ~45 launches per
    model-step of ``FusedELBOStep``.  Each model keeps its own ``FusedELBOStep`` (descriptor, flat gradient buffer,
    ``out`` flags, ``check()``, the Q4 test ``applies()``); ``steps`` may pass existing ones to build on."""

    MAX_M = 64

    def __init__(self, models, elbos, steps=None):
        ok, why = self.supported(models)
        if not ok:
            raise RuntimeError("small-model ELBO step not applicable: " + why)
        self.steps = list(steps) if steps is not None else [FusedELBOStep(m, e) for m, e in zip(models, elbos)]
        if len(self.steps) != len(models) or any(s.model is not m for s, m in zip(self.steps, models)):
            raise ValueError("steps must be the FusedELBOStep of each model, in order")
        self.lib = _bind()
        self._descs = (StepDesc * len(self.steps))()

    @staticmethod
    def supported(models):
        models = list(models)
        if not models:
            return False, "no models"
        for m in models:
            ok, why = FusedELBOStep.supported(m)
            if not ok:
                return False, why
            if getattr(m, m.name_hidden_layer + "0").num_inducing > SmallModelsELBOStep.MAX_M:
                return False, "more than %d inducing points" % SmallModelsELBOStep.MAX_M
        return True, ""

    def __call__(self, batches, eps=None, num_samples=1, accumulate=False, check_shortcut=True, pin_workspace=False):
        """``batches[i] = (x, y, fid)`` of model i (each model its own B), or None: model i sits this step out.
        ``eps[i]``: optional per-layer normals of model i, as ``FusedELBOStep``; ``num_samples``: one S for all models
        or one per model.  Returns ``[(loss, kl)]`` per model (views of each model's result buffer; None for a model
        that sat out)."""
        if len(batches) != len(self.steps):
            raise ValueError("one batch (or None) per model expected")
        run, keeps = [], []
        for i, (step, b) in enumerate(zip(self.steps, batches)):
            if b is None:
                continue
            e = None if eps is None else eps[i]
            S = num_samples[i] if isinstance(num_samples, (list, tuple)) else num_samples
            keeps.append(step._stage(b[0], b[1], b[2], e, S, accumulate, check_shortcut, pin_workspace, small=True))
            self._descs[len(run)] = step._desc
            run.append(step)
        if run:
            _lib.check(self.lib.mobo_elbo_step_small(self._descs, len(run), _lib.stream_ptr()),
                       "mobo_elbo_step_small")
        res = {id(s): s._launched(k) for s, k in zip(run, keeps)}
        return [res.get(id(s)) for s in self.steps]


class GraphedSmallModelsELBOStep(object):
    """``SmallModelsELBOStep`` plus every model's own ``Adam`` update captured in one CUDA graph per combination of
    minibatch shapes (a ragged last batch gets its own graph) and replayed per step: one graph launch for all models.
    Each optimiser reads its own model's ``out[6]`` as skip flag, so a model whose step failed skips only its own
    update.  ``optimizers[i]`` must be ``Adam(..., capturable=True)`` over model i's parameters.  The training normals
    are drawn inside the graph unless ``static_eps`` (the caller passes them on every call)."""

    def __init__(self, small, optimizers, num_samples=1, warmup=3, static_eps=False):
        if len(optimizers) != len(small.steps):
            raise ValueError("one optimiser per model expected")
        for o in optimizers:
            if not isinstance(o, Adam) or not o.capturable:
                raise ValueError("GraphedSmallModelsELBOStep needs mobocmf_b200.fused.Adam(capturable=True)")
        self.small, self.optimizers, self.S = small, list(optimizers), int(num_samples)
        for o, st in zip(self.optimizers, small.steps):
            o.skip_flag = st.skip_flag
        self.static_eps, self._warmup = static_eps, warmup
        self.graphs = {}     # (batch shape or None per model) -> (static batches, static normals, graph, results)

    def _run(self, static, static_eps):
        res = self.small(static, eps=static_eps, num_samples=self.S, check_shortcut=False, pin_workspace=True)
        for o, b in zip(self.optimizers, static):
            if b is not None:
                o.step()
        return res

    def _capture(self, batches, eps):
        dev = self.small.steps[0].device
        static, static_eps = [], None if not self.static_eps else []
        for i, (st, b) in enumerate(zip(self.small.steps, batches)):
            static.append(None if b is None else (b[0].detach().clone(), b[1].detach().clone().reshape(-1, 1),
                                                  b[2].detach().clone().reshape(-1, 1)))
            if self.static_eps:
                B = 0 if b is None else b[0].shape[0]
                static_eps.append([None] + [torch.zeros(B * self.S, dtype=torch.float64, device=dev)
                                            for _ in range(1, st.L)])
        # warm-up and capture run real updates: they must not count as training steps
        snaps = [o.snapshot() for o in self.optimizers]
        outs = [st.out.clone() for st in self.small.steps]
        self._stage(static, static_eps, batches, eps)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(self._warmup):
                self._run(static, static_eps)
        torch.cuda.current_stream().wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            res = self._run(static, static_eps)
        for o, snap in zip(self.optimizers, snaps):
            o.restore(snap)
        with torch.no_grad():
            for st, o in zip(self.small.steps, outs):
                st.out.copy_(o)      # sticky status flags: staging data of the warm-up steps does not count
        return static, static_eps, graph, res

    def _stage(self, static, static_eps, batches, eps):
        for i, (dst, b) in enumerate(zip(static, batches)):
            if dst is None:
                continue
            dst[0].copy_(b[0]); dst[1].copy_(b[1].reshape(-1, 1)); dst[2].copy_(b[2].reshape(-1, 1))
            if static_eps is not None:
                if eps is None:
                    raise ValueError("this graph was built with static_eps=True: pass eps")
                for l in range(1, self.small.steps[i].L):
                    static_eps[i][l].copy_(eps[i][l].reshape(-1))

    def __call__(self, batches, eps=None, check_shortcut=True):
        """``batches[i] = (x, y, fid)`` of model i, or None (model i sits this step out: no step, no update).
        Returns ``[(loss, kl)]`` per model (None for one that sat out)."""
        if check_shortcut:
            for st, b in zip(self.small.steps, batches):
                if b is not None and not st.applies(b[0]):
                    raise RuntimeError("x_batch equals the inducing inputs (quirk Q4 shortcut): use the composable "
                                       "path for that model")
        key = tuple(None if b is None else tuple(b[0].shape) for b in batches)
        if key not in self.graphs:
            self.graphs[key] = self._capture(batches, eps)
        static, static_eps, graph, res = self.graphs[key]
        self._stage(static, static_eps, batches, eps)
        graph.replay()
        for st in self.small.steps:
            for layer in st.layers:
                layer._ops_cache = None
        return res
