"""Training orchestration — mirror of ``mobocmf/util/blackbox_mfdgp_fitter.py``: ``MFDGPHandler``,
``BlackBoxMFDGPFitter`` with the ELBO step (``_update_model``, :156-173), the conditioned step
(``_update_conditioned_models``, :272-346) and the theta / omega factors (:227-243).  Orchestration stays Python;
every MFDGP forward / backward inside the steps runs on the sm_100a kernels.

``sample_and_store_pareto_solution`` (:181-225) draws one RFF function sample per black box
(``MFDGP.sample_function_from_each_layer``) and extracts the Pareto set with ``mobocmf_b200.util.moop.MOOP``; the grid
evaluation and the non-dominated cull run on the GPU (SURVEY.md §8f-3).
"""
import sys
import warnings
from copy import deepcopy

import numpy as np
import torch

from ..fused import Adam
from ..gp import settings
from ..mlls.variational_elbo_mf import VariationalELBOMF
from ..models.mfdgp import MFDGP, TL
from .moop import MOOP, NotFeasiblePoints

ITER_PRINT = 1000


def _prod(t, dim):
    """torch.prod(t, dim) as a chain of multiplications: the derivative of torch.prod reads a zero count back to the
    host (a device synchronisation in every backward, and illegal inside a CUDA-graph capture); the chain has the same
    derivative, zeros included, and the reduced dimension is a handful of black boxes."""
    parts = torch.unbind(t, dim)
    if len(parts) == 0:
        return torch.ones(t.shape[:dim] + t.shape[dim + 1:], dtype=t.dtype, device=t.device)
    out = parts[0]
    for q in parts[1:]:
        out = out * q
    return out


def _normal_cdf(x):
    return 0.5 * (1.0 + torch.erf(x / np.sqrt(2.0)))


class _Loader(object):
    """DataLoader(TensorDataset(x, y, fid), batch_size, shuffle=True) on the device (fitter.py:35-36)."""

    def __init__(self, x, y, f, batch_size, shuffle=True):
        self.x, self.y, self.f, self.batch_size, self.shuffle = x, y, f, batch_size, shuffle
        # small data sets (the reference's own configurations): a host copy of x, so that the "batch equals the
        # inducing inputs" test of the fused step (quirk Q4) is answered on the host instead of by a device
        # synchronisation in every step
        self.x_host = x.detach().cpu() if x.shape[0] <= 4096 else None

    def __iter__(self):
        n = self.x.shape[0]
        # the permutation comes from torch's CPU generator, like the reference's DataLoader(shuffle=True)
        perm_host = torch.randperm(n) if self.shuffle else torch.arange(n)
        perm = perm_host.to(self.x.device)
        for i in range(0, n, self.batch_size):
            idx = perm[i:i + self.batch_size]
            xb = self.x[idx]
            if self.x_host is not None:
                xb._mobo_host = self.x_host[perm_host[i:i + self.batch_size]]
            yield xb, self.y[idx], self.f[idx]


class MFDGPHandler():
    MAX_TRIES_FOR_FEASIBLE_GRID = 50

    def __init__(self, x_train, y_train, fidelities_train, num_fidelities, batch_size, type_lengthscale,
                 previously_trained_model=None, init_params_to_prior_and_fix_them=False,
                 use_only_highest_fidelity=False, device=None):
        self.mfdgp = MFDGP(x_train.cpu(), y_train.cpu(), fidelities_train.cpu(), num_fidelities=num_fidelities,
                           type_lengthscale=type_lengthscale, previously_trained_model=previously_trained_model,
                           use_only_highest_fidelity=use_only_highest_fidelity,
                           init_params_to_prior_and_fix_them=init_params_to_prior_and_fix_them)
        self.mfdgp.double()
        if device is None:
            device = x_train.device if x_train.is_cuda else torch.device("cuda")
        self.device = device
        self.mfdgp.to(device)
        self.elbo = VariationalELBOMF(self.mfdgp, x_train.shape[-2], num_fidelities=num_fidelities)
        self.x, self.y, self.f = x_train.to(device), y_train.to(device), fidelities_train.to(device)
        self.train_loader = _Loader(self.x, self.y, self.f, batch_size, shuffle=True)
        self.iter_train_loader = None
        self.num_data = x_train.shape[0]
        self.num_fidelities = num_fidelities


class _GraphedConditionedStep(object):
    """One conditioned iteration (``_update_conditioned_models``, fitter.py:272-354: three MFDGP forwards per black
    box — minibatch, Pareto set, x-tilde —, the theta / omega factors, backward, Adam) captured ONCE in a CUDA graph
    and replayed per iteration.  At the reference's sizes the iteration is a few hundred small kernels and ~13 ms of
    Python / autograd dispatch when enqueued eagerly; a replay is one launch.  The minibatches are staged into static
    buffers, x-tilde and the training normals are drawn inside the graph by torch's graph-safe generator.  An
    iteration whose minibatch equals the inducing inputs (quirk Q4 changes the arithmetic) runs eagerly."""

    def __init__(self, fitter, handlers_objs, handlers_cons, optimizer, warmup=2, static_noise=False):
        self.fitter, self.optimizer, self.warmup = fitter, optimizer, warmup
        # static_noise (parity tests): x-tilde and the training normals are staged by the caller on every call instead
        # of being drawn inside the graph, so that a replay can be compared with the eager iteration
        self.static_noise = static_noise
        self.hs_o, self.hs_c = list(handlers_objs), list(handlers_cons)
        self.keys = [("obj", i) for i in range(len(self.hs_o))] + [("con", k) for k in range(len(self.hs_c))]
        self.handlers = self.hs_o + self.hs_c
        dev = self.handlers[0].device
        # everything the iteration reads must already live on the device: a host-to-device copy cannot be captured
        fitter.pareto_set = fitter.pareto_set.to(dev)
        fitter.pareto_front = fitter.pareto_front.to(dev)
        fitter.thresholds_cons = fitter.thresholds_cons.to(dev)
        self.x_tilde = torch.zeros(10, fitter.pareto_set.shape[1], dtype=torch.float64, device=dev)
        # The upstream `torch.equal(x, Z)` shortcut (quirk Q4) is a device comparison = a synchronisation, illegal
        # inside a capture.  It can only fire for an input with Z's shape (N == pareto_set_size or N == 10 rows do
        # happen): answer it HERE, once, on the host.  x-tilde is redrawn uniformly every iteration and never equals
        # Z; the Pareto set is fixed, so one comparison per model settles it (if it does equal some model's Z the
        # arithmetic changes and the iteration stays eager).
        self.x_tilde._mobo_not_z = True
        ps_host = fitter.pareto_set.detach().cpu()
        self.capturable = True
        for h in self.handlers:
            z = getattr(h.mfdgp, h.mfdgp.name_hidden_layer + "0")._Zx().detach().cpu()
            if z.shape == ps_host.shape and bool(torch.equal(z, ps_host)):
                self.capturable = False
        if self.capturable:
            fitter.pareto_set._mobo_not_z = True
        self.graphs = {}       # minibatch shapes -> (static buffers, graph, loss): the ragged last batch of an epoch
        #                        gets its own graph (the reference's DataLoader yields it like any other)

    def _fetch(self):
        out = {}
        for key, h in zip(self.keys, self.handlers):
            try:
                out[key] = next(h.iter_train_loader)
            except Exception:
                h.iter_train_loader = iter(h.train_loader)
                out[key] = next(h.iter_train_loader)
        return out

    def _hits_shortcut(self, batches):
        for key, h in zip(self.keys, self.handlers):
            if getattr(h.mfdgp, h.mfdgp.name_hidden_layer + "0")._equals_inducing(batches[key][0]):
                return True
        return False

    def _iteration(self, static, static_eps=None):
        if not self.static_noise:
            self.x_tilde.uniform_()
        loss = self.fitter.conditioned_loss(self.hs_o, self.hs_c, x_tilde=self.x_tilde, batches=static,
                                            eps=static_eps)
        loss.backward()
        self.optimizer.step()
        return loss.detach()

    def _layers(self):
        for h in self.handlers:
            m = h.mfdgp
            for i in range(m.num_hidden_layers):
                yield getattr(m, m.name_hidden_layer + str(i))

    def _capture(self, batches, eps=None):
        static = {}
        for key in self.keys:
            bufs = tuple(t.detach().clone() for t in batches[key])
            bufs[0]._mobo_not_z = True          # checked on the host for every minibatch (_hits_shortcut)
            static[key] = bufs
        static_eps = None
        if self.static_noise:
            static_eps = {key: {w: [None if e is None else e.detach().clone() for e in lst]
                                for w, lst in eps[key].items()} for key in self.keys}
        snap = self.optimizer.snapshot()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(self.warmup):
                self.optimizer.zero_grad(set_to_none=True)
                self._iteration(static, static_eps)
        torch.cuda.current_stream().wait_stream(side)
        self.optimizer.zero_grad(set_to_none=True)
        for layer in self._layers():
            layer._ops_cache = None
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            loss = self._iteration(static, static_eps)
        self.optimizer.restore(snap)    # warm-up and capture do not count as training iterations
        return static, graph, loss, static_eps

    def __call__(self, batches=None, x_tilde=None, eps=None):
        if batches is None:
            batches = self._fetch()
        if self.static_noise:
            self.x_tilde.copy_(x_tilde)
        if not self.capturable or self._hits_shortcut(batches):
            self.optimizer.zero_grad()
            loss = self.fitter.conditioned_loss(self.hs_o, self.hs_c, batches=batches, eps=eps,
                                                x_tilde=self.x_tilde if self.static_noise else None)
            loss.backward()
            self.optimizer.step()
            return loss.detach()
        shape_key = tuple(tuple(t.shape) for key in self.keys for t in batches[key])
        if shape_key not in self.graphs:
            self.graphs[shape_key] = self._capture(batches, eps)
        static, graph, loss, static_eps = self.graphs[shape_key]
        for key in self.keys:
            for dst, src in zip(static[key], batches[key]):
                dst.copy_(src)
            if static_eps is not None:
                for w, lst in static_eps[key].items():
                    for dst, src in zip(lst, eps[key][w]):
                        if dst is not None:
                            dst.copy_(src)
        graph.replay()
        for layer in self._layers():
            layer._ops_cache = None       # the cached operators belong to the graph's memory pool
        return loss


class BlackBoxMFDGPFitter():

    def __init__(self, num_fidelities, batch_size, lr_1=0.003, lr_2=0.001, num_epochs_1=5000, num_epochs_2=15000,
                 pareto_set_size=50, opt_grid_size=1000, eps=1e-8, decoupled_evals=False,
                 type_lengthscale=TL.MEDIAN, device=None, use_cuda_graph=False, concurrent_models=False):
        self.num_obj = 0
        self.num_con = 0
        self.models_uncond_trained = False
        self.mfdgp_handlers_objs = {}
        self.mfdgp_handlers_cons = {}
        self.device = device
        self.thresholds_cons = torch.tensor([], dtype=torch.double)
        self.x_train = None
        self.objs_train = torch.tensor([], dtype=torch.double)
        self.cons_train = torch.tensor([], dtype=torch.double)
        self.num_fidelities = num_fidelities
        self.batch_size = batch_size
        self.points_to_sample = batch_size
        self.lr_1, self.lr_2 = lr_1, lr_2
        self.num_epochs_1, self.num_epochs_2 = num_epochs_1, num_epochs_2
        self.pareto_set_size = pareto_set_size
        self.opt_grid_size = opt_grid_size
        self.eps = eps
        self.decoupled_evals = decoupled_evals
        self.type_lengthscale = type_lengthscale
        # one CUDA-graph launch per step instead of ~55 kernel launches: the regime of the reference's examples
        # (full batch, M = N of a few tens) is launch-latency bound
        self.use_cuda_graph = use_cuda_graph
        # the black boxes' MFDGPs are independent during unconditioned training (fitter.py:134-152 loops over them):
        # with concurrent_models their steps are enqueued round-robin on one CUDA stream each, so the latency-bound
        # kernel chains of the K models overlap on the GPU (the reference trains them one after the other; the order
        # in which the models consume torch's random stream changes, their distribution does not)
        self.concurrent_models = concurrent_models
        self.pareto_set = None
        self.pareto_front = None
        self.verbose = True

    def initialize_mfdgp(self, x_train, y_train, fidelities, blackbox_name, threshold_constraint=0.0,
                         is_constraint=False, previously_trained_model=None,
                         init_params_to_prior_and_fix_them=False, use_only_highest_fidelity=False):
        if self.x_train is None:
            self.x_train = x_train
        else:
            assert torch.equal(self.x_train, x_train), "The inputs for this new mfdgp do not match with inputs " \
                "for previous mfdgp models. This class is not currently prepared for a decoupled evaluation setting."
        handler = MFDGPHandler(x_train, y_train, fidelities, self.num_fidelities, self.batch_size,
                               type_lengthscale=self.type_lengthscale,
                               previously_trained_model=previously_trained_model,
                               init_params_to_prior_and_fix_them=init_params_to_prior_and_fix_them,
                               use_only_highest_fidelity=use_only_highest_fidelity, device=self.device)
        if is_constraint:
            self.cons_train = torch.cat((self.cons_train, y_train.cpu()), 1)
            self.mfdgp_handlers_cons[blackbox_name] = handler
            self.thresholds_cons = torch.cat((self.thresholds_cons,
                                              torch.tensor([threshold_constraint], dtype=torch.double)), 0)
            self.num_con += 1
        else:
            self.objs_train = torch.cat((self.objs_train, y_train.cpu()), 1)
            self.mfdgp_handlers_objs[blackbox_name] = handler
            self.num_obj += 1

    # ---- the ELBO step (fitter.py:156-173) ----
    @staticmethod
    def _fused_step(model, elbo):
        """The fused kernel sequence for this (model, elbo) pair, or None when its preconditions do not hold
        (only-HF models, per-layer inducing inputs); cached on the elbo object."""
        cached = getattr(elbo, "_fused_step", None)
        if cached is None:
            from ..fused import FusedELBOStep
            ok, _ = FusedELBOStep.supported(model)
            cached = FusedELBOStep(model, elbo) if ok else False
            elbo._fused_step = cached
        return cached or None

    @staticmethod
    def _graphed_step(fused, optimizer, batch_size):
        """CUDA-graph replay of (fused step + Adam) for this minibatch shape; built on first use, keyed by the
        optimiser (a new phase creates a new optimiser) and the batch size."""
        cache = fused.__dict__.setdefault("_graphs", {})
        key = (id(optimizer), batch_size)
        if key not in cache:
            from ..fused import GraphedELBOStep
            cache[key] = GraphedELBOStep(fused, optimizer, batch_size)
        return cache[key]

    @staticmethod
    def _update_model(model, elbo, optimizer, train_loader, eps=None):
        loss_iter = 0.0
        kl_iter = 0.0
        fused = BlackBoxMFDGPFitter._fused_step(model, elbo)
        graphed = fused is not None and getattr(optimizer, "capturable", False) and eps is None
        guarded = isinstance(optimizer, Adam)
        for (x_batch, y_batch, fidelities) in train_loader:
            use_fused = fused is not None and fused.applies(x_batch)
            if guarded:
                # a fused step that fails (NotPSDError / NanError upstream) must not reach the parameters: its Adam
                # update is skipped on the device; the error itself is raised at the next reporting boundary
                optimizer.skip_flag = fused.skip_flag if use_fused else None
            if graphed and use_fused:
                loss, kl = BlackBoxMFDGPFitter._graphed_step(fused, optimizer, x_batch.shape[0])(
                    x_batch, y_batch, fidelities, check_shortcut=False)   # forward, ELBO, backward AND the Adam update
                loss_iter += loss.detach().clone()
                kl_iter += kl.detach().clone()
                continue
            if use_fused:
                # forward, ELBO and backward in one enqueue; gradients are overwritten, so no zero_grad
                loss, kl = fused(x_batch, y_batch, fidelities, eps=eps, check_shortcut=False)
                optimizer.step()
                loss_iter += loss.detach().clone()
                kl_iter += kl.detach().clone()
                continue
            with settings.num_likelihood_samples(1):
                optimizer.zero_grad()
                output = model(x_batch, eps=eps)
                res = elbo(output, y_batch.T, fidelities)
                loss, kl = -res[0], res[1]
                loss.backward()
                optimizer.step()
                loss_iter += loss.detach()
                kl_iter += kl.detach()
        return loss_iter, kl_iter

    # Where one CTA per model (mobo_elbo_step_small) beats one stream + graph per model (mobo_elbo_step), measured by
    # tools/small_models_bench.py on an NVIDIA B200 at a 1000 W power limit (profiles/r03_small_models_bench.json,
    # "sweep_S1"): for every group size K = 1, 3, 6 only up to M = 16 inducing points (at M = 24 it loses for K = 1, 3)
    # and, at M = 16, up to 32 rows per model (at 64 rows it loses for K = 1, 3).
    SMALL_STEP_MAX_INDUCING = 16
    SMALL_STEP_MAX_ROWS = 32

    def _small_group(self, hs, opts):
        """The graphed single-kernel step of the models ``hs`` when it applies (SmallModelsELBOStep.supported: shared
        inducing inputs, M <= 64) and pays (at most SMALL_STEP_MAX_INDUCING inducing points and SMALL_STEP_MAX_ROWS
        rows per minibatch), and every model's loader yields the same number of batches per epoch (one replay per
        batch index covers them all); else None."""
        from ..fused import GraphedSmallModelsELBOStep, SmallModelsELBOStep
        models = [h.mfdgp for h in hs]
        ok, _ = SmallModelsELBOStep.supported(models)
        if not ok:
            return None
        nbatches = {-(-h.num_data // h.train_loader.batch_size) for h in hs}
        rows = max(min(h.num_data, h.train_loader.batch_size) for h in hs)
        inducing = max(getattr(m, m.name_hidden_layer + "0").num_inducing for m in models)
        if len(nbatches) != 1 or rows > self.SMALL_STEP_MAX_ROWS or inducing > self.SMALL_STEP_MAX_INDUCING:
            return None
        steps = [self._fused_step(h.mfdgp, h.elbo) for h in hs]
        key = tuple(id(s) for s in steps)
        cache = self.__dict__.setdefault("_small_steps", {})
        if key not in cache:
            cache[key] = SmallModelsELBOStep(models, [h.elbo for h in hs], steps=steps)
        # the graph joins each member step's cache of the graphs it is replayed in (see _graphed_step), keyed by the
        # group's optimisers: a new phase has new ones
        okey = ("small",) + tuple(id(o) for o in opts)
        graphs = steps[0].__dict__.setdefault("_graphs", {})
        if okey not in graphs:
            g = GraphedSmallModelsELBOStep(cache[key], opts)
            for s in steps:
                s.__dict__.setdefault("_graphs", {})[okey] = g
        return graphs[okey]

    @staticmethod
    def _update_small_group(group, hs, opts):
        """One epoch of every model of ``group``: per batch index one replay of the graphed small step.  A model whose
        minibatch equals its inducing inputs (quirk Q4) takes ``_update_model``'s path for that batch."""
        loss = [0.0] * len(hs)
        kl = [0.0] * len(hs)
        for batches in zip(*[h.train_loader for h in hs]):
            active = [st.applies(b[0]) for st, b in zip(group.small.steps, batches)]
            for n, (h, opt, b, a) in enumerate(zip(hs, opts, batches, active)):
                if not a:
                    l_n, k_n = BlackBoxMFDGPFitter._update_model(h.mfdgp, h.elbo, opt, [b])
                    loss[n] += l_n
                    kl[n] += k_n
            if not any(active):
                continue
            for o, st in zip(opts, group.small.steps):
                o.skip_flag = st.skip_flag
            res = group([b if a else None for b, a in zip(batches, active)], check_shortcut=False)
            for n, r in enumerate(res):
                if r is not None:
                    loss[n] += r[0].detach().clone()
                    kl[n] += r[1].detach().clone()
        return list(zip(loss, kl))

    def _train_mfdgp(self, func_update_model, fix_variational_hypers, num_epochs, lr):
        for kind, handlers in (("OBJ", self.mfdgp_handlers_objs), ("CON", self.mfdgp_handlers_cons)):
            opts = []
            for h in handlers.values():
                h.mfdgp.fix_variational_hypers(fix_variational_hypers)
                opts.append(Adam([{'params': h.mfdgp.parameters()}], lr=lr, capturable=self.use_cuda_graph))
            hs = list(handlers.values())

            def report(n, i, loss_iter, kl_iter):
                if (i % ITER_PRINT) == 0 or ((i + 1) == num_epochs):
                    # the only place the training loop synchronises: surface NotPSDError / NanError of any step
                    # since the last boundary (upstream raises inside the step)
                    self._check_status(hs[n])
                    if self.verbose:
                        print("[%s: " % kind, n, "] Epoch:", i, "/", num_epochs, ". Avg. Neg. ELBO per epoch:",
                              loss_iter.item(), "\t KL per epoch:", kl_iter.item())
                        sys.stdout.flush()

            group = None
            if self.concurrent_models and self.use_cuda_graph and func_update_model == self._update_model:
                group = self._small_group(hs, opts)
            if group is not None:
                # every model's step of one batch index in one graph replay (mobo_elbo_step_small + the K Adams)
                for i in range(num_epochs):
                    sums = self._update_small_group(group, hs, opts)
                    for n, (loss_iter, kl_iter) in enumerate(sums):
                        report(n, i, loss_iter, kl_iter)
                continue
            if self.concurrent_models and len(hs) > 1:
                cur = torch.cuda.current_stream(hs[0].device)
                streams = [torch.cuda.Stream(device=h.device) for h in hs]
                for st in streams:
                    st.wait_stream(cur)
                for i in range(num_epochs):
                    for n, (h, optimizer, st) in enumerate(zip(hs, opts, streams)):
                        with torch.cuda.stream(st):
                            loss_iter, kl_iter = func_update_model(h.mfdgp, h.elbo, optimizer, h.train_loader)
                            report(n, i, loss_iter, kl_iter)
                for st in streams:
                    cur.wait_stream(st)
                continue
            for n, (h, optimizer) in enumerate(zip(hs, opts)):
                for i in range(num_epochs):
                    loss_iter, kl_iter = func_update_model(h.mfdgp, h.elbo, optimizer, h.train_loader)
                    report(n, i, loss_iter, kl_iter)

    @staticmethod
    def _check_status(handler):
        from .. import functional as F
        fused = getattr(handler.elbo, "_fused_step", None)
        if fused:
            fused.check()
        F.check_status(handler.device)

    def train_mfdgps(self):
        self._train_mfdgp(self._update_model, fix_variational_hypers=True, num_epochs=self.num_epochs_1,
                          lr=self.lr_1)
        self._train_mfdgp(self._update_model, fix_variational_hypers=False, num_epochs=self.num_epochs_2,
                          lr=self.lr_2)
        self.models_uncond_trained = True

    def _sample_and_store_pareto_solution(self):
        """fitter.py:181-217: one function sample of the top layer per objective; constraints are re-drawn until the
        grid has a feasible point (MAX_TRIES_FOR_FEASIBLE_GRID), then the least infeasible point is accepted."""
        l_samples_objs = [h.mfdgp.sample_function_from_each_layer()[-1] for h in self.mfdgp_handlers_objs.values()]
        inputs = self.x_train
        global_optimizer = None
        for _ in range(MFDGPHandler.MAX_TRIES_FOR_FEASIBLE_GRID):
            l_samples_cons = [h.mfdgp.sample_function_from_each_layer()[-1] for h in self.mfdgp_handlers_cons.values()]
            global_optimizer = MOOP(l_samples_objs, l_samples_cons, input_dim=inputs.shape[1],
                                    grid_size=self.opt_grid_size * inputs.shape[1],
                                    pareto_set_size=self.pareto_set_size,
                                    feasible_values=-1.0 * self.thresholds_cons.cpu().numpy())
            res = global_optimizer.compute_pareto_solution_from_samples(inputs)
            if res is not None:
                self.pareto_set, self.pareto_front, self.samples_objs, self.samples_cons = res
                return res
        res = global_optimizer.compute_pareto_solution_from_samples(inputs, allow_negative_constraints=True)
        if res is not None:
            self.pareto_set, self.pareto_front, self.samples_objs, self.samples_cons = res
            return res
        raise NotFeasiblePoints("[ERROR] No feasible points were found in the constraint space! # tries: %d."
                                % MFDGPHandler.MAX_TRIES_FOR_FEASIBLE_GRID)

    def sample_and_store_pareto_solution(self):
        while True:
            try:
                return self._sample_and_store_pareto_solution()
            except NotFeasiblePoints:
                print("Not feasible solution found, trying another time!")
                sys.stdout.flush()

    # ---- theta / omega factors (fitter.py:227-243) ----
    def loss_theta_factors(self, cs_mean, cs_var, threshold):
        gamma_c_star = (cs_mean - threshold) / torch.sqrt(cs_var)
        cdf = _normal_cdf(gamma_c_star)
        return torch.sum(np.log(1.0 - self.eps) * cdf + np.log(self.eps) * (1.0 - cdf))

    def loss_omega_factors(self, fs_mean, fs_var, cs_mean, cs_var, pareto_front):
        thr = self.thresholds_cons.to(cs_mean.device)
        gamma_c = (cs_mean - thr[:, None]) / torch.sqrt(cs_var)
        gamma_f_star = (pareto_front[:, :, None] - fs_mean) / torch.sqrt(fs_var)
        prod = _prod(_normal_cdf(gamma_c), 0) * _prod(_normal_cdf(gamma_f_star), 1)
        return torch.sum(np.log(self.eps) * prod + np.log(1 - self.eps) * (1.0 - prod))

    # ---- the conditioned step (fitter.py:272-346) ----
    def conditioned_loss(self, handlers_objs, handlers_cons, x_tilde=None, batches=None, eps=None):
        """Loss of one conditioned iteration.  ``batches`` / ``eps`` (optional, for parity tests): per black box the
        minibatch ``(x, y, fid)`` and a dict ``{"batch", "pareto", "tilde"}`` of per-layer normals."""
        handlers_objs, handlers_cons = list(handlers_objs), list(handlers_cons)
        dev = handlers_objs[0].device if handlers_objs else handlers_cons[0].device
        pareto_set = self.pareto_set.to(dev)
        pareto_front = self.pareto_front.to(dev)
        thr = self.thresholds_cons.to(dev)
        if x_tilde is None:
            x_tilde = torch.rand(size=(10, pareto_set.shape[1]), device=dev).double()
        loss = 0.0

        def next_batch(h, key):
            if batches is not None:
                return batches[key]
            try:
                return next(h.iter_train_loader)
            except Exception:
                h.iter_train_loader = iter(h.train_loader)
                return next(h.iter_train_loader)

        def e(key, which):
            return None if eps is None else eps[key][which]

        # The black boxes' models are coupled only through the omega factors below: the three forwards of each of them
        # (minibatch, Pareto set, x-tilde) run on the model's own stream, forked from and joined back into the current
        # one, so their kernel chains overlap (also as parallel branches of the captured graph, and again in the
        # backward, which autograd runs on the streams of the forward).
        cur = torch.cuda.current_stream(dev)
        nmodels = len(handlers_objs) + len(handlers_cons)
        if not self.__dict__.get("_cond_streams"):
            # gradients produced on the models' streams are accumulated into parameters that live on the current one:
            # intended (autograd synchronises the streams), so the advisory warning about it is switched off
            quiet = getattr(torch.autograd.graph, "set_warn_on_accumulate_grad_stream_mismatch", None)
            if quiet is not None:
                quiet(False)
        streams = self.__dict__.setdefault("_cond_streams", [])
        while len(streams) < nmodels:
            streams.append(torch.cuda.Stream(device=dev))
        sub = self.__dict__.setdefault("_cond_substreams", [])
        while len(sub) < 2 * nmodels:
            sub.append(torch.cuda.Stream(device=dev))
        terms, fm, fv, cm, cv = [], [], [], [], []
        for n, (kind, i, h) in enumerate([("obj", i, h) for i, h in enumerate(handlers_objs)] +
                                         [("con", k, h) for k, h in enumerate(handlers_cons)]):
            key = (kind, i)
            x_batch, y_batch, fidelities = next_batch(h, key)
            st = streams[n] if nmodels > 1 else cur
            s_par, s_til = sub[2 * n], sub[2 * n + 1]
            st.wait_stream(cur)
            with torch.cuda.stream(st), settings.num_likelihood_samples(1):
                # the operator chains of the model once, then its three row passes side by side
                for l in range(h.mfdgp.num_hidden_layers):
                    getattr(h.mfdgp, h.mfdgp.name_hidden_layer + str(l)).operators()
                s_par.wait_stream(st)
                s_til.wait_stream(st)
                output = h.mfdgp(x_batch, eps=e(key, "batch"))
                t_batch = -h.elbo(output, y_batch.T, fidelities)[0] / x_batch.shape[0] * h.num_data
                with torch.cuda.stream(s_par):
                    if kind == "obj":
                        output = h.mfdgp(pareto_set, eps=e(key, "pareto"))
                        pareto_fidelities = torch.ones(size=(pareto_front.shape[0], 1), device=dev) * \
                            (h.num_fidelities - 1)
                        t_pareto = -h.elbo(output, pareto_front[:, i:(i + 1)].T, pareto_fidelities,
                                           include_kl_term=False)
                    else:
                        output = h.mfdgp(pareto_set, eps=e(key, "pareto"))[h.num_fidelities - 1]
                        t_pareto = -self.loss_theta_factors(output.mean, output.variance, thr[i])
                with torch.cuda.stream(s_til):
                    output = h.mfdgp(x_tilde, eps=e(key, "tilde"))[h.num_fidelities - 1]
                    (fm if kind == "obj" else cm).append(output.mean[None, :])
                    (fv if kind == "obj" else cv).append(output.variance[None, :])
                st.wait_stream(s_par)
                st.wait_stream(s_til)
                terms.append(t_batch + t_pareto)
        for n in range(nmodels if nmodels > 1 else 0):
            cur.wait_stream(streams[n])
        for t in terms:
            loss = loss + t
        z = torch.zeros(0, x_tilde.shape[0], dtype=torch.double, device=dev)
        loss = loss + -self.loss_omega_factors(torch.cat(fm, 0) if fm else z, torch.cat(fv, 0) if fv else z,
                                               torch.cat(cm, 0) if cm else z, torch.cat(cv, 0) if cv else z,
                                               pareto_front)
        return loss

    def _update_conditioned_models(self, handlers_objs, handlers_cons, optimizer):
        if self.use_cuda_graph and getattr(optimizer, "capturable", False):
            cache = self.__dict__.setdefault("_cond_graphs", {})
            if id(optimizer) not in cache:
                cache.clear()
                cache[id(optimizer)] = _GraphedConditionedStep(self, handlers_objs, handlers_cons, optimizer)
            return cache[id(optimizer)]()
        optimizer.zero_grad()
        if isinstance(optimizer, Adam):
            optimizer.skip_flag = None
        loss = self.conditioned_loss(handlers_objs, handlers_cons)
        loss.backward()
        optimizer.step()
        return loss.detach()

    def _train_conditioned_mfdgps(self, func_update_model, fix_variational_hypers, num_iters, lr):
        params = list()
        for h in list(self.mfdgp_handlers_objs.values()) + list(self.mfdgp_handlers_cons.values()):
            h.mfdgp.fix_variational_hypers_cond(fix_variational_hypers)
            params = params + list(h.mfdgp.parameters())
        optimizer = Adam([{'params': params}], lr=lr, capturable=self.use_cuda_graph)
        for i in range(num_iters):
            loss_iter = func_update_model(self.mfdgp_handlers_objs.values(), self.mfdgp_handlers_cons.values(),
                                          optimizer)
            if (i % ITER_PRINT) == 0 or ((i + 1) == num_iters):
                from .. import functional as F
                F.check_status()
                if not bool(torch.isfinite(loss_iter)):
                    from ..errors import NanError
                    raise NanError("NanError: the conditioned loss is not finite")
                if self.verbose:
                    print("Iter:", i, "/", num_iters, ". Neg. ELBO per iter:", loss_iter.item())
                    sys.stdout.flush()

    def train_conditioned_mfdgps(self):
        self._train_conditioned_mfdgps(self._update_conditioned_models, fix_variational_hypers=True,
                                       num_iters=self.num_epochs_2, lr=self.lr_2)
        for h in list(self.mfdgp_handlers_objs.values()) + list(self.mfdgp_handlers_cons.values()):
            h.iter_train_loader = None

    def mfdgps_to_train_mode(self):
        for h in list(self.mfdgp_handlers_objs.values()) + list(self.mfdgp_handlers_cons.values()):
            h.mfdgp.train()

    def mfdgps_to_eval_mode(self):
        """fitter.py:363-368, as written there: the objectives' models to eval(), the constraints' to train()."""
        for h in self.mfdgp_handlers_objs.values():
            h.mfdgp.eval()
        for h in self.mfdgp_handlers_cons.values():
            h.mfdgp.train()

    def copy_uncond(self):
        if self.models_uncond_trained is False:
            warnings.warn("(Warning) The mfdgp models have not been trained yet.")
        handlers = list(self.mfdgp_handlers_objs.values()) + list(self.mfdgp_handlers_cons.values())
        for h in handlers:
            h.mfdgp.eval()
            h.iter_train_loader = None
        graphs = self.__dict__.pop("_cond_graphs", None)      # captured CUDA graphs / streams do not travel through
        self.__dict__.pop("_cond_streams", None)              # deepcopy
        self.__dict__.pop("_cond_substreams", None)
        small = self.__dict__.pop("_small_steps", None)        # ctypes descriptors and graphs, like the elbos' steps
        self_copy = deepcopy(self)
        if graphs is not None:
            self._cond_graphs = graphs
        if small is not None:
            self._small_steps = small
        for h in handlers:
            h.mfdgp.train()
        for h in list(self_copy.mfdgp_handlers_objs.values()) + list(self_copy.mfdgp_handlers_cons.values()):
            h.mfdgp.train()
        return self_copy

    def get_model(self, name: str, is_constraint=False):
        if is_constraint:
            return self.mfdgp_handlers_cons[name].mfdgp
        return self.mfdgp_handlers_objs[name].mfdgp
