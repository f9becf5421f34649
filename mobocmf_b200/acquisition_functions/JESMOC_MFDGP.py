"""JES acquisition over MFDGPs — mirror of ``mobocmf/acquisition_functions/JESMOC_MFDGP.py``
(``_JES_MFDGP``, ``JESMOC_MFDGP``).  BoTorch is not a dependency: ``_JES_MFDGP`` keeps BoTorch's contract
(``X (b, 1, d) -> (b,)``, differentiable w.r.t. X) and the multi-start optimiser lives in
``mobocmf_b200.util.optimize``."""
import torch
from torch import Tensor

from ..gp import settings
from ..models.mfdgp import MFDGP


class _JES_MFDGP(torch.nn.Module):
    def __init__(self, fidelity: int, mfdgp_uncond: MFDGP, mfdgp_cond: MFDGP, model=None) -> None:
        assert model is None
        super().__init__()
        self.fidelity = fidelity
        self.mfdgp_uncond = mfdgp_uncond
        self.mfdgp_cond = mfdgp_cond

    def forward(self, X: Tensor) -> Tensor:
        """0.5 * clamp(log v_uncond - log v_cond, 0)  (acquisition_functions/JESMOC_MFDGP.py:38-52)."""
        self.mfdgp_uncond.eval()
        with settings.num_likelihood_samples(1):
            _, pred_variances_uncond = self.mfdgp_uncond.predict_for_acquisition(X, self.fidelity)
        self.mfdgp_uncond.train()
        self.mfdgp_cond.eval()
        with settings.num_likelihood_samples(1):
            _, pred_variances_cond = self.mfdgp_cond.predict_for_acquisition(X, self.fidelity)
        self.mfdgp_cond.train()
        # with X.requires_grad the variances carry a graph and the JES term is torch arithmetic over two n-vectors; on
        # the fused chain that graph holds X, not the chain's rows (its backward recomputes them, mobo_acq_moments_bwd)
        if not (pred_variances_uncond.requires_grad or pred_variances_cond.requires_grad) and \
                pred_variances_uncond.is_cuda:
            from .. import _lib
            out = torch.empty_like(pred_variances_uncond)
            _lib.check(_lib.load().mobo_jes(_lib.ptr(pred_variances_uncond.contiguous()),
                                            _lib.ptr(pred_variances_cond.contiguous()), out.numel(), 0,
                                            _lib.ptr(out), _lib.stream_ptr()), "mobo_jes")
            return out
        return 0.5 * torch.clamp(torch.log(pred_variances_uncond) - torch.log(pred_variances_cond), min=0.0)


class JESMOC_MFDGP():
    def __init__(self, model, num_fidelities: int = 1, model_cond=None, standard_bounds=None,
                 eval_highest_fidelity: bool = False) -> None:
        self.standard_bounds = standard_bounds
        self.eval_highest_fidelity = eval_highest_fidelity
        self.blackbox_mfdgp_fitter_uncond = model.copy_uncond()
        if model_cond is None:
            # acquisition_functions/JESMOC_MFDGP.py:73-77: one Pareto-set sample (RFF function samples + MOOP, on the
            # GPU), then the conditioned training.  A Pareto set already stored on the fitter (tests, replays of a
            # given sample) is kept instead of drawing a new one.
            if getattr(model, "pareto_set", None) is None:
                self.pareto_set, self.pareto_front, self.samples_objs, self.samples_cons = \
                    model.sample_and_store_pareto_solution()
            else:
                self.pareto_set, self.pareto_front = model.pareto_set, model.pareto_front
            model.train_conditioned_mfdgps()
            self.blackbox_mfdgp_fitter_cond = model
        else:
            self.pareto_set = model_cond.pareto_set
            self.pareto_front = model_cond.pareto_front
            self.blackbox_mfdgp_fitter_cond = model_cond
        self.num_fidelities = num_fidelities
        self.objectives = {}
        self.constraints = {}
        self.costs_blackboxes = {}
        for n_f in range(0, num_fidelities):
            self.objectives[n_f] = {}
            self.constraints[n_f] = {}
            self.costs_blackboxes[n_f] = {}
            self.costs_blackboxes[n_f]["total"] = 0.0

    def add_blackbox(self, fidelity: int, blackbox_name: str, cost_evaluation: float = 1.0, is_constraint=False):
        mfdgp_uncond = self.blackbox_mfdgp_fitter_uncond.get_model(blackbox_name, is_constraint=is_constraint)
        mfdgp_cond = self.blackbox_mfdgp_fitter_cond.get_model(blackbox_name, is_constraint=is_constraint)
        jes_mfdgp = _JES_MFDGP(fidelity, mfdgp_uncond, mfdgp_cond)
        if is_constraint:
            self.constraints[fidelity][blackbox_name] = jes_mfdgp
        else:
            self.objectives[fidelity][blackbox_name] = jes_mfdgp
        self.costs_blackboxes[fidelity]["total"] += cost_evaluation
        self.costs_blackboxes[fidelity][blackbox_name] = cost_evaluation
        return jes_mfdgp

    def decoupled_acq(self, X: Tensor, fidelity: int, blackbox_name: str, is_constraint=True) -> Tensor:
        if is_constraint:
            return self.constraints[fidelity][blackbox_name](X.double())
        return self.objectives[fidelity][blackbox_name](X.double())

    def coupled_acq(self, X: Tensor, fidelity: int, float32_accumulator: bool = True) -> Tensor:
        """Sum over objectives and constraints.  The reference accumulates into a float32 tensor in place
        (acquisition_functions/JESMOC_MFDGP.py:127-133, quirk Q8); pass ``float32_accumulator=False`` for fp64."""
        acq = torch.zeros(size=(X.shape[0],), device=X.device,
                          dtype=torch.float32 if float32_accumulator else torch.float64)

        def add(acq, term):
            # `acq(float32) += term(float64)` in place: torch computes the sum in the promoted type (fp64) and rounds
            # the RESULT to the accumulator's type once - not round(term) + acq in fp32
            return (acq.double() + term).to(acq.dtype)

        for name_obj, obj in self.objectives[fidelity].items():
            acq = add(acq, obj(X.double()))
        for name_con, con in self.constraints[fidelity].items():
            acq = add(acq, con(X.double()))
        return acq

    def _optimize(self, fidelities):
        """optimize_acqf (acquisition_functions/JESMOC_MFDGP.py:142-143,159-160) of the coupled acquisition of every
        fidelity in ``fidelities`` in ONE multi-start run: all restarts of all fidelities form one batch per L-BFGS
        iteration, whose value-and-gradient evaluation is replayed from a CUDA graph (util/optimize.py)."""
        from ..util.optimize import optimize_acqf_multi
        fns = [(lambda x, f=f: self.coupled_acq(x, fidelity=f)) for f in fidelities]
        out, self.last_optimize_info = optimize_acqf_multi(fns, bounds=self.standard_bounds, q=1, num_restarts=5,
                                                           raw_samples=200, options={"maxiter": 200},
                                                           return_info=True)
        from .. import functional
        functional.check_status()       # a failed operator chain during the run surfaces here (one synchronisation)
        return out

    def _get_nextpoint_coupled_highest_fidelity(self, iteration=None, verbose=False):
        if verbose:
            assert (iteration is not None)
        fidelity_to_evaluate = self.num_fidelities - 1
        (current_candidate, current_value), = self._optimize([self.num_fidelities - 1])
        current_value_weighted = current_value / self.costs_blackboxes[0]["total"]
        nextpoint = current_candidate[0, :]
        if verbose:
            print("Iter:", iteration, "Acquisition: " + str(current_value_weighted.cpu().numpy()) +
                  " Evaluating fidelity", fidelity_to_evaluate, "at", nextpoint.cpu().numpy())
        return nextpoint, fidelity_to_evaluate

    def _get_nextpoint_coupled(self, iteration=None, verbose=False):
        if verbose:
            assert (iteration is not None)
        current_value_weighted = 0.0
        results = self._optimize(list(range(self.num_fidelities)))      # the reference loops over the fidelities
        for fidelity, (new_candidate, new_values) in enumerate(results):
            new_values_weighted = new_values / self.costs_blackboxes[fidelity]["total"]
            if (fidelity == 0) or (current_value_weighted < new_values_weighted):
                fidelity_to_evaluate = fidelity
                current_value_weighted = new_values_weighted
                current_candidate = new_candidate
        nextpoint = current_candidate[0, :]
        if verbose:
            print("Iter:", iteration, "Acquisition: " + str(
                current_value_weighted.cpu().numpy() * self.costs_blackboxes[fidelity_to_evaluate]["total"]) +
                " Evaluating fidelity", fidelity_to_evaluate, "at", nextpoint.cpu().numpy())
        return nextpoint, fidelity_to_evaluate

    def get_nextpoint_coupled(self, iteration=None, verbose=False):
        if self.eval_highest_fidelity:
            return self._get_nextpoint_coupled_highest_fidelity(iteration=iteration, verbose=verbose)
        return self._get_nextpoint_coupled(iteration=iteration, verbose=verbose)


def jes_sweep(X: Tensor, fidelity: int, blackboxes, chunk: int = 1 << 17) -> Tensor:
    """Coupled JES acquisition averaged over P Pareto-set samples (BASELINE.json configs[4]; the reference conditions on
    ONE sample, acquisition_functions/JESMOC_MFDGP.py:73-77, so P > 1 is the average of P single-sample acquisitions,
    SURVEY.md fact F5):

        acq(x) = 1/P sum_p sum_k 1/2 max(0, log v_u,k(x) - log v_c,k,p(x))

    ``blackboxes``: one ``(uncond MFDGP, [cond MFDGP of Pareto sample p, ...])`` pair per objective / constraint.
    X: (n, d) or (n, 1, d) fp64 CUDA.  Without gradients every model chain is ONE enqueue of the fused acquisition
    kernels (``mobo_acq_moments`` + ``mobo_jes``), candidates in chunks of ``chunk`` that bound the n * S scratch.
    With ``X.requires_grad`` the same fused chain is differentiable (what optimize_acqf consumes): its backward
    recomputes each model's rows in chunks of ``MFDGP.ACQ_GRAD_CHUNK`` candidates (``mobo_acq_moments_bwd``), so a
    chain keeps O(n) memory, a few doubles per candidate, between the forward and the backward.
    Candidates are independent: shard X across GPUs with ``util.distributed.shard_bounds``, no collective."""
    from .. import _lib
    if X.dim() > 2:
        assert X.shape[1] == 1
        X = X[:, 0, :]
    n = X.shape[0]
    P = len(blackboxes[0][1])
    want_grad = torch.is_grad_enabled() and X.requires_grad
    if want_grad:
        total = torch.zeros(n, dtype=torch.float64, device=X.device)
        for unc, conds in blackboxes:
            unc.eval()
            _, vu = unc.predict_for_acquisition(X, fidelity)
            unc.train()
            lvu = torch.log(vu)
            for c in conds:
                c.eval()
                _, vc = c.predict_for_acquisition(X, fidelity)
                c.train()
                total = total + 0.5 * torch.clamp(lvu - torch.log(vc), min=0.0)
        return total / P
    lib = _lib.load()
    out = torch.zeros(n, dtype=torch.float64, device=X.device)
    with torch.no_grad():
        for a in range(0, n, chunk):
            xa = X[a:a + chunk].contiguous()
            oa = out[a:a + chunk]
            for unc, conds in blackboxes:
                unc.eval()
                _, vu = unc.predict_for_acquisition(xa, fidelity)
                unc.train()
                for c in conds:
                    c.eval()
                    _, vc = c.predict_for_acquisition(xa, fidelity)
                    c.train()
                    _lib.check(lib.mobo_jes(_lib.ptr(vu), _lib.ptr(vc), xa.shape[0], 1, _lib.ptr(oa),
                                            _lib.stream_ptr()), "mobo_jes")
        out.div_(P)
    return out
