"""Multi-fidelity deep GP — host-side mirror of ``mobocmf/models/mfdgp.py`` (``MFDGP``, ``TL``): same constructor,
attribute names (``hidden_layer_{i}``, ``hidden_layer_likelihood_{i}``), ``forward`` / ``predict`` /
``predict_for_acquisition`` / freeze helpers, with the layer arithmetic on the sm_100a kernels.

``predict_for_acquisition`` does not materialise the S-fold tiling of the candidates (models/mfdgp.py:248): layer 0
runs on the n candidates, the upper layers on n*S rows that index their candidate (row i*S+s = point i, sample s),
which is the same arithmetic per row.
"""
from enum import Enum

import numpy as np
import torch
from torch import nn

from ..gp import GaussianLikelihood, GaussianMoments, Interval, settings
from ..layers.mfdgp_hidden_layer import MFDGPHiddenLayer
from ..layers.mfdgp_hidden_layer_only_hf import MFDGPHiddenLayer as MFDGPHiddenLayer_only_hf
from ..util.util import compute_dist, triu_indices


class TL(Enum):  # type of lengthscale initialisation (models/mfdgp.py:15-18)
    ONES = 1
    MEDIAN = 2
    CENTESIMAL = 3


class _DeepGPVariationalStrategy(object):
    """``model.variational_strategy.kl_divergence()``: sum over the layers, each counted once (quirk Q12)."""

    def __init__(self, model):
        self.model = model

    def kl_divergence(self):
        m = self.model
        return sum(getattr(m, m.name_hidden_layer + str(i))._kl_divergence() for i in range(m.num_hidden_layers))


class MFDGP(nn.Module):

    def __init__(self, x_train, y_train, fidelities, num_fidelities, type_lengthscale=TL.MEDIAN,
                 num_samples_for_acquisition=25, previously_trained_model=None, ini_inducing_using_layer_0=False,
                 use_only_highest_fidelity=False, init_params_to_prior_and_fix_them=False, num_inducing=None,
                 init_lengthscale=None):
        """Reference signature (models/mfdgp.py:22-25) plus two extensions the reference lacks (SURVEY.md §8f-1):
        ``num_inducing`` keeps only the first M training inputs as inducing inputs (the reference always uses all
        N, models/mfdgp.py:297-298) and ``init_lengthscale`` overrides the O(N^2) median heuristic."""
        super().__init__()
        self.num_inducing = num_inducing
        self._init_lengthscale_override = init_lengthscale
        hidden_layers = []
        self.init_params_to_prior_and_fix_them = init_params_to_prior_and_fix_them
        self._eval_mode = False
        self.num_samples_for_acquisition = num_samples_for_acquisition
        self.use_only_highest_fidelity = use_only_highest_fidelity
        self.ini_inducing_using_layer_0 = ini_inducing_using_layer_0
        self.input_dims = x_train.shape[-1]
        y_high_std = np.std(y_train[(fidelities == num_fidelities - 1).flatten()].cpu().numpy())

        for i in range(num_fidelities):
            previously_trained_layer = None
            if previously_trained_model is not None:
                previously_trained_layer = getattr(previously_trained_model,
                                                   previously_trained_model.name_hidden_layer + str(i))
            inducing_points, inducing_values = self.find_good_initial_inducing_points_and_values(
                x_train, y_train, fidelities, i)
            init_lengthscale = self.get_init_lengthscale(type_lengthscale,
                                                         inputs=x_train[(fidelities == i).flatten(), :])
            if i == 0:
                hidden_layers.append(MFDGPHiddenLayer(
                    input_dims=self.input_dims, num_layer=0, inducing_points=inducing_points,
                    inducing_values=inducing_values, init_lengthscale=init_lengthscale,
                    num_fidelities=num_fidelities, num_samples_for_acquisition=num_samples_for_acquisition,
                    previously_trained_layer=previously_trained_layer,
                    init_params_to_prior_and_fix_them=self.init_params_to_prior_and_fix_them))
            else:
                cls = MFDGPHiddenLayer_only_hf if use_only_highest_fidelity is True else MFDGPHiddenLayer
                hidden_layers.append(cls(
                    input_dims=self.input_dims + 1, num_layer=i, inducing_points=inducing_points,
                    inducing_values=inducing_values, num_fidelities=num_fidelities,
                    init_lengthscale=init_lengthscale, y_high_std=y_high_std,
                    num_samples_for_acquisition=num_samples_for_acquisition,
                    previously_trained_layer=previously_trained_layer,
                    init_params_to_prior_and_fix_them=self.init_params_to_prior_and_fix_them,
                    previous_layer_in_hierarchy=hidden_layers[-1]))

        self.name_hidden_layer = "hidden_layer_"
        self.name_hidden_layer_likelihood = "hidden_layer_likelihood_"
        self.name_hidden_layer_likelihood_noiseless = "hidden_layer_likelihood_noiseless_"
        self.num_hidden_layers = num_fidelities
        self.num_fidelities = num_fidelities

        for i, hidden_layer in enumerate(hidden_layers):
            y_std = np.std(y_train[(fidelities == i).flatten()].cpu().numpy())
            setattr(self, self.name_hidden_layer + str(i), hidden_layer)
            likelihood = GaussianLikelihood(noise_constraint=Interval(lower_bound=1e-8, upper_bound=0.1 * y_std))
            if i == self.num_fidelities - 1:
                likelihood.noise = 1e-2 * y_high_std
            else:
                likelihood.noise = 1e-6
            setattr(self, self.name_hidden_layer_likelihood + str(i), likelihood)

    @property
    def variational_strategy(self):
        return _DeepGPVariationalStrategy(self)

    def get_init_lengthscale(self, type_lengthscale, inputs=None):
        if self._init_lengthscale_override is not None:
            return torch.as_tensor(self._init_lengthscale_override, dtype=torch.float64)
        if type_lengthscale == TL.ONES:
            return torch.ones(self.input_dims)
        elif type_lengthscale == TL.MEDIAN:
            return self.median_lengthscale(inputs)
        elif type_lengthscale == TL.CENTESIMAL:
            return 0.01 * np.ones(self.input_dims)
        raise ValueError("Wrong type of lengthscale.")

    @staticmethod
    def median_lengthscale(inputs, literal=False, use_cuda=None):
        """``sqrt(median(dists[triu_indices(n, 1)]))`` of models/mfdgp.py:143-144 INCLUDING quirk Q2: the (2, K)
        LongTensor indexes ROWS of the distance matrix (util/util.py:27-30), so the reference takes the median of a
        (2, K, n) gather, n^2 (n - 1) values — unusable beyond a few hundred points.  Every row of the matrix occurs
        exactly n - 1 times in that gather, so the multiset is n - 1 copies of the full matrix and torch.median's
        lower-middle element is the order statistic ((n^2 (n-1) - 1) // 2) // (n - 1) of the n^2 matrix entries:
        one k-th value over n^2 numbers (on the GPU when there is one), bit-identical to the literal formula."""
        n = inputs.shape[0]
        if literal or n < 2:
            dists_x_train = compute_dist(inputs)
            return torch.sqrt(torch.median(dists_x_train[triu_indices(n, 1)]))
        x = inputs
        if use_cuda is None:
            use_cuda = torch.cuda.is_available() and n > 2048
        if use_cuda and not x.is_cuda:
            x = x.cuda()
        flat = compute_dist(x).reshape(-1)
        k = ((n * n * (n - 1) - 1) // 2) // (n - 1)
        return torch.sqrt(torch.kthvalue(flat, k + 1).values).to(inputs.device)

    def train_mode(self):
        for i in range(self.num_hidden_layers):
            getattr(self, self.name_hidden_layer + str(i)).train_mode()
        self._eval_mode = False

    def eval_mode(self):
        for i in range(self.num_hidden_layers):
            getattr(self, self.name_hidden_layer + str(i)).eval_mode()
        self._eval_mode = True

    def forward(self, inputs, max_fidelity=None, eps=None, num_samples=1):
        """models/mfdgp.py:174-196.  ``eps`` (optional): list indexed by layer of the training-mode normals
        (reference: float32 ``torch.normal`` of shape (1, B), quirk Q6).  ``num_samples`` = S > 1 (not in the
        reference, which always trains with one sample, SURVEY.md fact F4): layer 0 runs on the B rows, the upper
        layers on B*S rows (row b*S+s = point b, sample s) with independent normals per (row, layer)."""
        num_layers = self.num_hidden_layers if max_fidelity is None else max_fidelity + 1
        if num_samples > 1:
            return self._forward_multisample(inputs, num_layers, eps, num_samples)
        l_outputs = [None] * num_layers
        output_layer = None
        for i in range(num_layers):
            hidden_layer = getattr(self, self.name_hidden_layer + str(i))
            if i == 0:
                output_layer = hidden_layer(inputs)
            else:
                if self.use_only_highest_fidelity is True:
                    output_layer = output_layer.mean.reshape(1, -1) * 0.0
                output_layer = hidden_layer(inputs, output_layer, eps=None if eps is None else eps[i])
            l_outputs[i] = output_layer
        return l_outputs

    def _forward_multisample(self, inputs, num_layers, eps, S):
        B = inputs.shape[0]
        x = inputs.contiguous()
        outs = []
        layer0 = getattr(self, self.name_hidden_layer + "0")
        mu, var = layer0._moments(x)
        ns = settings.num_likelihood_samples.value_()
        outs.append(GaussianMoments(mu.unsqueeze(0).expand(ns, -1), var.unsqueeze(0).expand(ns, -1)))
        R = B
        for i in range(1, num_layers):
            layer = getattr(self, self.name_hidden_layer + str(i))
            e = None if eps is None else eps[i]
            if e is None:
                e = torch.randn(B * S, device=x.device, dtype=torch.float32)
            e = e.to(device=x.device, dtype=torch.float64).reshape(-1).contiguous()
            mu, var = layer._moments(x, mu, var, e, xrep=S, prep=(B * S) // R, eps_mod=B * S, R=B * S)
            R = B * S
            d = GaussianMoments(mu, var)
            d.samples_per_point = S
            outs.append(d)
        return outs

    def fix_variational_hypers(self, value):
        for i in range(self.num_hidden_layers):
            getattr(self, self.name_hidden_layer_likelihood + str(i)).raw_noise.requires_grad = not value
        for i in range(self.num_hidden_layers):
            hidden_layer = getattr(self, self.name_hidden_layer + str(i))
            hidden_layer.variational_strategy._variational_distribution.chol_variational_covar.requires_grad = \
                not value

    def fix_variational_hypers_cond(self, value):
        for i in range(self.num_hidden_layers):
            getattr(self, self.name_hidden_layer_likelihood + str(i)).raw_noise.requires_grad = not value
        for i in range(self.num_hidden_layers):
            hidden_layer = getattr(self, self.name_hidden_layer + str(i))
            for (name, param) in hidden_layer.covar_module.named_parameters():
                param.requires_grad = not value

    def predict(self, test_x, fidelity_layer=0):
        assert fidelity_layer >= 0 and fidelity_layer < self.num_fidelities
        likelihood = getattr(self, self.name_hidden_layer_likelihood + str(fidelity_layer))
        preds = likelihood(self(test_x, max_fidelity=fidelity_layer)[fidelity_layer])
        return preds.mean, preds.variance

    def predict_for_acquisition(self, test_x, fidelity_layer=0):
        """models/mfdgp.py:237-262: S fixed normals per layer, moment matching over the S samples."""
        if len(test_x.shape) > 2:
            assert test_x.shape[1] == 1
            test_x = test_x[:, 0, :]
        assert fidelity_layer >= 0 and fidelity_layer < self.num_fidelities
        S = self.num_samples_for_acquisition
        n = test_x.shape[0]
        x = test_x.contiguous()
        if self._fused_acquisition_applies(x):
            return self._predict_for_acquisition_fused(x, fidelity_layer)
        self.eval_mode()
        layer0 = getattr(self, self.name_hidden_layer + "0")
        mu, var = layer0._moments(x)                                    # identical for the S copies of a point
        R = n
        for i in range(1, fidelity_layer + 1):
            layer = getattr(self, self.name_hidden_layer + str(i))
            smp = layer._samples_on(x.device)
            if self.use_only_highest_fidelity is True:
                mu, var = layer._moments(x, f_direct=torch.zeros(n * S, dtype=x.dtype, device=x.device), xrep=S,
                                         R=n * S)
            else:
                mu, var = layer._moments(x, mu, var, smp, xrep=S, prep=(n * S) // R, eps_mod=S, R=n * S)
            R = n * S
        self.train_mode()
        noise = getattr(self, self.name_hidden_layer_likelihood + str(fidelity_layer)).noise.reshape(())
        vars_tilde = GaussianMoments(mu, var + noise).variance
        if R == n:                                                      # fidelity 0: the S copies coincide
            mus_tilde = mu.unsqueeze(1).expand(n, S)
            vars_tilde = vars_tilde.unsqueeze(1).expand(n, S)
        else:
            mus_tilde = mu.reshape(n, S)
            vars_tilde = vars_tilde.reshape(n, S)
        mus = torch.mean(mus_tilde, 1)
        second_moment = torch.mean(vars_tilde + mus_tilde ** 2, 1)
        return mus, second_moment - mus ** 2

    # ---- fused acquisition chain (mobo_acq_moments, backward mobo_acq_moments_bwd): one enqueue per model and chunk ----
    ACQ_CHUNK = 1 << 18      # candidates per enqueue (bounds the n * S scratch)
    # candidates per backward enqueue.  The backward recomputes the chunk's forward and keeps t and u of every row of
    # every layer: about (2 MP + 2 + d)(1 + fidelity S) + (MP + 3) S doubles per candidate, 264 KB at M = 256, S = 25,
    # fidelity 2 (C5), so 4096 candidates take 1.08 GB of work, whatever the total n (more layers take more per
    # candidate).  A multiple of 32, so that every chunk starts its rows on the same tile and warp-group boundaries as
    # one unchunked call: dX does not depend on the chunking.
    ACQ_GRAD_CHUNK = 4096

    def clip_inducing_values(self, x_0, x_1, y_1):
        """y_1 at the point of x_1 nearest to each row of x_0 (models/mfdgp.py:125-135)."""
        return y_1[torch.argmin(torch.cdist(x_0, x_1), dim=1)]

    # ---- function samples of every layer (models/mfdgp.py:264-288) ----
    def sample_function_from_each_layer(self, nFeatures=500):
        result, last = [], None
        for i in range(self.num_hidden_layers):
            last = getattr(self, self.name_hidden_layer + str(i)).sample_from_posterior(self.input_dims, last,
                                                                                        nFeatures=nFeatures)
            result.append(last)
        return result

    def sample_function_from_prior_each_layer(self, nFeatures=500):
        result, last = [], None
        for i in range(self.num_hidden_layers):
            last = getattr(self, self.name_hidden_layer + str(i)).sample_from_prior(self.input_dims, last,
                                                                                    nFeatures=nFeatures)
            result.append(last)
        return result

    def _fused_acquisition_applies(self, x):
        if self.training or self.use_only_highest_fidelity is True or not x.is_cuda or x.dtype != torch.float64:
            return False
        layers = [getattr(self, self.name_hidden_layer + str(i)) for i in range(self.num_hidden_layers)]
        for lay in layers[1:]:
            lay._propagated_inducing_column()
            if not lay._dev_cache.get("shared", False):
                return False
        return True

    def _predict_for_acquisition_fused(self, x, fidelity_layer):
        from .. import functional as F
        layers = [getattr(self, self.name_hidden_layer + str(i)) for i in range(fidelity_layer + 1)]
        with torch.no_grad():
            trip = [lay.operators() for lay in layers]
            ops = [t[0].detach() for t in trip]
            theta = [t[1].detach().contiguous() for t in trip]
            zf = [None if t[2] is None else t[2].detach().contiguous() for t in trip]
            smp = [None] + [lay._samples_on(x.device) for lay in layers[1:]]
            lik = getattr(self, self.name_hidden_layer_likelihood + str(fidelity_layer))
            c = lik.noise_covar.raw_noise_constraint
            key = ("noise_bounds", fidelity_layer)
            if key not in layers[0]._dev_cache:
                layers[0]._dev_cache[key] = (float(c.lower_bound), float(c.upper_bound))
            lo, hi = layers[0]._dev_cache[key]
        chain = F.AcqChain(fidelity_layer, layers[0].num_inducing, self.num_samples_for_acquisition, layers[0]._Zx(),
                           zf, theta, ops, smp, lo, hi)
        # with X.requires_grad, differentiable with respect to X and the likelihood's raw_noise (the one parameter the
        # eval-mode chain does not hold constant, as on the composable path)
        return F.acq_moments(chain, x, lik.noise_covar.raw_noise, self.ACQ_CHUNK, self.ACQ_GRAD_CHUNK)

    def find_good_initial_inducing_points_and_values(self, x_train, y_train, fidelities, layer):
        """models/mfdgp.py:290-317, vectorised: nearest same-fidelity neighbour by the reference's expansion
        ``|a|^2 - 2 a.b + |b|^2`` (first minimum wins, like argmin); float32 values (quirk Q1)."""
        sel = fidelities[:, 0] == layer
        inducing_points = x_train[sel, :] if self.use_only_highest_fidelity is True else x_train
        if self.num_inducing is not None:
            inducing_points = inducing_points[:self.num_inducing]
        xs, ys = x_train[sel, :], y_train[sel, :]
        xs2 = (xs ** 2).sum(1, keepdim=True)
        to_sel = []
        for a in range(0, inducing_points.shape[0], 4096):        # chunked: the N_l x M distance block stays small
            ip = inducing_points[a:a + 4096]
            d = xs2 - 2.0 * xs.mm(ip.T) + (ip ** 2).sum(1)[None, :]
            to_sel.append(torch.argmin(d, dim=0))
        to_sel = torch.cat(to_sel)
        inducing_values = ys[to_sel, 0].to(torch.float32)
        if layer != 0:
            inducing_points = torch.cat((inducing_points, inducing_values[:, None]), 1)
        return inducing_points, inducing_values
