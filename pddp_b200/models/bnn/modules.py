"""MC-dropout Bayesian neural network dynamics (mirror of pddp/models/bnn/modules.py).

The module tree is the reference's (`model.model` is a BSequential of fc_0, drop_0, nonlin_0, fc_1, drop_1,
nonlin_1, fc_out; dropout modules hold `rate`, `reg`, `noise`, CDropout additionally `logit_p`, `temperature`,
`concrete_noise`), so state dicts and attribute accesses carry over.  None of the arithmetic runs in PyTorch:

* eval-mode forward (particles -> MLP -> moment matching, modules.py:200-264, 287-386) is `pddp_linearize_bnn` /
  `pddp_rollout_bnn`, fed by `descriptor()` (weights, the persistent [P, H] masks and eps_in as data);
* training (`fit`, modules.py:131-198 with the regulariser of modules.py:434-447, 517-530 and the likelihood of
  losses.py:20-38) is `pddp_bnn_train`: forward, backward and the Adam(amsgrad) update of every step on the device.
"""
import ctypes as C
import math
from collections import OrderedDict

import torch
from torch.nn import Parameter

from ... import _lib
from ...solver import BNNDynamics
from ...utils.angular import augment_state, infer_augmented_state_size
from ..base import DynamicsModel, geometry_of
from .losses import gaussian_log_likelihood


class BDropout(torch.nn.Module):
    """Binary dropout with a persistent mask.  ref: pddp/models/bnn/modules.py:413-491"""

    def __init__(self, rate=0.1, reg=1.0, **kwargs):
        super().__init__()
        self.register_buffer("rate", torch.tensor(float(rate)))
        self.p = 1 - self.rate
        self.register_buffer("reg", torch.tensor(float(reg)))
        self.register_buffer("noise", torch.bernoulli(self.p))

    def regularization(self, weight, bias):
        """reg * (p * sum(W^2) + sum(b^2)) for the layer that FOLLOWS the dropout.  ref: modules.py:434-447"""
        self.p = 1 - self.rate
        weight_reg = self.p * (weight ** 2).sum()
        bias_reg = (bias ** 2).sum() if bias is not None else 0
        return self.reg * (weight_reg + bias_reg)

    def resample(self, generator=None):
        """ref: modules.py:449-451"""
        self._update_noise(self.noise, generator)

    def _update_noise(self, x, generator=None):
        self.p = 1 - self.rate
        self.noise.data = torch.bernoulli(self.p.expand(x.shape), generator=generator)

    def ensure(self, P, H, generator=None):
        """Eval-mode mask for P particles (drawn when the stored one has another shape, modules.py:476-478)."""
        if tuple(self.noise.shape) != (P, H):
            self._update_noise(torch.empty(P, H), generator)
        return self.mask

    @property
    def mask(self):
        return self.noise

    @mask.setter
    def mask(self, value):
        self.noise.data = value

    def forward(self, x, **kwargs):
        raise NotImplementedError("pddp_b200: dropout masks are applied inside the CUDA kernels (model(z, u, i) / "
                                  "model.fit); there is no PyTorch forward")

    def extra_repr(self):
        return "rate={}".format(self.rate)


class CDropout(BDropout):
    """Concrete dropout.  Eval mask = sigmoid((logit_p + log r - log(1-r)) / temperature) for the stored uniform
    noise r, computed when first needed and KEPT: `resample()` redraws r but the effective eval mask only changes
    when its shape does, or after training (SURVEY quirk 10).  ref: pddp/models/bnn/modules.py:494-590"""

    def __init__(self, temperature=0.1, rate=0.5, reg=1.0, **kwargs):
        super().__init__(rate, reg, **kwargs)
        self.temperature = Parameter(torch.tensor(float(temperature)), requires_grad=False)
        self.logit_p = Parameter(-torch.log(self.p.reciprocal() - 1.0))
        self.concrete_noise = None

    def regularization(self, weight, bias):
        """ref: modules.py:517-530.  The reference assigns p.data = sigmoid(logit_p) and then calls
        BDropout.regularization, whose first statement rebinds self.p = 1 - self.rate: the regulariser (and its
        entropy term) is always evaluated at the INITIAL keep-probability and no gradient reaches logit_p."""
        reg = super().regularization(weight, bias)
        return reg - (-(1 - self.p) * (1 - self.p).log() - self.p * self.p.log())

    def _update_noise(self, x, generator=None):
        self.noise.data = torch.rand(x.shape, generator=generator)

    def _update_concrete_noise(self, noise):
        """ref: modules.py:540-548"""
        lp = self.logit_p.detach().to(noise.device)
        self.concrete_noise = ((lp + noise.log() - (1 - noise).log()) / self.temperature.detach().to(noise.device)).sigmoid()

    def ensure(self, P, H, generator=None):
        if self.concrete_noise is None or tuple(self.concrete_noise.shape) != (P, H):
            self._update_noise(torch.empty(P, H), generator)
            self._update_concrete_noise(self.noise)
        return self.concrete_noise

    @property
    def mask(self):
        return self.concrete_noise

    @mask.setter
    def mask(self, value):
        self.concrete_noise = value

    def extra_repr(self):
        return "rate={}, temperature={}, regularizer_scale={}".format(1 - self.logit_p.sigmoid(), self.temperature,
                                                                       self.reg)


class BSequential(torch.nn.Sequential):
    """ref: pddp/models/bnn/modules.py:740-789"""

    def resample(self, generator=None):
        for child in self.children():
            if isinstance(child, BDropout):
                child.resample(generator)

    def regularization(self):
        """Sum over dropout layers of their regulariser on the NEXT layer with weights.  ref: modules.py:749-766"""
        reg = 0
        children = list(self._modules.values())
        for i, child in enumerate(children):
            if isinstance(child, BDropout):
                for nxt in children[i:]:
                    if hasattr(nxt, "weight") and hasattr(nxt, "bias"):
                        reg = reg + child.regularization(nxt.weight, nxt.bias)
                        break
        return reg

    def forward(self, x, resample=False, **kwargs):
        raise NotImplementedError("pddp_b200: the network is evaluated by the CUDA kernels (model(z, u, i) in eval "
                                  "mode, model.fit for training); there is no PyTorch forward")


def bayesian_model(in_features, out_features, hidden_features, nonlin=torch.nn.ReLU, output_nonlin=None,
                   weight_initializer=None, bias_initializer=None, initial_p=0.5, dropout_layers=CDropout,
                   input_dropout=None):
    """ref: pddp/models/bnn/modules.py:792-864: fc_i -> drop_i -> nonlin_i ..., fc_out; Xavier-normal weights with
    the ReLU gain, biases U(-0.1, 0.1).  The kernels implement ReLU hidden layers with a dropout after each one."""
    if nonlin is not torch.nn.ReLU or output_nonlin is not None or input_dropout is not None:
        raise NotImplementedError("pddp_b200: the BNN kernels implement ReLU hidden layers, a linear output layer and "
                                  "no input dropout")
    if not isinstance(dropout_layers, (list, tuple)):
        dropout_layers = [dropout_layers] * len(hidden_features)
    dims = [in_features] + list(hidden_features)
    modules = OrderedDict()
    for i, (din, dout) in enumerate(zip(dims[:-1], dims[1:])):
        drop = dropout_layers[i]
        if isinstance(drop, type):
            drop = drop(rate=initial_p)
        if not isinstance(drop, BDropout) or type(drop) not in (BDropout, CDropout):
            raise NotImplementedError("pddp_b200: hidden layers need a BDropout or CDropout (TLNDropout is not built)")
        modules["fc_%d" % i] = torch.nn.Linear(din, dout)
        modules["drop_%d" % i] = drop
        modules["nonlin_%d" % i] = nonlin()
    modules["fc_out"] = torch.nn.Linear(dims[-1], out_features)
    net = BSequential(modules)
    for m in net.modules():
        if isinstance(m, torch.nn.Linear):
            if weight_initializer is None:
                torch.nn.init.xavier_normal_(m.weight, gain=torch.nn.init.calculate_gain("relu"))
            else:
                weight_initializer(m.weight)
            if bias_initializer is None:
                torch.nn.init.uniform_(m.bias, -0.1, 0.1)
            else:
                bias_initializer(m.bias)
    return net


class TrainConfig(C.Structure):
    """include/pddp_b200.h: pddp_bnn_train_config"""
    _fields_ = [(n, C.c_int32) for n in ("dtype", "K0", "H0", "H1", "D", "n_data", "batch", "n_iter", "dropout")] + [
        (n, C.c_double) for n in ("lr", "beta1", "beta2", "eps", "reg_scale", "temperature", "reg0", "reg1", "rate0",
                                  "rate1")] + [("seed", C.c_uint64)]


def _standardised(P, D, generator=None):
    eps = torch.randn(P, D, generator=generator)
    return (eps - eps.mean(0)) / eps.std(0)                                  # ref: modules.py:321-329


def bnn_dynamics_model_factory(state_size, action_size, hidden_features, angular_indices=None,
                               non_angular_indices=None, constrain_min=None, constrain_max=None, particles=False,
                               **kwargs):
    """ref: pddp/models/bnn/modules.py:44-391.  Returns a BNNDynamicsModel class."""
    if constrain_min is not None or constrain_max is not None or particles:
        raise NotImplementedError("pddp_b200: bnn_dynamics_model_factory(constrain_min / constrain_max / particles) "
                                  "is not built (the reference squashes U through constrain() in forward and fit, "
                                  "modules.py:118-121,162,227; the kernels do not)")
    if len(hidden_features) != 2:
        raise NotImplementedError("pddp_b200: BNN kernels need two hidden layers")
    ang = [] if angular_indices is None else [int(i) for i in angular_indices]
    non = [i for i in range(state_size) if i not in ang]
    geo = geometry_of(state_size, ang)
    nu = _lib.GEO_INFO[geo][1]
    if action_size != nu:
        raise NotImplementedError("pddp_b200: the BNN kernels of this state geometry (D=%d, angles %s) take action_size "
                                  "%d; got %d" % (state_size, tuple(ang), nu, action_size))
    DA = infer_augmented_state_size(ang, non)
    _state_size, _ang = state_size, ang

    class BNNDynamicsModel(DynamicsModel):
        state_size = _state_size
        action_size = nu
        angular_indices = torch.tensor(_ang).long()
        non_angular_indices = torch.tensor(non).long()
        is_bnn = True

        def __init__(self, n_particles=100):
            super().__init__()
            self.model = bayesian_model(DA + nu, 2 * _state_size, list(hidden_features), **kwargs)
            self.n_particles = n_particles
            for n, v in (("X_mean", 0.0), ("X_std", 1.0), ("X_std_inv", 1.0), ("dX_mean", 0.0), ("dX_std", 1.0),
                         ("dX_std_inv", 1.0)):
                self.register_buffer(n, torch.tensor(v))                        # ref: modules.py:93-98
            self.eps_in = {}
            self.eps_out = {}
            self._version = 0            # bumped whenever weights / masks / noise change: device copies are rebuilt

        def _dropouts(self):
            return [self.model.drop_0, self.model.drop_1]

        def resample(self, generator=None):
            """ref: modules.py:281-285, 117-119: forget eps_in / eps_out (redrawn on first use) and resample the
            dropout noise.  For CDropout the effective eval mask survives this (SURVEY quirk 10)."""
            self.eps_in = {}
            self.eps_out = {}
            self.model.resample(generator)
            self._version += 1

        def load_reference(self, ref_model):
            """Copies weights, normalisation buffers, the dropout masks and every eps_in / eps_out a reference
            BNNDynamicsModel object currently holds (bit-exact mask / particle indexing)."""
            for name in ("fc_0", "fc_1", "fc_out"):
                src, dst = getattr(ref_model.model, name), getattr(self.model, name)
                dst.weight.data.copy_(src.weight.data)
                dst.bias.data.copy_(src.bias.data)
            for li, drop in enumerate(self._dropouts()):
                src = getattr(ref_model.model, "drop_%d" % li)
                drop.noise.data = src.noise.detach().clone()
                if isinstance(drop, CDropout):
                    drop.logit_p.data.copy_(src.logit_p.data)
                    drop.concrete_noise = None if src.concrete_noise is None else src.concrete_noise.detach().clone()
            self.eps_in = {int(i): e.detach().clone() for i, e in ref_model.eps_in.items()}
            self.eps_out = {int(i): e.detach().clone() for i, e in getattr(ref_model, "eps_out", {}).items()}
            if 0 in self.eps_in:
                self.n_particles = self.eps_in[0].shape[0]
            for n in ("X_mean", "X_std", "X_std_inv", "dX_mean", "dX_std", "dX_std_inv"):
                setattr(self, n, getattr(ref_model, n).detach().clone())
            self._version += 1
            return self

        # ------------------------------------------------------------------ training on the device
        def flat_parameters(self, dtype=None, device=None):
            """[W0 | b0 | W1 | b1 | W2 | b2 | logit_p0 | logit_p1] -- the layout pddp_bnn_train updates in place."""
            m = self.model
            parts = [m.fc_0.weight, m.fc_0.bias, m.fc_1.weight, m.fc_1.bias, m.fc_out.weight, m.fc_out.bias]
            parts += [d.logit_p if isinstance(d, CDropout) else torch.zeros(()) for d in self._dropouts()]
            return torch.cat([p.detach().reshape(-1).to(dtype=dtype or p.dtype, device=device or p.device) for p in parts])

        def _store_flat(self, flat):
            m = self.model
            o = 0
            for p in (m.fc_0.weight, m.fc_0.bias, m.fc_1.weight, m.fc_1.bias, m.fc_out.weight, m.fc_out.bias):
                p.data.copy_(flat[o:o + p.numel()].reshape(p.shape))
                o += p.numel()
            for d in self._dropouts():
                if isinstance(d, CDropout):
                    d.logit_p.data.copy_(flat[o])
                o += 1

        def fit(self, X, U, dX, n_iter=500, batch_size=128, reg_scale=1.0, learning_rate=1e-4,
                likelihood=gaussian_log_likelihood, resample=True, normalize=True, quiet=False, batch_indices=None,
                noise=None, seed=None, return_diagnostics=False, **kw):
            """ref: modules.py:131-198.  n_iter steps of Adam(amsgrad) on
                -gaussian_log_likelihood(dX, mean, exp(log_std)).mean() + reg_scale * regularization() / N
            with a fresh concrete / Bernoulli mask per (row, unit) at every step, all on the GPU
            (`pddp_bnn_train`).  batch_indices [n_iter, batch] (int, -1 = empty slot) and noise
            [n_iter, batch, H0 + H1] (uniforms) replace the shuffled mini-batches / the device RNG when given
            (parity tests against the reference's training step)."""
            if likelihood is not gaussian_log_likelihood or not resample:
                raise NotImplementedError("pddp_b200: BNN training implements the reference's defaults "
                                          "(gaussian_log_likelihood, resample=True)")
            dev = next((t.device for t in (X, U, dX, self.model.fc_0.weight) if t.is_cuda), None)
            if dev is None:
                if not torch.cuda.is_available():
                    raise RuntimeError("pddp_b200: BNN training runs on a CUDA device (no CPU fallback)")
                dev = torch.device("cuda", torch.cuda.current_device())
            dtype = self.model.fc_0.weight.dtype
            X_ = torch.cat([augment_state(X.detach(), _ang, non), U.detach()], -1).to(device=dev, dtype=dtype).contiguous()
            dXd = dX.detach().to(device=dev, dtype=dtype).contiguous()
            Nd = X_.shape[0]
            if normalize:                                                       # ref: modules.py:166-172
                self.X_mean, self.X_std = X_.mean(0), X_.std(0)
                self.X_std_inv = self.X_std.reciprocal()
                self.dX_mean, self.dX_std = dXd.mean(0), dXd.std(0)
                self.dX_std_inv = self.dX_std.reciprocal()
            H0, H1 = self.model.fc_0.out_features, self.model.fc_1.out_features
            if batch_indices is None:        # DataLoader(shuffle=True) cycled for n_iter steps (modules.py:177-180)
                bs = min(batch_size, Nd)
                per_epoch = (Nd + bs - 1) // bs
                rows = []
                g = None if seed is None else torch.Generator().manual_seed(int(seed))
                while len(rows) < n_iter:
                    perm = torch.randperm(Nd, generator=g)
                    perm = torch.cat([perm, torch.full((per_epoch * bs - Nd,), -1, dtype=perm.dtype)])
                    rows.extend(perm.reshape(per_epoch, bs))
                batch_indices = torch.stack(rows[:n_iter])
            idx = torch.as_tensor(batch_indices).to(device=dev, dtype=torch.int32).contiguous()
            n_iter, bs = int(idx.shape[0]), int(idx.shape[1])
            drops = self._dropouts()
            concrete = isinstance(drops[0], CDropout)
            if any(isinstance(d, CDropout) != concrete for d in drops):
                raise NotImplementedError("pddp_b200: both dropout layers must be of the same kind")
            cfg = self.train_config(dtype, Nd, bs, n_iter, learning_rate, reg_scale, seed)
            lib = _lib.load()
            params = self.flat_parameters(dtype, dev).contiguous()
            grads = torch.zeros_like(params)
            loss = torch.zeros(n_iter, dtype=dtype, device=dev)
            nbytes = lib.pddp_bnn_train_workspace_bytes(C.byref(cfg))
            if nbytes < 0:
                _lib.check(int(nbytes), "bnn_train_workspace_bytes")
            ws = torch.zeros(int(nbytes), dtype=torch.uint8, device=dev)
            vec = lambda b: None if b.dim() == 0 else b.to(device=dev, dtype=dtype).contiguous()
            keep = [vec(self.X_mean), vec(self.X_std_inv), vec(self.dX_mean), vec(self.dX_std)]
            nz = None if noise is None else torch.as_tensor(noise).to(device=dev, dtype=dtype).contiguous()
            if nz is not None and tuple(nz.shape) != (n_iter, bs, H0 + H1):
                raise ValueError("noise must be [n_iter, batch, H0 + H1]")
            with torch.cuda.device(dev):
                _lib.check(lib.pddp_bnn_train(C.byref(cfg), _lib.ptr(X_), _lib.ptr(dXd), *[_lib.ptr(t) for t in keep],
                                              _lib.ptr(idx), _lib.ptr(nz), _lib.ptr(params), _lib.ptr(grads),
                                              _lib.ptr(loss), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()), "bnn_train")
            self._store_flat(params.to(self.model.fc_0.weight.device))
            for d in drops:                  # training leaves [batch, H]-shaped masks behind: the next eval use
                if isinstance(d, CDropout):  # redraws them (modules.py:565-573)
                    d.concrete_noise = None
                else:
                    d.noise.data = torch.bernoulli((1 - d.rate).expand(1))
            self._version += 1
            if return_diagnostics:
                return loss, grads
            return None

        def train_config(self, dtype, n_data, batch, n_iter, learning_rate, reg_scale, seed=None):
            """The pddp_bnn_train configuration of fit(): input width K0 = augmented state + action."""
            drops = self._dropouts()
            concrete = isinstance(drops[0], CDropout)
            H0, H1 = self.model.fc_0.out_features, self.model.fc_1.out_features
            return TrainConfig(_lib.dtype_code(dtype), DA + nu, H0, H1, _state_size, n_data, batch, n_iter,
                               0 if concrete else 1, float(learning_rate), 0.9, 0.999, 1e-8, float(reg_scale),
                               float(drops[0].temperature) if concrete else 0.0, float(drops[0].reg),
                               float(drops[1].reg), float(drops[0].rate), float(drops[1].rate),
                               int(torch.seed() if seed is None else seed) & ((1 << 63) - 1))

        # ------------------------------------------------------------------ what the kernels read
        def descriptor(self, model_opts=None, N=None):
            """BNNDynamics for the kernels.  model_opts selects how input particles are formed
            (ref: modules.py:320-358): infer_noise_variables=False needs eps_in[i] for every step
            i < N; steps the model has not seen yet are drawn here, in step order, the way the
            reference draws them on first use (modules.py:321-329)."""
            opts = model_opts or {}
            P = self.n_particles
            m = self.model
            if 0 not in self.eps_in:
                self.eps_in[0] = _standardised(P, _state_size)
            P = self.eps_in[0].shape[0]
            masks = [d.ensure(P, fc.out_features) for d, fc in zip(self._dropouts(), (m.fc_0, m.fc_1))]
            mode, eps_in = _lib.BNN_INPUT_INFER, None
            if not opts.get("sample_input_distribution", True):
                mode = _lib.BNN_INPUT_MEAN
            elif not opts.get("infer_noise_variables", True):
                mode = _lib.BNN_INPUT_RESAMPLE
                if N is None:
                    raise ValueError("infer_noise_variables=False needs the horizon N to lay out eps_in")
                for i in range(N):
                    if i not in self.eps_in:
                        self.eps_in[i] = _standardised(P, _state_size)
                eps_in = torch.stack([self.eps_in[i] for i in range(N)])
            eps_out = None
            if opts.get("use_predicted_std", False):        # ref: modules.py:242-262, eps_out[i] drawn on first use
                if N is None:
                    raise ValueError("use_predicted_std=True needs the horizon N to lay out eps_out")
                for i in range(N):
                    if i not in self.eps_out:
                        self.eps_out[i] = _standardised(P, _state_size)
                eps_out = torch.stack([self.eps_out[i] for i in range(N)])
            vec = lambda b: None if b.dim() == 0 else b
            return BNNDynamics(geo, [m.fc_0.weight, m.fc_1.weight, m.fc_out.weight],
                               [m.fc_0.bias, m.fc_1.bias, m.fc_out.bias], masks,
                               self.eps_in[0], vec(self.X_mean), vec(self.X_std_inv), vec(self.dX_mean),
                               vec(self.dX_std), input_mode=mode, eps_in=eps_in, eps_out=eps_out,
                               independent_noise=bool(opts.get("independent_noise", False)))

    return BNNDynamicsModel


def check_model_opts(model, model_opts):
    """Options the kernels implement: infer_noise_variables, sample_input_distribution, use_predicted_std and
    independent_noise either way (BNNDynamics.input_mode / eps_out); resample=True (fresh noise on every call) is
    not: all noise is data on this path."""
    if not getattr(model, "is_bnn", False):
        return
    want = dict(resample=False)
    for k, v in model_opts.items():
        if k in want and bool(v) != want[k]:
            raise NotImplementedError("pddp_b200: model option %s=%r is not built (SURVEY 8f rank 2); supported: %r"
                                      % (k, v, want))
