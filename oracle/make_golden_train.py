"""Golden vectors for BNN TRAINING (SURVEY 8f rank 4): runs the UNMODIFIED reference's
`BNNDynamicsModel.fit` (pddp/models/bnn/modules.py:131-198, via oracle/refshim.py) on a small synthetic
dataset and records everything the run consumed and produced:

  inputs   dataset (X, U, dX), initial weights / logit_p, the mini-batch rows of every step (recovered by
           matching the normalised rows the network was fed against the dataset) and the uniform dropout
           noise of every step (`torch.rand_like` is wrapped to record what it returns)
  outputs  the loss of every step (recomputed from the recorded tensors with the reference's own modules),
           the gradients of the FIRST step, and all parameters after the last step

`tests/test_gpu_train.py` replays the same batches and noise through `pddp_bnn_train` and compares.
Run in the build container only (needs /root/reference):   python oracle/make_golden_train.py
TEST INFRASTRUCTURE ONLY."""
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import refshim  # noqa: E402

warnings.filterwarnings("ignore")
refshim.import_reference()

from pddp.models.bnn import bnn_dynamics_model_factory  # noqa: E402
from pddp.models.bnn.modules import BDropout, CDropout  # noqa: E402
from pddp.models.bnn.losses import gaussian_log_likelihood  # noqa: E402
from pddp.examples.cartpole.model import CartpoleDynamicsModel  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")


def flat(model):
    m = model.model
    parts = [m.fc_0.weight, m.fc_0.bias, m.fc_1.weight, m.fc_1.bias, m.fc_out.weight, m.fc_out.bias]
    parts += [getattr(d, "logit_p", torch.zeros(())) for d in (m.drop_0, m.drop_1)]
    return torch.cat([p.detach().reshape(-1) for p in parts])


def flat_grads(model):
    m = model.model
    parts = [m.fc_0.weight, m.fc_0.bias, m.fc_1.weight, m.fc_1.bias, m.fc_out.weight, m.fc_out.bias]
    parts += [getattr(d, "logit_p", None) for d in (m.drop_0, m.drop_1)]
    return torch.cat([(torch.zeros(1, dtype=torch.get_default_dtype()) if p is None or p.grad is None else p.grad).reshape(-1)
                      for p in parts])


def run(tag, dropout, dtype, n_data, hidden, n_iter, batch_size, lr, reg_scale, seed):
    torch.set_default_dtype(dtype)
    torch.manual_seed(seed)
    D, ang, non = 4, CartpoleDynamicsModel.angular_indices, CartpoleDynamicsModel.non_angular_indices
    kwargs = {} if dropout == "concrete" else {"dropout_layers": BDropout, "initial_p": 0.25}
    model = bnn_dynamics_model_factory(D, 1, hidden, ang, non, **kwargs)(n_particles=10)
    X = torch.randn(n_data, D)
    U = 2.0 * torch.randn(n_data, 1)
    dX = 0.1 * torch.randn(n_data, D) + 0.05 * X
    p_init = flat(model).clone()

    # record the uniform noise of every dropout call and the rows every step was fed
    noises, fed, targets = [], [], []
    real_rand_like, real_bernoulli = torch.rand_like, torch.bernoulli

    def rand_like(x, *a, **k):
        r = real_rand_like(x, *a, **k)
        noises.append(r.detach().clone())
        return r

    def bernoulli(p, *a, **k):                 # BDropout(resample=True) draws bernoulli(p.expand(x.shape)) directly:
        u = real_rand_like(p)                  # replace it by a recorded uniform compared with p (same distribution)
        noises.append(u.detach().clone())
        return (u < p).to(p.dtype)

    def likelihood(dx, mean, std):
        targets.append(dx.detach().clone())
        return gaussian_log_likelihood(dx, mean, std)

    hook = model.model.register_forward_pre_hook(lambda mod, inp: fed.append(inp[0].detach().clone()))
    first_grads = []
    real_step = torch.optim.Adam.step

    def step(self, *a, **k):
        if not first_grads:
            first_grads.append(flat_grads(model).clone())
        return real_step(self, *a, **k)

    torch.rand_like, torch.optim.Adam.step = rand_like, step
    if dropout != "concrete":
        torch.bernoulli = bernoulli
    try:
        model.train()
        model.fit(X, U, dX, n_iter=n_iter, batch_size=batch_size, reg_scale=reg_scale, learning_rate=lr,
                  likelihood=likelihood, quiet=True)
    finally:
        torch.rand_like, torch.optim.Adam.step, torch.bernoulli = real_rand_like, real_step, real_bernoulli
        hook.remove()
    p_final = flat(model).clone()

    # mini-batch rows: match the normalised rows the network saw against the (normalised) dataset
    from pddp.utils.angular import augment_state
    X_ = torch.cat([augment_state(X, ang, non), U], -1)
    Xn = (X_ - model.X_mean) * model.X_std_inv
    bs = max(f.shape[0] for f in fed)
    idx = -np.ones((n_iter, bs), dtype=np.int32)
    noise = 0.5 * np.ones((n_iter, bs, sum(hidden)), dtype=np.float64)
    for it, f in enumerate(fed):
        d = (f[:, None, :] - Xn[None, :, :]).abs().sum(-1)
        rows = d.argmin(1)
        assert float(d.min(1).values.max()) == 0.0, "fed rows must be dataset rows bit for bit"
        assert torch.equal(dX[rows], targets[it])
        idx[it, :len(rows)] = rows.numpy()
        n0, n1 = noises[2 * it], noises[2 * it + 1]
        noise[it, :len(rows), :hidden[0]] = n0.double().numpy()
        noise[it, :len(rows), hidden[0]:] = n1.double().numpy()
    assert len(noises) == 2 * n_iter

    # loss of every step, recomputed with the reference's modules from the recorded tensors would need the
    # parameters of every step; instead store the first step's loss (initial parameters are known)
    model2 = bnn_dynamics_model_factory(D, 1, hidden, ang, non, **kwargs)(n_particles=10)
    o = 0
    m2 = model2.model
    for p in (m2.fc_0.weight, m2.fc_0.bias, m2.fc_1.weight, m2.fc_1.bias, m2.fc_out.weight, m2.fc_out.bias):
        p.data.copy_(p_init[o:o + p.numel()].reshape(p.shape))
        o += p.numel()
    for buf in ("X_mean", "X_std", "X_std_inv", "dX_mean", "dX_std", "dX_std_inv"):
        getattr(model2, buf).data = getattr(model, buf).data.clone()
    model2.train()
    queue = [noises[0], noises[1]]
    torch.rand_like = lambda x, *a, **k: queue.pop(0)
    if dropout != "concrete":
        torch.bernoulli = lambda p, *a, **k: (queue.pop(0) < p).to(p.dtype)
    try:
        out = model2.model(fed[0], resample=True)
        mean, log_std = out.split([D, D], dim=-1)
        mean, log_std = model2._scale_output(mean, log_std)
        loss0 = -gaussian_log_likelihood(targets[0], mean, log_std.exp()).mean() + reg_scale * model2.model.regularization() / n_data
    finally:
        torch.rand_like, torch.bernoulli = real_rand_like, real_bernoulli

    os.makedirs(OUT, exist_ok=True)
    np.savez_compressed(
        os.path.join(OUT, tag + ".npz"), dropout=0 if dropout == "concrete" else 1, hidden=np.array(hidden), n_iter=n_iter,
        batch_size=batch_size, lr=lr, reg_scale=reg_scale, X=X.numpy(), U=U.numpy(), dX=dX.numpy(), p_init=p_init.numpy(),
        p_final=p_final.numpy(), grads0=first_grads[0].numpy(), loss0=float(loss0), batch_idx=idx,
        X_mean=model.X_mean.numpy(), X_std_inv=model.X_std_inv.numpy(), dX_mean=model.dX_mean.numpy(),
        dX_std=model.dX_std.numpy(), rate=float(model.model.drop_0.rate), reg=float(model.model.drop_0.reg))
    # the noise is most of the bytes and barely compresses: its own file keeps each under 1 MB (tests/train_util.py)
    np.savez_compressed(os.path.join(OUT, tag + ".noise.npz"),
                        noise=noise.astype(np.float64 if dtype == torch.float64 else np.float32))
    print("%-28s steps %d  batches of <= %d  loss0 %.6f  |dp| %.3e" % (tag, n_iter, bs, float(loss0),
                                                                      float((p_final - p_init).abs().max())))


if __name__ == "__main__":
    run("train_cartpole_concrete_f64", "concrete", torch.float64, 150, [48, 40], 7, 64, 1e-3, 1.0, 0)
    run("train_cartpole_concrete_f32", "concrete", torch.float32, 300, [200, 200], 5, 128, 1e-3, 1.0, 1)
    run("train_cartpole_bernoulli_f64", "bernoulli", torch.float64, 100, [32, 56], 6, 32, 2e-3, 0.5, 2)
