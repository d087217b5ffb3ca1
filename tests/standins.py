"""Seeded, frozen stand-ins for the LaLiGAN autoencoder and Lie generator.

The symmetry regularisers (`model_utils.py` symmreg_i / symmreg_r / symmreg_f) take a trained autoencoder and
generator as frozen inputs; the reference's checkpoints for them are not shipped (SURVEY.md §8c) and both
modules are outside the hot path. These minimal modules expose exactly the attributes the regularisers touch
(`encode`, `decode`, `decoder`, `encoder[-2].bias`, `get_full_basis_list`, `get_deterministic_group_elems`,
`Li`) with the same tensor shapes: x (B, n_comps, input_dim) <-> z (B, n_comps, latent_dim), generators
(n_comps·latent_dim)². Used identically by the golden generator (with the reference's regularisers) and by the
GPU parity tests (with ours). `make_reference_tree` lays out an empty stand-in of the reference checkout for the
launcher's import-resolution tests.
"""
import torch
import torch.nn as nn


class StandInAutoEncoder(nn.Module):
    def __init__(self, input_dim=2, latent_dim=2, n_comps=2, hidden=32):
        super().__init__()
        self.n_comps, self.latent_dim = n_comps, latent_dim

        class Flat(nn.Module):
            def forward(self, x):
                return x.reshape(-1, x.shape[-1])

        class Unflat(nn.Module):
            def forward(self, x):
                return x.reshape(-1, n_comps, x.shape[-1])

        # encoder[-2] is the last BatchNorm, whose bias is the default latent centre (model_utils.py:45-46)
        self.encoder = nn.Sequential(
            nn.Linear(input_dim, hidden), nn.Tanh(),
            nn.Linear(hidden, hidden), nn.Tanh(),
            nn.Linear(hidden, latent_dim),
            Flat(), nn.BatchNorm1d(latent_dim), Unflat(),
        )
        self.decoder = nn.Sequential(
            nn.Linear(latent_dim, hidden), nn.Tanh(),
            nn.Linear(hidden, hidden), nn.Tanh(),
            nn.Linear(hidden, input_dim),
        )

    @property
    def device(self):
        return next(self.parameters()).device

    def encode(self, x):
        return self.encoder(x)

    def decode(self, z):
        return self.decoder(z)

    def forward(self, x):
        z = self.encode(x)
        return z, self.decode(z)


class StandInGenerator(nn.Module):
    def __init__(self, n_dims=4, n_gens=2, seed=0):
        super().__init__()
        g = torch.Generator().manual_seed(1000 + seed)
        self.Li = nn.ParameterList([nn.Parameter(0.5 * torch.randn(n_dims, n_dims, generator=g)) for _ in range(n_gens)])
        self.sigma = [1.0] * n_gens

    def get_full_basis_list(self, split_channel=True):
        return [L for L in self.Li]

    def get_deterministic_group_elems(self, split_channel=False, scale=1.0):
        return [torch.matrix_exp(s * L * scale) for s, L in zip(self.sigma, self.Li)]


STANDIN_REFERENCE_MODULES = ("sindy.py", "model_utils.py", "gan.py", "autoencoder.py", "dataset.py", "parser_utils.py",
                             "evaluation/__init__.py", "evaluation/eval_eq.py", "data_utils/__init__.py",
                             "data_utils/ode.py", "data_utils/smoothing.py", "data_utils/damped_oscillator.py",
                             "data_utils/growth.py", "data_utils/lotka.py", "data_utils/selkov.py")


def make_reference_tree(path):
    """A directory laid out like the reference checkout (the module names the launcher and the drop-in modules resolve,
    `train.py` with a `train_lassi`), each module empty: enough to test where imports resolve without the reference's
    code. Returns the directory."""
    import os
    for rel in STANDIN_REFERENCE_MODULES:
        f = os.path.join(path, rel)
        os.makedirs(os.path.dirname(f), exist_ok=True)
        with open(f, "w") as fh:
            fh.write('"""Stand-in for the reference module of the same name."""\n')
    with open(os.path.join(path, "train.py"), "w") as fh:
        fh.write('"""Stand-in for the reference\'s train.py."""\n\n\ndef train_lassi(*args, **kwargs):\n    pass\n')
    return path


def make_standins(seed=0, input_dim=2, n_comps=2, hidden=32, latent_dim=None, state_dict=None, device="cpu"):
    latent_dim = input_dim if latent_dim is None else latent_dim
    torch.manual_seed(10_000 + seed)
    ae = StandInAutoEncoder(input_dim, latent_dim, n_comps, hidden)
    bn = ae.encoder[-2]
    with torch.no_grad():  # non-trivial eval-mode statistics and centre
        bn.running_mean.copy_(0.1 * torch.randn(latent_dim))
        bn.running_var.copy_(1.0 + 0.2 * torch.rand(latent_dim))
        bn.weight.copy_(1.0 + 0.1 * torch.randn(latent_dim))
        bn.bias.copy_(0.2 * torch.randn(latent_dim))
    gen = StandInGenerator(n_comps * latent_dim, 2, seed)
    if state_dict is not None:
        ae.load_state_dict(state_dict)
    for m in (ae, gen):
        m.eval()
        for q in m.parameters():
            q.requires_grad_(False)
    return ae.to(device), gen.to(device)
