"""Evaluation drivers of the reference's lipschitz.py (lines 23-222) on the B200 kernels: the train loop, the per-cell
KL / local-Lipschitz sweeps in X- and Z-space and the data-based estimates, with the reference's names, signatures,
return values and RNG call order -- but batched (SURVEY.md 8(f) rank 3): one encode, TWO decodes, ONE ratio-kernel
launch, ONE batched quantile and ONE device->host copy for all K*K cells instead of up to 513 sequential estimator calls
with three `.item()` syncs each.  Per-cell results equal the one-cell `utils.estimate_local_lipschitz` call.

    python -m vae_song_b200.lipschitz --model lidvae --IL 0.2 --beta 0.001 --K 8 --std 0.3 --epochs 50 \\
        --hidden_channels 128 64 64 32 16 8 4 2 --batch_size 256 --device cuda        # README.md:41-59 of the reference

The CLI keeps the reference's flags (lipschitz.py:225-279).  Plots are not produced (matplotlib is a host-side
concern, out of scope); the per-cell arrays and the summary go to `<output_dir>/metrics.npz` / `summary.json`.
"""
from __future__ import annotations

import argparse
import json
import os
import random

import numpy as np
import torch

from . import model as _model
from .train import train_model  # noqa: F401  (lipschitz.py:23-44, same signature)
from .utils import (estimate_lipschitz_allpairs, estimate_local_lipschitz, estimate_local_lipschitz_batched,
                    estimate_local_lipschitz_jacobian, reparameterize)

DEFAULT_EMPTY_CELL_FILL_VALUE = -5.0     # lipschitz.py:19


def _kl_per_sample(mu, log_var):
    return -0.5 * torch.sum(1 + log_var - mu.pow(2) - log_var.exp(), dim=1)      # lipschitz.py:62,132,219


def _fill(n, v):
    return np.full(n, v, dtype=np.float32)


def _get_kl_and_lipschitz_for_x_cells(model, test_dataset, K, device, nsamples_z=10, num_pairs_lips=100,
                                      empty_cell_fill_value=DEFAULT_EMPTY_CELL_FILL_VALUE):
    """lipschitz.py:48-86.  Cells are `test_dataset.y == cell_idx`; KL is the cell mean of the per-sample KL of the encoded
    points; the Lipschitz triple comes from `nsamples_z` posterior samples per point.  Returns (kl, lips, inv_lips,
    bi_lips) float32 arrays of K*K entries, empty cells filled with `empty_cell_fill_value`."""
    n = K * K
    kl_vals, lips_vals, inv_vals, bi_vals = (_fill(n, empty_cell_fill_value) for _ in range(4))
    model.eval()
    with torch.no_grad():
        X, y = test_dataset.X.to(device), test_dataset.y.to(device)
        keep = (y >= 0) & (y < n)
        X, y = X[keep], y[keep]
        if X.size(0) == 0:
            return kl_vals, lips_vals, inv_vals, bi_vals
        order = torch.argsort(y, stable=True)                  # same within-cell order as boolean-mask indexing
        Xs, ys = X[order], y[order]
        counts = torch.bincount(ys, minlength=n).tolist()
        mu, log_var = model.encode(Xs)                         # eval-mode BatchNorm: per-sample, so ONE encode for all cells
        kl = _kl_per_sample(mu, log_var)
        cell_sum = torch.zeros(n, device=kl.device, dtype=kl.dtype).index_add_(0, ys, kl)
        cnt_t = torch.tensor(counts, device=kl.device, dtype=kl.dtype)
        kl_mean = (cell_sum / cnt_t.clamp(min=1)).cpu().numpy()
        z_cells, cell_ids, off = [], [], 0
        for c in range(n):
            k = counts[c]
            if k == 0:
                continue
            kl_vals[c] = kl_mean[c]
            if k >= 2:      # per-cell reparameterize calls, in cell order: the reference's RNG stream
                zc = reparameterize(mu[off:off + k], log_var[off:off + k], nsamples=nsamples_z).reshape(-1, mu.size(-1))
                z_cells.append(zc)
                cell_ids.append(c)
            off += k
        if z_cells:
            res = estimate_local_lipschitz_batched(model.decode, z_cells, num_pairs=num_pairs_lips)
            for c, (inv_l, l, bi) in zip(cell_ids, res):
                inv_vals[c], lips_vals[c], bi_vals[c] = inv_l, l, bi
    return kl_vals, lips_vals, inv_vals, bi_vals


def _get_kl_and_lipschitz_for_z_cells(model, K_z, z_min, z_max, actual_latent_dim, device, nsamples_z_per_cell=100,
                                      num_pairs_lips=100, empty_cell_fill_value=DEFAULT_EMPTY_CELL_FILL_VALUE):
    """lipschitz.py:89-154.  For each of the K_z*K_z grid centres: 100 samples centre + 0.1*N(0,I), decode -> encode -> KL,
    and the Lipschitz triple of the decoder on those samples."""
    if actual_latent_dim != 2:
        raise ValueError(f"Skipping Z-space grid evaluation: Model's actual latent dimension is {actual_latent_dim}D, not 2D.")
    n = K_z * K_z
    kl_vals, lips_vals, inv_vals, bi_vals = (_fill(n, empty_cell_fill_value) for _ in range(4))
    model.eval()
    cx = np.linspace(z_min, z_max, K_z)
    centers = torch.tensor([[cx[xi], cx[yi]] for yi in range(K_z) for xi in range(K_z)], dtype=torch.float32, device=device)
    with torch.no_grad():
        # per-cell randn calls in cell order: the reference's RNG stream
        z_cells = [centers[c].repeat(nsamples_z_per_cell, 1)
                   + torch.randn(nsamples_z_per_cell, actual_latent_dim, device=device) * 0.1 for c in range(n)]
        z_all = torch.cat(z_cells, 0)
        x_recon = model.decode(z_all)                          # no autograd graph needed (reference defect D4)
        mu_re, log_var_re = model.encode(x_recon)
        kl = _kl_per_sample(mu_re, log_var_re).view(n, nsamples_z_per_cell).mean(1)
        kl_vals[:] = kl.cpu().numpy()
        if nsamples_z_per_cell >= 2:
            res = estimate_local_lipschitz_batched(model.decode, z_cells, num_pairs=num_pairs_lips)
            inv_vals[:], lips_vals[:], bi_vals[:] = res[:, 0], res[:, 1], res[:, 2]
    return kl_vals, lips_vals, inv_vals, bi_vals


def _data_based_samples(model, test_dataset, device, num_samples):
    """Shared front end of lipschitz.py:157-222: encode the data, subsample / oversample to `num_samples` posterior draws."""
    X = test_dataset.X.to(device)
    mu, log_var = model.encode(X)
    if X.size(0) < num_samples:
        z = reparameterize(mu, log_var, nsamples=num_samples // X.size(0) + 1).reshape(-1, mu.size(-1))[:num_samples]
        return z, mu, log_var
    idx = torch.randperm(X.size(0))[:num_samples].to(device)   # CPU generator, like the reference
    mu_s, lv_s = mu[idx], log_var[idx]
    return reparameterize(mu_s, lv_s, nsamples=1).squeeze(1), mu_s, lv_s


def _get_data_based_lipschitz(model, test_dataset, device, num_samples=5000, num_pairs_lips=5000,
                              empty_cell_fill_value=DEFAULT_EMPTY_CELL_FILL_VALUE, pairs="sampled"):
    """lipschitz.py:157-194 -> (inverse_lipschitz, lipschitz, bi_lipschitz) floats.  pairs="all" (an extension) takes the
    same triple over every pair of the same `num_samples` points instead of `num_pairs_lips` random pairs: exact
    quantiles, utils.estimate_lipschitz_allpairs(quantile=0.05).  pairs="jacobian" (an extension, LIDVAE only) takes it
    over the decoder's local constants at those points: the extreme singular values of its exact Jacobian,
    utils.estimate_local_lipschitz_jacobian(quantile=0.05)."""
    if pairs not in ("sampled", "all", "jacobian"):
        raise ValueError(f"pairs must be 'sampled', 'all' or 'jacobian', got {pairs!r}")
    if pairs == "jacobian" and not hasattr(model, "decode_jacobian"):
        raise ValueError(f"pairs='jacobian' needs a decoder with an exact Jacobian (LIDVAE), not {type(model).__name__}")
    model.eval()
    with torch.no_grad():
        z, _, _ = _data_based_samples(model, test_dataset, device, num_samples)
        if pairs == "jacobian":
            return estimate_local_lipschitz_jacobian(model, z, quantile=0.05)
        if pairs == "all":
            r = estimate_lipschitz_allpairs(model.decode, z, quantile=0.05)
            return r["inverse_lipschitz"], r["lipschitz"], r["bi_lipschitz"]
        return estimate_local_lipschitz(model.decode, z, num_pairs=num_pairs_lips)


def _get_data_based_kl(model, test_dataset, device, num_samples=5000):
    """lipschitz.py:197-222 -> average per-sample KL.  (The reference leaves `log_var_subset` undefined when the data set
    is smaller than num_samples -- defect D9; here that branch uses all encoded points.)"""
    model.eval()
    with torch.no_grad():
        _, mu_s, lv_s = _data_based_samples(model, test_dataset, device, num_samples)
        return _kl_per_sample(mu_s, lv_s).mean().item()


# ------------------------------------------------------------------------------------------------- synthetic data + CLI
class GaussianMixture2D(torch.utils.data.Dataset):
    """Synthetic stand-in for the reference's SimpleGaussianMixtureDataset (dataset.py:362-448; host-side numpy, out of
    scope): `num_components` isotropic Gaussians with centres uniform in [0, center_range)^2, `.X` [N,2] fp32 and
    `.y` [N] int64 component labels.  Pass the reference's own dataset object to the functions above for parity."""

    def __init__(self, num_components, total_samples, center_range=4.0, stds=0.2, pattern="uniform", seed=None):
        rng = np.random.default_rng(seed)
        centers = rng.uniform(0, center_range, size=(num_components, 2))
        w = np.ones(num_components)
        if pattern == "corner_heavy":
            w = 1.0 + 4.0 * (np.abs(centers / center_range - 0.5).max(1) > 0.3)
        elif pattern == "center_heavy":
            w = 1.0 + 4.0 * (np.abs(centers / center_range - 0.5).max(1) < 0.25)
        elif pattern == "sparse_random":
            w = rng.uniform(0.05, 1.0, num_components) ** 3
        lab = rng.choice(num_components, size=total_samples, p=w / w.sum())
        pts = centers[lab] + rng.normal(0, stds, size=(total_samples, 2))
        self.X = torch.tensor(pts, dtype=torch.float32)
        self.y = torch.tensor(lab, dtype=torch.int64)

    def __len__(self):
        return self.X.size(0)

    def __getitem__(self, i):
        return self.X[i], self.y[i]


def build_parser():
    p = argparse.ArgumentParser(description="VAE experiment for local Lipschitz and KL regularization (B200 kernels).")
    p.add_argument("--alpha", type=float, default=0.1)
    p.add_argument("--IL", type=float, default=0.0)
    p.add_argument("--model", type=str, default="lrvae", choices=["lrvae", "lidvae"])
    p.add_argument("--K", type=int, default=16)
    p.add_argument("--std", type=float, default=0.1)
    p.add_argument("--epochs", type=int, default=1000)
    p.add_argument("--lr", type=float, default=1e-3)
    p.add_argument("--beta", type=float, default=1.0)
    p.add_argument("--batch_size", type=int, default=256)
    p.add_argument("--device", type=str, default="cuda")
    p.add_argument("--output_dir", type=str, default="results/ablation")
    p.add_argument("--train_total_samples", type=int, default=10000)
    p.add_argument("--test_total_samples", type=int, default=10000)
    p.add_argument("--distribution_pattern", type=str, default="corner_heavy",
                   choices=["uniform", "corner_heavy", "center_heavy", "sparse_random"])
    p.add_argument("--seed", type=int, default=None)
    p.add_argument("--latent_dim", type=int, default=2)
    p.add_argument("--hidden_channels", nargs="+", type=int, default=[64, 128, 64, 2])
    p.add_argument("--num_training_components", type=int, default=8)
    p.add_argument("--K_z", type=int, default=16)
    p.add_argument("--z_min", type=float, default=-3.0)
    p.add_argument("--z_max", type=float, default=3.0)
    p.add_argument("--grad_clip_enabled", action="store_true")
    p.add_argument("--grad_clip_type", type=str, default="norm", choices=["norm", "value"])
    p.add_argument("--grad_clip_max_norm", type=float, default=1.0)
    p.add_argument("--grad_clip_norm_type", type=float, default=2.0)
    p.add_argument("--grad_clip_value", type=float, default=1.0)
    p.add_argument("--wu_strat", type=str, default="linear", choices=["linear", "exponential", "repeat_linear", "kl_adaptive"])
    p.add_argument("--wu_start_epoch", type=int, default=0)
    p.add_argument("--wu_up_amount", type=float, default=None)
    p.add_argument("--wu_repeat_interval", type=int, default=10)
    p.add_argument("--precision", type=str, default="fp32", choices=["fp32", "f16x3", "tf32x3", "tf32"],
                   help="arithmetic of the ICNN contractions (extension; fp32 = the parity path)")
    p.add_argument("--lipschitz_pairs", type=str, default="sampled", choices=["sampled", "all", "jacobian"],
                   help="pairs of the data-based Lipschitz estimate (extension): the reference's random pairs, every "
                        "pair of the 5000 samples with exact quantiles, or (lidvae only) no pairs but the singular values "
                        "of the decoder's exact Jacobian at the 5000 samples; the per-cell grids always sample")
    return p


def evaluate(model, dataset, K, K_z, z_min, z_max, latent_dim, device, num_pairs_cells=2000, num_pairs_data=5000,
             lipschitz_pairs="sampled"):
    """Steps 4-6 of lipschitz.main (lipschitz.py:423-520) without the plots; `lipschitz_pairs` as in
    _get_data_based_lipschitz."""
    out = {}
    kx = _get_kl_and_lipschitz_for_x_cells(model, dataset, K, device, nsamples_z=10, num_pairs_lips=num_pairs_cells)
    out.update(dict(zip(("kl_x", "lips_x", "inv_lips_x", "bi_lips_x"), kx)))
    if latent_dim == 2:
        kz = _get_kl_and_lipschitz_for_z_cells(model, K_z, z_min, z_max, latent_dim, device, nsamples_z_per_cell=100,
                                               num_pairs_lips=num_pairs_cells)
        out.update(dict(zip(("kl_z", "lips_z", "inv_lips_z", "bi_lips_z"), kz)))
    inv_l, l, bi = _get_data_based_lipschitz(model, dataset, device, num_samples=5000, num_pairs_lips=num_pairs_data,
                                             pairs=lipschitz_pairs)
    out["data_inv_lips"], out["data_lips"], out["data_bi_lips"] = inv_l, l, bi
    out["data_kl"] = _get_data_based_kl(model, dataset, device, num_samples=5000)
    return out


def main(argv=None):
    args = build_parser().parse_args(argv)
    if args.lipschitz_pairs == "jacobian" and args.model != "lidvae":
        raise ValueError("--lipschitz_pairs jacobian needs --model lidvae (the decoder's exact Jacobian)")
    os.makedirs(args.output_dir, exist_ok=True)
    seed = 42 if args.seed is None else args.seed
    random.seed(seed); np.random.seed(seed); torch.manual_seed(seed)
    if torch.cuda.is_available():
        torch.cuda.manual_seed_all(seed)
    latent_dim = args.hidden_channels[-1]
    train_dataset = GaussianMixture2D(args.num_training_components, args.train_total_samples, center_range=args.K,
                                      stds=args.std, pattern=args.distribution_pattern, seed=seed)
    g_loader = torch.Generator(device="cpu").manual_seed(seed)
    loader = torch.utils.data.DataLoader(train_dataset, batch_size=args.batch_size, shuffle=True, drop_last=True,
                                         generator=g_loader)
    if args.model == "lidvae":
        model = _model.LIDVAE(inverse_lipschitz=args.IL, beta=args.beta, dataset="pinwheel",
                              hidden_channels=args.hidden_channels, precision=args.precision)
    else:
        model = _model.LRVAE(alpha=args.alpha, dataset="pinwheel", hidden_channels=args.hidden_channels)
        model.beta, model.alpha, model.wu_alpha = args.beta, args.alpha, 1.0
    clip = dict(enabled=args.grad_clip_enabled, clip_type=args.grad_clip_type, max_norm=args.grad_clip_max_norm,
                norm_type=args.grad_clip_norm_type, clip_value=args.grad_clip_value)
    train_model(model, loader, args.epochs, args.lr, args.device, grad_clip=clip, wu_strat=args.wu_strat,
                wu_start_epoch=args.wu_start_epoch, wu_up_amount=args.wu_up_amount,
                wu_repeat_interval=args.wu_repeat_interval)
    z_min, z_max = args.z_min, args.z_max
    model.eval()
    if latent_dim == 2:      # Z-grid extent from the encoded data, like lipschitz.py:400-420
        with torch.no_grad():
            mu, lv = model.encode(train_dataset.X.to(args.device))
            zt = reparameterize(mu, lv, nsamples=1).squeeze(1)
            z_min, z_max = float(zt[:, 0].min()), float(zt[:, 0].max())
    if args.model != "lidvae":
        model.alpha = model.wu_alpha = args.alpha
    res = evaluate(model, train_dataset, args.K, args.K_z, z_min, z_max, latent_dim, args.device,
                   lipschitz_pairs=args.lipschitz_pairs)
    arrays = {k: v for k, v in res.items() if isinstance(v, np.ndarray)}
    scalars = {k: float(v) for k, v in res.items() if not isinstance(v, np.ndarray)}
    np.savez(os.path.join(args.output_dir, "metrics.npz"), **arrays)
    with open(os.path.join(args.output_dir, "summary.json"), "w") as f:
        json.dump(dict(args=vars(args), z_extent=[z_min, z_max], data_lipschitz_pairs=args.lipschitz_pairs, **scalars), f,
                  indent=1)
    print(json.dumps(scalars))
    return res


if __name__ == "__main__":
    main()
