"""Host-side helpers with the reference's utils.py signatures for the hot path
(reparameterize utils.py:40-47, kld :140-141, apply_grad_clip :12-38, estimate_local_lipschitz :532-567)
plus the tiled all-pairs estimator the north_star adds."""
from __future__ import annotations

import torch

from . import ops


def flops_decode(d, H):
    """Algorithmic flops per sample of one ICNN decode (psi + grad psi), multiply-add = 2 (SURVEY.md 8(d)):
    forward P0 x1 (2H^2) + reverse P0^T g1 (2H^2) + four [d,H] products + the P1 dot + A2."""
    return 4 * H * H + 8 * d * H + 2 * H + 4 * d


def flops_train(d, H):
    """Decode + double-backward per sample (SURVEY.md 8(d)): adds P0 q1, g1^T q1, A0 v, A1 v, three [H,d] outer products."""
    return 8 * H * H + 22 * d * H


def trained_like_icnn_(icnn, rng):
    """O(1)-scale, mixed-sign weights for synthetic benchmarks (the default exp(W) ~ 1 init gives ~1e10 outputs,
    SURVEY Appendix B.8).  `rng`: numpy Generator."""
    import numpy as np
    H = icnn.hidden_channel
    with torch.no_grad():
        icnn.W[0].param.copy_(torch.tensor(rng.normal(np.log(1.0 / H), 1.0, (H, H)), dtype=torch.float32))
        icnn.W[1].param.copy_(torch.tensor(rng.normal(np.log(2.0 / H), 1.0, (1, H)), dtype=torch.float32))
        icnn.A[0].bias.copy_(torch.tensor(rng.normal(-0.3, 1.0, (H,)), dtype=torch.float32))
    return icnn


def apply_grad_clip(model, grad_clip_cfg):
    """Same config contract as the reference: {'enabled', 'clip_type': 'norm'|'value', 'max_norm',
    'norm_type', 'clip_value'}; anything else is a no-op."""
    if not grad_clip_cfg or not grad_clip_cfg.get("enabled", False):
        return
    kind = grad_clip_cfg.get("clip_type", "norm")
    if kind == "norm":
        torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm=float(grad_clip_cfg.get("max_norm", 1.0)),
                                       norm_type=float(grad_clip_cfg.get("norm_type", 2.0)))
    elif kind == "value":
        torch.nn.utils.clip_grad_value_(model.parameters(), float(grad_clip_cfg.get("clip_value", 1.0)))


def reparameterize(mu, logvar, nsamples=1, generator=None):
    """Posterior samples [batch, nsamples, nz] (fused kernel; eps drawn exactly like the reference:
    randn_like on the expanded [B,ns,nz] std)."""
    B, nz = mu.size()
    eps = torch.randn_like(mu.unsqueeze(1).expand(B, nsamples, nz))          # [B,ns,nz], same RNG stream
    z = ops.ReparamFn.apply(mu, logvar, eps.permute(1, 0, 2).contiguous())   # kernel layout [L,B,D]
    return z.permute(1, 0, 2).contiguous()      # the reference returns a contiguous tensor: lipschitz.py:68 calls .view() on it


def kld(mu, log_var):
    _, kl, _ = ops.VaeLossFn.apply(None, None, mu.detach(), log_var.detach(), None, None, False)
    return kl.item()


# ---- end-of-run latent metrics (utils.py:49-164; SURVEY.md 8(f) rank 4) ------------------------------------------------------
def calc_au_per_batch(z, eps=0.01):
    """utils.py:49-50: fraction of latent dimensions whose batch variance (biased) is >= eps."""
    return (torch.mean((z - z.mean(dim=0, keepdim=True)) ** 2, dim=0) >= eps).float().mean().item()


def log_sum_exp(value, dim=None, keepdim=False):
    """utils.py:74-85."""
    return torch.logsumexp(value, dim=dim, keepdim=keepdim) if dim is not None else torch.logsumexp(value.reshape(-1), 0)


def calc_mi(mu, logvar, eps=None):
    """utils.py:87-107 (Wang et al.): I(x,z) ~= E log q(z|x) - E log q(z).  The aggregate-posterior term is the tiled
    all-pairs kernel b200vae_mi_logqz (online logsumexp; no [B,B,nz] tensor).  `eps` may be injected for tests."""
    import math
    from . import _C
    B, nz = mu.size()
    mu, logvar = ops._req(mu.detach(), "mu"), ops._req(logvar.detach(), "logvar")
    neg_entropy = (-0.5 * nz * math.log(2 * math.pi) - 0.5 * (1 + logvar).sum(-1)).mean()
    if eps is None:
        z = reparameterize(mu, logvar, 1).reshape(B, nz).contiguous()
    else:
        z = (mu + eps * (0.5 * logvar).exp()).contiguous()
    log_qz = torch.empty(B, dtype=torch.float32, device=mu.device)
    _C.check(_C.load().b200vae_mi_logqz(ops._ptr(z), ops._ptr(mu), ops._ptr(logvar), B, nz, ops._ptr(log_qz), ops._stream()),
             "mi_logqz")
    return (neg_entropy - log_qz.mean()).item()


def eval_inference_dist(mu, logvar, z):
    """utils.py:128-138: log q(z|x) for z [B,ns,nz]."""
    import math
    nz = z.size(2)
    mu, logvar = mu.unsqueeze(1), logvar.unsqueeze(1)
    return -0.5 * (((z - mu) ** 2) / logvar.exp()).sum(dim=-1) - 0.5 * (nz * math.log(2 * math.pi) + logvar.sum(-1))


_iw_scratch = {}


def nll_iw(mu, log_var, loss_rec, nsamples=100, eps=None):
    """utils.py:109-120: importance-weighted NLL estimate (a scalar over the whole batch, like the reference).  One fused
    kernel (b200vae_nll_iw_lse): eps is drawn exactly like utils.reparameterize does (randn_like on the expanded
    [B,ns,nz] std), so the same seed gives the reference's samples; z and the [B,ns] log-density tensors are never formed.
    `eps` [B,ns,nz] may be injected for tests."""
    import math
    from . import _C
    lib = _C.load()
    mu, log_var = ops._req(mu.detach(), "mu"), ops._req(log_var.detach(), "log_var")
    B, nz = mu.shape
    if eps is None:
        eps = torch.randn_like(mu.unsqueeze(1).expand(B, nsamples, nz))
    eps = ops._req(eps, "eps")
    key = (mu.device, torch.cuda.current_stream().cuda_stream)
    scr = _iw_scratch.get(key)
    if scr is None:
        scr = _iw_scratch[key] = torch.zeros(lib.b200vae_nll_iw_scratch_bytes(), dtype=torch.uint8, device=mu.device)
    out = torch.empty(1, dtype=torch.float32, device=mu.device)
    _C.check(lib.b200vae_nll_iw_lse(ops._ptr(mu), ops._ptr(log_var), ops._ptr(eps), B, eps.shape[1], nz, ops._ptr(out),
                                    ops._ptr(scr), ops._stream()), "nll_iw_lse")
    rec = loss_rec.detach().float().reshape(()) if torch.is_tensor(loss_rec) else float(loss_rec)
    return -(out[0] - rec - math.log(eps.shape[1])).item()


def measure_pc_runmodel(model, loader, device):
    """utils.py:144-164: (AU, KL, MI, NLL, sum of variances) on the FIRST batch of the loader."""
    au_sum = kl_sum = mi_sum = nll_sum = var_sum = 0
    for i, data in enumerate(loader):
        if i > 0:
            break
        x = data[0].to(device)
        res = model(x)
        recon, mu, log_var = res[0], res[1], res[2]
        z_in = res[3] if len(res) > 3 else None
        z_rec = res[4] if len(res) > 4 else None
        _, loss_rec, _, _ = model.loss(x, recon, mu, log_var, z_input=z_in, z_recon=z_rec)
        au_sum += calc_au_per_batch(mu.detach())
        kl_sum += kld(mu, log_var)
        mi_sum += calc_mi(mu, log_var)
        nll_sum += nll_iw(mu, log_var, loss_rec.detach() if torch.is_tensor(loss_rec) else loss_rec)
        if torch.is_tensor(log_var):
            var_sum += log_var.detach().exp().sum().item()
    return au_sum, kl_sum, mi_sum, nll_sum, var_sum


def compute_local_reg(model, loader, K):
    """utils.py:509-530: per grid cell, the model's regularisation loss part divided by the cell's sample count (0.0 for
    an empty cell) -> numpy array [K*K].  `loader.dataset` carries `.X` and `.y` (cell labels)."""
    import numpy as np
    device = next(model.parameters()).device
    model.eval()
    regs = []
    with torch.no_grad():
        X_all, y_all = loader.dataset.X, loader.dataset.y
        for cell in range(K * K):
            mask = (y_all == cell)
            if mask.sum() == 0:
                regs.append(0.0)
                continue
            X_cell = X_all[mask].to(device)
            recon, mu, log_var, z_input, z_recon = model(X_cell)
            _, _, loss_reg_term, _ = model.loss(X_cell, recon, mu, log_var, z_input, z_recon)
            regs.append(float(loss_reg_term) / X_cell.size(0))
    return np.array(regs)


def _plotting_out_of_scope(name):
    def fn(*args, **kwargs):
        raise NotImplementedError(f"utils.{name}: matplotlib plotting is outside the hot path this package covers (DESIGN.md, "
                                  "'Out of scope'); the name exists so that the reference's drivers import unchanged")
    fn.__name__ = name
    return fn


plot_heatmap = _plotting_out_of_scope("plot_heatmap")
plot_2d_histogram = _plotting_out_of_scope("plot_2d_histogram")


def estimate_local_lipschitz(func, X, num_pairs=2000, metric=2, quantile=0.05, eps=1e-3, generator=None,
                             use_grad=False):
    """Random-pair local Lipschitz estimate, reference semantics (utils.py:532-567):
    returns (inverse_lipschitz, lipschitz, bi_lipschitz) as Python floats."""
    if X.size(0) < 2:
        return 0.0, 0.0, 0.0
    N = X.size(0)
    if generator is None:
        generator = torch.Generator(device=X.device).manual_seed(0)
    idx1 = torch.randint(0, N, (num_pairs,), device=X.device, generator=generator)
    idx2 = torch.randint(0, N, (num_pairs,), device=X.device, generator=generator)
    x1, x2 = X[idx1], X[idx2]
    if use_grad:   # kept for API parity: our decode needs no autograd graph (reference defect D4)
        x1 = x1.detach().clone().requires_grad_(True)
        x2 = x2.detach().clone().requires_grad_(True)
        y1, y2 = func(x1), func(x2)
    else:
        with torch.no_grad():
            y1, y2 = func(x1), func(x2)
    if metric == 2:
        Xc = torch.cat([x1.detach().reshape(num_pairs, -1), x2.detach().reshape(num_pairs, -1)], 0)
        Yc = torch.cat([y1.detach().reshape(num_pairs, -1), y2.detach().reshape(num_pairs, -1)], 0)
        ar = torch.arange(num_pairs, device=X.device)
        ratio = ops.lipschitz_pair_ratios(Xc, Yc, ar, ar + num_pairs, eps)
    else:
        dy = (y1 - y2).reshape(num_pairs, -1).norm(dim=1, p=metric).clamp(min=eps)
        dx = (x1 - x2).reshape(num_pairs, -1).norm(dim=1, p=metric).clamp(min=eps)
        ratio = (dy / dx).detach()
    A = torch.quantile(ratio, quantile).clamp(min=eps)
    Bq = torch.quantile(ratio, 1 - quantile)
    invA = 1.0 / A
    res = torch.stack([invA, Bq, torch.maximum(invA, Bq)]).tolist()   # one sync instead of three
    return res[0], res[1], res[2]


def estimate_local_lipschitz_jacobian(model, Z, quantile=0.05, eps=1e-3):
    """The reference's (inverse_lipschitz, lipschitz, bi_lipschitz) triple (utils.py:563-567) on the decoder's LOCAL
    constants instead of finite-pair ratios: per point, the smallest and largest singular values of the exact Jacobian
    (model.decode_jacobian), A = max(quantile(sigma_min, q), eps), B = quantile(sigma_max, 1 - q) (torch.quantile's linear
    rule) -> (1/A, B, max(1/A, B)) as Python floats; (0, 0, 0) for an empty Z."""
    if Z.size(0) == 0:
        return 0.0, 0.0, 0.0
    _, _, s = model.decode_jacobian(Z)
    A = torch.quantile(s[:, -1], quantile).clamp(min=eps)
    Bq = torch.quantile(s[:, 0], 1 - quantile)
    invA = 1.0 / A
    res = torch.stack([invA, Bq, torch.maximum(invA, Bq)]).tolist()
    return res[0], res[1], res[2]


def estimate_local_lipschitz_batched(func, X_list, num_pairs=2000, quantile=0.05, eps=1e-3, use_grad=False):
    """`estimate_local_lipschitz` for MANY sample sets at once (the per-cell loops of lipschitz.py:48-154 call the
    estimator up to 512 times, each with 2 small decodes, 2 sorts and 3 `.item()` syncs).  Here all cells share
    TWO decodes, ONE ratio-kernel launch, ONE batched quantile and ONE device->host copy.  Pair indices are drawn
    exactly like the reference (a fresh seed-0 generator on X.device per cell), so every cell's result equals the
    one-cell call.  Returns a float64 numpy array [n_cells, 3] = (inverse_lipschitz, lipschitz, bi_lipschitz);
    cells with fewer than 2 samples get (0, 0, 0) like the reference."""
    import numpy as np
    out = np.zeros((len(X_list), 3), dtype=np.float64)
    live = [i for i, X in enumerate(X_list) if X.size(0) >= 2]
    if not live:
        return out
    dev = X_list[live[0]].device
    i1s, i2s, offs, off = [], [], [], 0
    for i in live:
        N = X_list[i].size(0)
        gen = torch.Generator(device=dev).manual_seed(0)
        i1s.append(torch.randint(0, N, (num_pairs,), device=dev, generator=gen) + off)
        i2s.append(torch.randint(0, N, (num_pairs,), device=dev, generator=gen) + off)
        offs.append(off)
        off += N
    Xall = torch.cat([X_list[i].detach().reshape(X_list[i].size(0), -1) for i in live], 0)
    i1, i2 = torch.cat(i1s), torch.cat(i2s)
    x1, x2 = Xall[i1], Xall[i2]
    shape_tail = X_list[live[0]].shape[1:]
    with torch.no_grad():                       # our decode needs no autograd graph (use_grad kept for API parity)
        y1 = func(x1.reshape(-1, *shape_tail))
        y2 = func(x2.reshape(-1, *shape_tail))
    P = i1.numel()
    ar = torch.arange(P, device=dev)
    ratio = ops.lipschitz_pair_ratios(torch.cat([x1, x2], 0), torch.cat([y1.reshape(P, -1), y2.reshape(P, -1)], 0),
                                      ar, ar + P, eps).view(len(live), num_pairs)
    q = torch.quantile(ratio, torch.tensor([quantile, 1 - quantile], device=dev), dim=1)     # [2, n_live]
    invA = 1.0 / q[0].clamp(min=eps)
    res = torch.stack([invA, q[1], torch.maximum(invA, q[1])], 1).double().cpu().numpy()     # one sync
    out[live] = res
    return out


def estimate_lipschitz_allpairs(func, X, eps=1e-3, process_group=None, nbins=0, hist_range=(-20.0, 20.0), peer=None,
                                shard_decode=True, quantile=None):
    """All-pairs max / min / mean of |f(x)-f(y)|/|x-y| over every unordered pair (north_star kernel 4).
    With a process group (X replicated on every rank) BOTH stages shard: rank r decodes rows [r*per, (r+1)*per) and the
    outputs are all-gathered; the 64x64 pair tiles are split by range (`tile_range`) and the per-rank statistics combined
    with ONE exchange -- `peer` (a peer.PeerComm: an own all-gather kernel over NVLink peer memory, ~13 us) or one
    torch.distributed all_gather.  Returns dict(max, min, mean, count[, hist]).

    `quantile` = q adds the reference's estimate (utils.py:563-567) over EVERY pair instead of sampled ones: the exact
    quantiles v(q), v(1-q) of the same ratios (ops.lipschitz_allpairs_quantiles: torch.quantile's linear rule, ranks in
    fp64), A = max(v(q), eps), B = v(1-q) -> keys inverse_lipschitz = 1/A, lipschitz = B, bi_lipschitz = max(1/A, B) and
    quantiles = (v(q), v(1-q)); (0, 0, 0) for fewer than 2 points.  Sharded like the statistics, each of the three passes'
    histograms summed with one all_reduce.  One difference from the sampled estimator: its random pairs may draw i == j
    (ratio 1.0 through both clamps), all pairs i < j never do."""
    import torch.distributed as dist
    rank, world = 0, 1
    if process_group is not None or (dist.is_available() and dist.is_initialized()):
        rank, world = dist.get_rank(process_group), dist.get_world_size(process_group)
    N = X.shape[0]
    with torch.no_grad():
        if world > 1 and shard_decode and N >= world:
            per = (N + world - 1) // world
            lo_r, hi_r = min(rank * per, N), min((rank + 1) * per, N)
            Yl = func(X[lo_r:hi_r]) if hi_r > lo_r else None
            tail = tuple(Yl.shape[1:]) if Yl is not None else None
            if tail is None:          # a rank without rows still needs the output shape: decode one row
                tail = tuple(func(X[:1]).shape[1:])
            pad = torch.zeros(per, *tail, dtype=torch.float32, device=X.device)
            if Yl is not None:
                pad[:hi_r - lo_r] = Yl
            if pad.is_cuda:
                full = torch.empty(world * per, *tail, dtype=torch.float32, device=X.device)
                dist.all_gather_into_tensor(full, pad, group=process_group)          # one NCCL call, no concatenation
                Y = full[:N]
            else:
                gathered = [torch.empty_like(pad) for _ in range(world)]
                dist.all_gather(gathered, pad, group=process_group)
                Y = torch.cat(gathered, 0)[:N]
        else:
            Y = func(X)
    nt = ops.lipschitz_num_tiles(N)
    lo, hi = tile_range(nt, rank, world)
    stats, hist = ops.lipschitz_allpairs(X, Y, eps, lo, hi, nbins, *hist_range)
    if world > 1:
        stats, hist = combine_allpairs(stats, hist, process_group, peer)
    mx, mn, sm, cnt = stats.tolist()
    out = dict(max=mx, min=mn, mean=sm / max(cnt, 1.0), count=int(cnt))
    if hist is not None:
        out["hist"] = hist
    if quantile is not None:
        if N < 2:
            out.update(inverse_lipschitz=0.0, lipschitz=0.0, bi_lipschitz=0.0, quantiles=(0.0, 0.0))
            return out
        reduce_hist = None
        if world > 1:
            reduce_hist = lambda h: dist.all_reduce(h, op=dist.ReduceOp.SUM, group=process_group)   # noqa: E731
        v = ops.lipschitz_allpairs_quantiles(X, Y, (quantile, 1.0 - quantile), eps, lo, hi, reduce_hist)[:2].tolist()
        inv = 1.0 / max(v[0], eps)
        out.update(inverse_lipschitz=inv, lipschitz=v[1], bi_lipschitz=max(inv, v[1]), quantiles=(v[0], v[1]))
    return out


def tile_range(num_tiles, rank, world):
    """Contiguous, balanced tile ranges per rank (host logic; unit-tested on CPU)."""
    base, rem = divmod(num_tiles, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def combine_allpairs(stats, hist, process_group=None, peer=None):
    """Combine per-rank [max, min, sum, count] fp64 statistics (+ histogram) with ONE exchange: every rank gathers all
    ranks' statistics (peer-memory all-gather kernel when `peer` is given, else torch.distributed.all_gather) and reduces
    them locally in rank order -- identical results on every rank."""
    import torch.distributed as dist
    if peer is not None:
        allst = peer.allgather(stats.view(torch.float32)).contiguous().view(torch.float64)       # [world, 4] bit-exact
    else:
        outs = [torch.empty_like(stats) for _ in range(dist.get_world_size(process_group))]
        dist.all_gather(outs, stats, group=process_group)
        allst = torch.stack(outs)
    comb = torch.stack([allst[:, 0].max(), allst[:, 1].min(), allst[:, 2].sum(), allst[:, 3].sum()])
    if hist is not None:
        hist = hist.clone()
        dist.all_reduce(hist, op=dist.ReduceOp.SUM, group=process_group)
    return comb, hist
