"""Oracle for the sampler's top-k / top-p filter with processed logprobs (pipelinerl_b200/csrc/sample_filter.cu).

TEST INFRASTRUCTURE (see oracle/__init__.py).  Torch on CPU.

Restates vLLM 0.22's `apply_top_k_top_p_pytorch` followed by `log_softmax` of the masked logits (the reference's eval
handle samples with top_p 0.95 / top_k 50 and vLLM runs with logprobs-mode processed_logprobs, conf/base.yaml:52-65).
Pinned against vLLM's own function by tests/golden/topk_topp_cases.npz (make_golden_topk_topp.py), checked in
tests/test_sampling_filters.py.

For one row of fp32 logits l at temperature T, z = l * fp32(1/T):
  top-k (1 <= k < V): keep {z >= the k-th largest z}; every tie with the k-th value is kept (vLLM: logits_sort < kth).
  top-p (p < 1): over the top-k survivors, renormalised, keep a token iff the mass of the tokens ranked strictly above
         it is < p (vLLM: ascending cumsum <= 1 - p is dropped, the most likely token is always kept).
  Tie rule (the one deviation): every token tied with the top-p boundary value is kept, so the kept set is always
  {z >= tau}.  vLLM's unstable sort may split such a tie; the goldens hold no exact tie at a top-p boundary.
  processed logprob = z - logsumexp(z over the kept set).
Disabled values, as vLLM validates them: top_k in {-1, 0} or >= V, top_p == 1.  Greedy rows ignore both filters.
"""
from __future__ import annotations

import torch


def filter_active(top_k: int, top_p: float, V: int) -> bool:
    return 1 <= top_k < V or top_p < 1.0


def scaled_logits(logits: torch.Tensor, temperature: float) -> torch.Tensor:
    """z = logits * (1/T) with the fp32 multiply the sampler kernels use."""
    inv = torch.tensor(1.0 / temperature, dtype=torch.float32)
    return logits.float() * inv


def kept_mask(z: torch.Tensor, top_k: int, top_p: float) -> torch.Tensor:
    """Boolean mask of the kept set of one row of scaled logits z [V]."""
    V = z.numel()
    zs = torch.sort(z, descending=True).values
    tau = zs[-1]
    if 1 <= top_k < V:
        tau = zs[top_k - 1]
    if top_p < 1.0:
        surv = zs[zs >= tau].double()
        w = torch.exp(surv - surv[0])
        above = (torch.cumsum(w, 0) - w) / w.sum()         # mass ranked strictly above, descending order
        last = int(torch.nonzero(above < top_p).max())     # row 0 has 0 above: always kept
        tau = torch.maximum(tau, zs[last])
    return z >= tau


def processed_logprobs(z: torch.Tensor, keep: torch.Tensor) -> torch.Tensor:
    """log_softmax of the masked row: z - logsumexp(z[keep]) on the kept set, -inf elsewhere (float64 inside)."""
    zd = z.double()
    lse = torch.logsumexp(zd[keep], 0)
    return torch.where(keep, zd - lse, torch.full_like(zd, -float("inf"))).to(z.dtype)


def ambiguity_band(z: torch.Tensor, top_k: int, top_p: float, tol: float = 1e-4) -> int:
    """Tokens among the top-k survivors whose exclusive-above mass (float64) lies within `tol` of p: fp32 cumulative
    sums in any order may legitimately place the top-p boundary anywhere inside this band."""
    if not top_p < 1.0:
        return 0
    V = z.numel()
    zs = torch.sort(z.double(), descending=True).values
    if 1 <= top_k < V:
        zs = zs[zs >= zs[top_k - 1]]
    w = torch.exp(zs - zs[0])
    above = (torch.cumsum(w, 0) - w) / w.sum()
    return int(((above - top_p).abs() <= tol).sum())


def synthetic_logits(kind: str, V: int, seed: int) -> torch.Tensor:
    """Rows of the golden (regenerated from the seed at V = 152064): 'flat' ~ a random-init model's near-uniform
    logits, 'peaked' ~ a trained model's, 'ties' ~ values on a coarse grid, so the k-th value is shared."""
    g = torch.Generator().manual_seed(seed)
    if kind == "flat":
        return torch.randn(V, generator=g) * 0.05
    if kind == "peaked":
        x = torch.randn(V, generator=g) * 2.0
        spikes = torch.randint(0, V, (8,), generator=g)
        x[spikes] += torch.linspace(14.0, 6.0, 8)
        return x
    if kind == "ties":
        return torch.round(torch.randn(V, generator=g) * 4.0) / 4.0
    raise KeyError(kind)
