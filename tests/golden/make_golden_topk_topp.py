"""Golden for the sampler's top-k / top-p filter: vLLM 0.22's OWN `apply_top_k_top_p_pytorch` + `log_softmax`
(vllm/v1/sample/ops/topk_topp_sampler.py: `forward_native` with logprobs-mode processed_logprobs), run on CPU (the
function is pure torch; it needs vLLM 0.22 importable, no GPU):

    python tests/golden/make_golden_topk_topp.py            -> tests/golden/topk_topp_cases.npz

Rows: near-uniform ('flat', random-init-like), 'peaked' and 'ties' (values on a coarse grid, so the k-th value is
shared) logits at temperatures {0.7, 1.0, 1.3} and (top_k, top_p) in {(50, 0.95) [the reference's eval handle],
(50, 1), (-1, 0.95), (-1, 0.5), (1, 1), (20, 0.3), (V-1, 1)}; the tie rows use the top-k-only configs, where vLLM's
rule and this package's agree on ties.  V = 1000 rows store their logits; V = 152064 rows are regenerated from a torch
CPU seed by oracle.sampling_oracle.synthetic_logits and carry a float64 checksum so that RNG drift fails loudly.

Per row: vLLM's kept count, the smallest kept z (the kept set is {z >= it}), logsumexp of z over the kept set,
processed logprobs at a fixed sample of ids, and the ambiguity band (tokens whose float64 exclusive-above mass lies
within 1e-4 of p: fp32 cumsums in any order may disagree inside it)."""
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent.parent
sys.path.insert(0, str(ROOT))
from oracle.sampling_oracle import ambiguity_band, scaled_logits, synthetic_logits  # noqa: E402

TEMPS = (0.7, 1.0, 1.3)
N_SAMPLE_IDS = 16


def configs(V):
    return [(50, 0.95), (50, 1.0), (-1, 0.95), (-1, 0.5), (1, 1.0), (20, 0.3), (V - 1, 1.0)]


def vllm_row(z: torch.Tensor, top_k: int, top_p: float):
    import vllm
    from vllm.v1.sample.ops.topk_topp_sampler import apply_top_k_top_p_pytorch
    assert vllm.__version__.startswith("0.22"), vllm.__version__
    V = z.numel()
    k = torch.tensor([top_k], dtype=torch.long) if 1 <= top_k < V else None
    p = torch.tensor([top_p], dtype=torch.float32) if top_p < 1.0 else None
    masked = apply_top_k_top_p_pytorch(z.clone()[None], k, p)[0]
    lp = masked.log_softmax(dim=-1, dtype=torch.float32)
    keep = torch.isfinite(masked)
    return keep, lp, torch.logsumexp(masked[keep], 0)


def main():
    rows = []
    stored = []                      # V = 1000 logits, indexed by row["logits_idx"]
    specs = []
    for kind, seed in (("flat", 101), ("peaked", 102)):
        for V in (1000, 152064):
            for T in TEMPS:
                for k, p in configs(V):
                    specs.append((kind, seed + V, V, T, k, p))
    for V in (1000, 152064):
        for k, p in ((50, 1.0), (1, 1.0), (20, 1.0), (V - 1, 1.0)):
            specs.append(("ties", 103 + V, V, 1.0, k, p))
    gen = torch.Generator().manual_seed(7)
    for kind, seed, V, T, k, p in specs:
        logits = synthetic_logits(kind, V, seed)
        z = scaled_logits(logits, T)
        keep, lp, lse = vllm_row(z, k, p)
        kept_ids = torch.nonzero(keep).flatten()
        top = kept_ids[torch.argsort(z[kept_ids], descending=True)][: N_SAMPLE_IDS // 2]
        rest = kept_ids[torch.randint(0, kept_ids.numel(), (N_SAMPLE_IDS - top.numel(),), generator=gen)]
        ids = torch.cat([top, rest])
        idx = -1
        if V <= 1000:
            idx = len(stored)
            stored.append(logits.numpy())
        rows.append(dict(kind=kind, seed=seed, V=V, T=T, k=k, p=p, logits_idx=idx,
                         checksum=float(logits.double().sum()), checksum_abs=float(logits.double().abs().sum()),
                         kept=int(keep.sum()), min_kept_z=float(z[keep].min()), lse=float(lse),
                         band=ambiguity_band(z, k, p), ids=ids.numpy(), lps=lp[ids].numpy()))
        print(f"{kind:6s} V={V:6d} T={T} k={k:6d} p={p:4.2f}: kept {rows[-1]['kept']:6d} band {rows[-1]['band']}")
    out = {k: np.array([r[k] for r in rows]) for k in ("seed", "V", "T", "k", "p", "logits_idx", "checksum",
                                                          "checksum_abs", "kept", "min_kept_z", "lse", "band")}
    out["kind"] = np.array([r["kind"] for r in rows])
    out["ids"] = np.stack([r["ids"] for r in rows]).astype(np.int64)
    out["lps"] = np.stack([r["lps"] for r in rows]).astype(np.float32)
    out["logits"] = np.stack(stored).astype(np.float32)
    dst = Path(__file__).resolve().parent / "topk_topp_cases.npz"
    np.savez_compressed(dst, **out)
    print(f"wrote {dst} ({len(rows)} rows)")


if __name__ == "__main__":
    main()
