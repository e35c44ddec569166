#!/usr/bin/env python
"""Cost of top-k / top-p sampling on one B200.

    python tools/sampler_bench.py [--iters 500] [--no-engine]

Kernel level: B = 64 rows, V = 152064 (Qwen2.5), near-uniform (random-init-like) and peaked logits.  Times
prl_sample_logprob_rows alone against prl_sample_logprob_rows + prl_sample_filter_rows with all 64 rows filtered, for
(top_k, top_p) = (50, 0.95) [the reference's eval handle], (-1, 0.95) and (50, 1).  CUDA events around `--iters`
launches after a warm-up, the variants alternated in rounds.  The inputs are L2-warm, as in the engine, where the
sampler has just read the 39 MB of logits that the filter re-reads.

Engine level: DecodeEngine.step() of bench.py's workload (Qwen2.5-7B random-init, 64 slots) with every slot filtered
at (50, 0.95) against none, alternated.

One JSON line, with the GPU name and power limit read in the same run."""
import argparse
import json
import subprocess
import sys
import types
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

CONFIGS = {"k50_p0.95": (50, 0.95), "p0.95": (-1, 0.95), "k50": (50, 1.0)}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def kernel_level(dev, iters, rounds=5):
    from pipelinerl_b200 import _lib
    lib = _lib.load()
    B, V = 64, 152064
    g = torch.Generator().manual_seed(0)
    inputs = {"flat": torch.randn(B, V, generator=g) * 0.05}
    peaked = torch.randn(B, V, generator=g) * 2.0
    peaked[torch.arange(B), torch.randint(0, V, (B,), generator=g)] += 14.0
    inputs["peaked"] = peaked
    inv_t = torch.ones(B, dtype=torch.float32, device=dev)
    greedy = torch.zeros(B, dtype=torch.uint8, device=dev)
    ws = torch.zeros(int(lib.prl_sample_workspace_bytes(B)), dtype=torch.uint8, device=dev)
    ids = torch.zeros(B, dtype=torch.int32, device=dev)
    lps = torch.zeros(B, dtype=torch.float32, device=dev)
    kept = torch.zeros(B, dtype=torch.int32, device=dev)
    out = {}
    for name, cpu_logits in inputs.items():
        logits = cpu_logits.to(dev)
        rows = {c: (torch.full((B,), k, dtype=torch.int32, device=dev), torch.full((B,), p, device=dev))
                for c, (k, p) in CONFIGS.items()}

        def launch(cfg, step):
            _lib.check(lib.prl_sample_logprob_rows(logits.data_ptr(), B, V, inv_t.data_ptr(), greedy.data_ptr(), 7, step,
                                                   ids.data_ptr(), lps.data_ptr(), ws.data_ptr(), ws.numel(), None))
            if cfg is not None:
                tk, tp = rows[cfg]
                _lib.check(lib.prl_sample_filter_rows(logits.data_ptr(), B, V, inv_t.data_ptr(), greedy.data_ptr(),
                                                      tk.data_ptr(), tp.data_ptr(), 7, step, ids.data_ptr(),
                                                      lps.data_ptr(), kept.data_ptr(), None, 0, None))
        variants = [None] + list(CONFIGS)
        for v in variants:                       # warm-up (module load, smem attribute) and the kept-set sizes
            for s in range(20):
                launch(v, s)
        torch.cuda.synchronize()
        kept_by = {}
        for c in CONFIGS:
            launch(c, 0)
            torch.cuda.synchronize()
            kept_by[c] = float(kept.float().mean())
        times = {v: [] for v in variants}
        per_round = max(1, iters // rounds)
        for _ in range(rounds):
            for v in variants:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for s in range(per_round):
                    launch(v, s)
                e1.record()
                torch.cuda.synchronize()
                times[v].append(e0.elapsed_time(e1) / per_round)
        base = sorted(times[None])[len(times[None]) // 2]
        res = {"sampler_only_ms": round(base, 5)}
        for c in CONFIGS:
            med = sorted(times[c])[len(times[c]) // 2]
            res[c] = {"sampler_plus_filter_ms": round(med, 5), "added_ms": round(med - base, 5),
                      "mean_kept": kept_by[c]}
        res["launches_per_variant"] = per_round * rounds
        out[name] = res
    return out


def engine_level(dev, steps=20, rounds=4):
    import bench
    args = types.SimpleNamespace(context=bench.CONTEXT, batch=64, steps=steps * rounds, warmup=3)
    cfg, eng = bench.build_engine(args, dev)
    B = eng.B

    def set_filtered(on):
        eng.top_k_rows.fill_(50 if on else -1)
        eng.top_p_rows.fill_(0.95 if on else 1.0)
        eng._n_filtered = B if on else 0
    for on in (False, True, False):
        set_filtered(on)
        for _ in range(3):
            eng.step()
    torch.cuda.synchronize()
    times = {False: [], True: []}
    for _ in range(rounds):
        for on in (False, True):
            set_filtered(on)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps // 2):
                eng.step()
            e1.record()
            torch.cuda.synchronize()
            times[on].append(e0.elapsed_time(e1) / (steps // 2))
    set_filtered(False)
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    return {"workload": f"Qwen2.5-7B random-init, {B} slots x {args.context}-token context",
            "step_ms_unfiltered": round(med[False], 4), "step_ms_all_filtered_k50_p0.95": round(med[True], 4),
            "added_ms": round(med[True] - med[False], 4),
            "rounds_ms": {"unfiltered": [round(t, 4) for t in times[False]],
                          "filtered": [round(t, 4) for t in times[True]]}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=500)
    ap.add_argument("--no-engine", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sampler_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    from pipelinerl_b200 import _build
    _build.build(verbose=False)
    out = {"gpu": gpu_info(), "note": "inputs L2-warm (as in the engine); medians over alternated rounds",
           "kernel": kernel_level(dev, args.iters)}
    if not args.no_engine:
        out["engine"] = engine_level(dev)
    out["gpu_after"] = gpu_info()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
