#!/usr/bin/env python
"""bench.py — headline measurement of the hot path (contract in the task statement / DESIGN.md §Measurement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Metric: rollout tokens/s (the reference's actor/output_tokens_per_second, pipelinerl/actor.py:98-106) of the
sampler's token step on random-init Qwen2.5-7B: 64 running sequences per GPU (actor.llm_max_rollouts,
conf/base.yaml:17,63), synthetic 8192-token prompts already in the paged KV cache, temperature 1.
A "step" = one token for each of the 64 sequences (one pass of hot path 1).  N > 1: one engine replica per
GPU (SURVEY §8e: the token step shards as replicas only, no data-path collective) -> weak scaling.

Under torchrun (N >= 2) the same run then re-partitions the N GPUs into the actor-learner split of the north star
(`components.pipeline`, tools/split_bench.py): 1+1 at N=2, 3+1 at N=4, 6+2 and 4+4 at N=8 -- samplers keep
generating while data-parallel learners train and push weights after every optimizer step; rollout tokens/s while
training, trainer tokens/s and steps/s, DP exchange ms, push ms, STALL ms, `bytes_identical`, `dp_equals_single`.
At N=1, `components.vllm_baseline` runs the same workload on vLLM 0.22 + FlashInfer (the engine the reference serves
rollouts with) in a subprocess on the same box.

ONE JSON line on stdout (rank 0).  Extra keys: roofline (dominant kernel = paged decode attention),
cpu_baseline (oracle port on the host cores, bounded sample), components (trainer side: fused AdamW and PG-loss
tail on 7B-sized inputs, and `trainer_step` = hot path 2 end to end on Qwen2.5-7B: 2 x 16 384-token micro-batches
through rl_step -> native backward -> fused AdamW; tools/train_bench.py).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

CONTEXT = 8192          # synthetic prompt tokens per sequence (BASELINE.json configs[1])
BATCH = 64              # running sequences per engine (conf/base.yaml:63 max-num-seqs)
METRIC = "rollout_tokens_per_s"
UNIT = "tokens/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--context", type=int, default=CONTEXT)
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--no-components", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pipeline", action="store_true", help="N >= 2: skip the inference + learner split run")
    ap.add_argument("--no-vllm", action="store_true", help="N = 1: skip the vLLM 0.22 A/B subprocess")
    ap.add_argument("--no-seq-parallel", action="store_true", help="N = 2: skip the sequence-parallel trainer step")
    ap.add_argument("--no-rollout", action="store_true", help="N = 1: skip the full-rollout run through the plugin API")
    ap.add_argument("--rollout-tokens", type=int, default=8192, help="max_tokens of the full-rollout component")
    ap.add_argument("--splits", default="", help="learner counts of the split runs, e.g. '2,4' (default: by N)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (sampled ids, their logprobs, the logits) as DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


def workload_config(args, n_gpus):
    return {"workload": f"Qwen2.5-7B random-init token step, {args.batch} seqs/GPU x {args.context}-token synthetic "
                        f"prompts in paged KV, temperature 1.0 (BASELINE.json configs[1], sampler side)",
            "batch_per_gpu": args.batch, "context": args.context, "parallelism": f"replicas x{n_gpus}",
            "lm_head": "fp32-equivalent (bf16 hi + bf16 lo operand streams, vllm_quantization.py:266-278)",
            "l2": "inputs_exceed_l2 (weights 16.3 GB + KV 30 GB read per step)", "cuda_graph": True}


# ----------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(r[1]) for r in self.rows if len(r) > 2 and r[1].isdigit())
        mx = [int(r[2]) for r in self.rows if len(r) > 2 and r[2].isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def ncu_traffic_bytes(algorithmic_bytes: int):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture
    (profiles/r1_attn_full_raw.csv: dram__bytes_read.sum 1.08266 GB + dram__bytes_write.sum 0.9 MB at B=64, S=8240 -> ratio
    to the algorithmic bytes 1.0004), scaled to the bytes of the launch timed here."""
    f = ROOT / "profiles" / "ncu_traffic.json"
    try:
        ratio = float(json.loads(f.read_text())["paged_attn_decode_kernel"]["traffic_over_algorithmic"])
    except Exception:  # noqa: BLE001
        return None
    return int(algorithmic_bytes * ratio)


def measured_peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        d = json.loads(f.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------
def build_engine(args, dev):
    import torch
    from pipelinerl_b200.engine import DecodeEngine, PAGE_SIZE
    from pipelinerl_b200.model import ModelConfig, ParamArena
    cfg = ModelConfig.qwen2_5_7b(fp32_head=True)   # the reference computes lm_head in fp32 on the sampler
    arena = ParamArena(cfg, dev).init_random(seed=42)
    # every step of the run (warm-up, the launch count, the timed and the end-to-end loops) must fit in max_new_tokens:
    # a slot that reaches it finishes and stops reading its KV, and the steps after that no longer run the workload
    steps_run = max(args.warmup, 3) + 1 + 2 * args.steps
    room = max(256 + args.steps + args.warmup * 2 + 64, steps_run + 1)
    eng = DecodeEngine(cfg, arena, max_batch=args.batch, max_seq_len=args.context + room, max_new_tokens=room,
                       eos_id=-1, seed=42, device=dev, use_cuda_graph=True)
    # synthetic rollout state: every slot has an args.context-token prompt resident in the KV cache
    g = torch.Generator(device=dev).manual_seed(1234)
    flat = eng.kv_cache
    step = 1 << 28
    for s in range(0, flat.numel(), step):
        n = min(step, flat.numel() - s)
        flat[s:s + n] = (torch.randn(n, generator=g, device=dev, dtype=torch.float32) * 0.5).to(torch.bfloat16)
    B, mb = eng.B, eng.max_blocks
    bt = torch.arange(1, 1 + B * mb, dtype=torch.int32, device=dev).view(B, mb)
    eng.block_table.copy_(bt)
    eng.free_pages.clear()
    eng.prompt_len.fill_(args.context)
    eng.positions.fill_(args.context)
    eng.seq_lens.fill_(args.context + 1)
    eng.max_new_t.fill_(room)
    eng.gen_count.zero_()
    eng.active.fill_(1)
    eng.tokens.copy_(torch.randint(0, 151643, (B,), generator=torch.Generator().manual_seed(1000)).int())
    eng.temperature, eng.greedy, eng.ignore_eos = 1.0, False, True
    return cfg, eng


def algorithmic_bytes(cfg, B, S):
    w_body = 2 * sum(n for n in [cfg.num_layers * (cfg.qkv_size * cfg.hidden_size + cfg.hidden_size * cfg.q_size +
                                                   3 * cfg.intermediate_size * cfg.hidden_size)])
    w_head = (4 if cfg.fp32_head else 2) * cfg.vocab_size * cfg.hidden_size   # hi + lo streams = an fp32 weight's bytes
    kv_per_layer = B * S * 2 * cfg.num_kv_heads * cfg.head_dim * 2
    return w_body + w_head, kv_per_layer


DUMP_LOGITS_BYTES = 48 << 20    # the dump stays under 64 MB at any --batch


def dump_outputs(out_dir: Path, eng, h_ids, h_lp):
    """The last end-to-end step's results as float arrays: the sampled ids and logprobs the host received, and the fp32
    logits they were sampled from (all rows, or a fixed seeded sample of rows when they exceed DUMP_LOGITS_BYTES).
    The inputs are seeded, so two builds run with the same arguments can be compared output for output."""
    import numpy as np
    import torch
    out_dir.mkdir(parents=True, exist_ok=True)
    np.save(out_dir / "sampled_ids.npy", h_ids.numpy().astype(np.float64))
    np.save(out_dir / "sampled_logprobs.npy", h_lp.numpy().astype(np.float32))
    rows = np.arange(eng.B)
    max_rows = DUMP_LOGITS_BYTES // (4 * eng.logits.shape[1])
    if eng.B > max_rows:
        rows = np.sort(np.random.default_rng(0).choice(eng.B, max_rows, replace=False))
    np.save(out_dir / "logits_rows.npy", rows.astype(np.float64))
    np.save(out_dir / "logits.npy", eng.logits.index_select(0, torch.from_numpy(rows).to(eng.logits.device)).cpu().numpy())


def run_ours(args):
    import torch
    import torch.distributed as dist
    from pipelinerl_b200 import _lib
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        # keep stdout to the single JSON line: NCCL writes its version banner / warnings to stdout unless told otherwise
        os.environ["NCCL_DEBUG"] = "WARN"
        os.environ["NCCL_DEBUG_FILE"] = "/dev/stderr"
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    _lib.load()
    cfg, eng = build_engine(args, dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    launches0 = _lib.launch_count()
    for _ in range(max(args.warmup, 3)):
        eng.step()
    torch.cuda.synchronize()
    # launches per step: model kernels are replayed from the graph (counted once at capture), so count one
    # eager enqueue of the same sequence
    c0 = _lib.launch_count()
    eng._step_kernels()
    eng._sample_and_advance()
    eng.step_count += 1
    torch.cuda.synchronize()
    launches_per_step = _lib.launch_count() - c0

    # ---- device-resident timing ----
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        eng.step()
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    clk = clocks.stop() if rank == 0 else None

    # ---- end-to-end through the host-facing call: token ids in from pinned host memory, ids + logprobs out ----
    h_tok = torch.zeros(eng.B, dtype=torch.int32).pin_memory()
    h_ids = torch.zeros(eng.B, dtype=torch.int32).pin_memory()
    h_lp = torch.zeros(eng.B, dtype=torch.float32).pin_memory()
    h_tok.copy_(eng.tokens)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng.tokens.copy_(h_tok, non_blocking=True)
        eng.step()
        h_ids.copy_(eng.sampled, non_blocking=True)
        h_lp.copy_(eng.sampled_lp, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        h_tok.copy_(h_ids)
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    if rank == 0 and args.dump_outputs:
        dump_outputs(Path(args.dump_outputs), eng, h_ids, h_lp)

    times = torch.tensor([ms, e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms, e2e_ms = times.tolist()
    tokens = eng.B * args.steps * world
    value = tokens / (ms / 1e3)
    e2e_value = tokens / (e2e_ms / 1e3)

    # ---- roofline of the dominant kernel (paged decode attention), timed alone with events on its stream ----
    import math
    w_bytes, kv_layer_bytes = algorithmic_bytes(cfg, eng.B, args.context + 1)
    lib = _lib.load()
    st = _lib.stream_ptr()

    def attn_all_layers():
        for l in range(cfg.num_layers):
            _lib.check(lib.prl_paged_attn_decode(eng.q.data_ptr(), eng.kv_cache.data_ptr(), eng.n_pages, cfg.num_layers, l,
                                                 eng.block_table.data_ptr(), eng.max_blocks, eng.seq_lens.data_ptr(), eng.B,
                                                 cfg.num_q_heads, cfg.num_kv_heads, cfg.head_dim, 64, eng.attn_splits,
                                                 1.0 / math.sqrt(cfg.head_dim), eng.attn_out.data_ptr(),
                                                 eng.attn_ws.data_ptr(), eng.attn_ws.numel(), st))
    attn_all_layers()
    torch.cuda.synchronize()
    ev0.record()
    reps = 3
    for _ in range(reps):
        attn_all_layers()
    ev1.record()
    torch.cuda.synchronize()
    attn_ms = ev0.elapsed_time(ev1) / (reps * cfg.num_layers)
    peak, peak_src = measured_peaks()
    seq_now = int(eng.seq_lens[0].item())
    kv_bytes = eng.B * seq_now * 2 * cfg.num_kv_heads * cfg.head_dim * 2
    achieved = kv_bytes / (attn_ms / 1e3) / 1e9
    step_bytes = w_bytes + cfg.num_layers * kv_bytes
    roofline = {"kernel": "paged_attn_decode_kernel(+combine)", "bound": "hbm", "achieved": round(achieved, 1),
                "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": round(achieved / peak, 4),
                "traffic": ncu_traffic_bytes(kv_bytes), "traffic_source": "ncu --set full dram__bytes_read.sum + "
                "dram__bytes_write.sum of this kernel (profiles/r1_attn_full_raw.csv: read 1.0004 x, read+write 1.0046 x algorithmic), scaled to this launch",
                "launch_ms": round(attn_ms, 4), "algorithmic_bytes_per_launch": kv_bytes,
                "share_of_step": round(attn_ms * cfg.num_layers / (ms / args.steps), 4),
                "whole_step": {"algorithmic_bytes": step_bytes,
                               "achieved_GBs": round(step_bytes / (ms / args.steps / 1e3) / 1e9, 1),
                               "frac": round(step_bytes / (ms / args.steps / 1e3) / 1e9 / peak, 4)}}

    out = {"metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps,
           "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 4), "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
           "config": workload_config(args, world),
           "e2e": {"value": round(e2e_value, 1), "unit": UNIT, "h2d_bytes_per_step": eng.B * 4,
                   "d2h_bytes_per_step": eng.B * 8, "ms_per_step": round(e2e_ms / args.steps, 4)},
           "gpu_launches": int(launches_per_step * args.steps), "launches_per_step": int(launches_per_step),
           "clocks": clk, "roofline": roofline, "impl": "ours"}

    if rank == 0 and not args.no_components:
        out["components"] = bench_components(dev, peak)
    if rank == 0 and world == 1 and not args.no_components:
        # hot path 2 end to end (rl_step -> backward -> fused AdamW) on the same model: needs the whole GPU, and runs in a
        # CHILD process (tools/train_bench.py) so that nothing it does can cost the headline line
        import gc
        del eng, attn_all_layers
        gc.collect()
        torch.cuda.empty_cache()
        out["components"]["trainer_step"] = run_tool(["tools/train_bench.py", "--steps", "2", "--warmup", "1"], 600)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(args, budget_s=25.0)
    if rank == 0 and world == 1 and not args.no_components and not args.no_rollout:
        # whole rollouts through the plugin API: prefill + decode growing 8192 -> 16384 (not a static-state microbench)
        out["components"]["rollout_full"] = run_tool(["tools/rollout_bench.py", "--max-tokens", str(args.rollout_tokens)], 600)
    if rank == 0 and world == 1 and not args.no_components and not args.no_vllm:
        out.setdefault("components", {})["vllm_baseline"] = vllm_baseline(args)
    if world > 1 and not args.no_components and not args.no_pipeline:
        # ---- the actor-learner split on the same N GPUs (north star: N inference + (8 - N) learner GPUs) ----
        import gc
        try:
            del eng, attn_all_layers
        except NameError:
            pass
        gc.collect()
        torch.cuda.empty_cache()
        out.setdefault("components", {})["pipeline"] = run_pipeline_splits(args, world, rank, out)
        if world == 2 and not args.no_seq_parallel:
            # the sequence-parallel learner on the same two GPUs: both ranks share every 16384-token row
            sp = run_seq_parallel_trainer(world, rank)
            if rank == 0:
                out["components"]["trainer_step_seq_parallel_2"] = sp
    if rank == 0:
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def default_splits(world: int) -> list[int]:
    """learner counts per world size: 1+1 (N=2), 3+1 (N=4), 6+2 and 4+4 (N=8: BASELINE.json configs[1] and [2])"""
    if world >= 8:
        return [2, 4]
    return [1]


def run_pipeline_splits(args, world, rank, headline):
    """All ranks.  Every rank runs its part of a split in a CHILD process (tools/split_bench.py with this rank's
    RANK / LOCAL_RANK / WORLD_SIZE and a fresh rendezvous port): a crash, a CUDA error or a hang inside the split can only
    cost the component -- the parent ranks keep their process group, time the child out, and rank 0 still prints the
    headline line."""
    import torch.distributed as dist
    splits = [int(x) for x in args.splits.split(",") if x] or default_splits(world)
    splits = [m for m in splits if 1 <= m < world]
    results = {"note": "samplers generate (64 seqs x 8192-token context each) WHILE the learners train 2 x 16384-token "
                       "micro-batches per learner per optimizer step and push weights after every step; "
                       "fp32-equivalent lm_head on samplers and learners; each split runs in child processes of the ranks"}
    base_port = int(os.environ.get("MASTER_PORT", "29500"))
    for k, m in enumerate(splits):
        key = f"{world - m}+{m}"
        # a fresh rendezvous for the children: rank 0's child hosts the store itself (the torchrun agent's store, which
        # TORCHELASTIC_USE_AGENT_STORE points the parents at, listens on the parents' port only)
        env = {k_: v for k_, v in os.environ.items() if not k_.startswith("TORCHELASTIC_")}
        env.update(MASTER_PORT=str(base_port + 101 + k), NCCL_DEBUG="WARN", NCCL_DEBUG_FILE="/dev/stderr")
        cmd = [sys.executable, str(ROOT / "tools" / "split_bench.py"), "--learners", str(m), "--updates", "3",
               "--context", str(args.context), "--batch", str(args.batch)]
        t0 = time.time()
        res = None
        try:
            done = subprocess.run(cmd, capture_output=True, text=True, timeout=420, env=env)
            lines = [l for l in done.stdout.splitlines() if l.startswith("{")]
            if done.returncode == 0 and lines:
                res = json.loads(lines[-1])
            elif rank == 0 or done.returncode != 0:
                res = {"error": f"rank {rank}: rc={done.returncode}: {(done.stderr or done.stdout)[-400:]}"}
        except subprocess.TimeoutExpired:
            res = {"error": f"rank {rank}: split timed out after 420 s"}
        except Exception as e:  # noqa: BLE001
            res = {"error": f"rank {rank}: {type(e).__name__}: {str(e)[:300]}"}
        if rank == 0:
            if isinstance(res, dict):
                res["wall_s"] = round(time.time() - t0, 1)
            results[key] = res
        dist.barrier()          # the parents stay in step between splits
    return results if rank == 0 else None


def run_seq_parallel_trainer(world, rank):
    """All ranks (N = 2).  tools/train_bench.py --seq-parallel 2 in child processes with a fresh rendezvous, like the splits:
    the 7B trainer step of `components.trainer_step` (2 x 16384-token rows per optimizer step) with the two ranks holding
    half of every row each (K / V all-gather + dK / dV reduce-scatter per layer, sharded AdamW exchange)."""
    import torch.distributed as dist
    env = {k_: v for k_, v in os.environ.items() if not k_.startswith("TORCHELASTIC_")}
    env.update(MASTER_PORT=str(int(os.environ.get("MASTER_PORT", "29500")) + 171), NCCL_DEBUG="WARN", NCCL_DEBUG_FILE="/dev/stderr")
    cmd = [sys.executable, str(ROOT / "tools" / "train_bench.py"), "--seq-parallel", str(world), "--steps", "2", "--warmup", "1"]
    t0 = time.time()
    try:
        done = subprocess.run(cmd, capture_output=True, text=True, timeout=420, env=env)
        lines = [l for l in done.stdout.splitlines() if l.startswith("{")]
        if done.returncode == 0 and (lines or rank != 0):
            res = json.loads(lines[-1]) if lines else {}
        else:
            res = {"error": f"rank {rank}: rc={done.returncode}: {(done.stderr or done.stdout)[-400:]}"}
    except subprocess.TimeoutExpired:
        res = {"error": f"rank {rank}: timed out after 420 s"}
    except Exception as e:  # noqa: BLE001
        res = {"error": f"rank {rank}: {type(e).__name__}: {str(e)[:300]}"}
    if isinstance(res, dict):
        res["child_process_wall_s"] = round(time.time() - t0, 1)
    dist.barrier()
    return res if rank == 0 else None


def run_tool(argv, timeout_s):
    """one of tools/*.py in a child process -> its last JSON line (or an error record); the GPU must be free"""
    t0 = time.time()
    try:
        res = subprocess.run([sys.executable, str(ROOT / argv[0]), *argv[1:]], capture_output=True, text=True, timeout=timeout_s,
                             env=dict(os.environ, WORLD_SIZE="1", RANK="0", LOCAL_RANK=os.environ.get("LOCAL_RANK", "0")))
        lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
        if res.returncode != 0 or not lines:
            return {"error": f"rc={res.returncode}: {(res.stderr or res.stdout)[-400:]}", "wall_s": round(time.time() - t0, 1)}
        out = json.loads(lines[-1])
        out["child_process_wall_s"] = round(time.time() - t0, 1)     # incl. interpreter start-up and model initialisation
        return out
    except subprocess.TimeoutExpired:
        return {"error": f"timeout after {timeout_s} s", "child_process_wall_s": round(time.time() - t0, 1)}
    except Exception as e:  # noqa: BLE001
        return {"error": f"{type(e).__name__}: {str(e)[:300]}"}


def vllm_baseline(args):
    """Same workload on vLLM 0.22 + FlashInfer sm_100 (the engine family the reference serves rollouts with; it pins
    0.18.1) on this box, in a subprocess (tools/vllm_baseline.py): a LIBRARY baseline for the A/B, not product code."""
    import gc
    import torch
    gc.collect()
    torch.cuda.empty_cache()
    env = dict(os.environ, BATCH=str(args.batch), CTX=str(args.context))
    t0 = time.time()
    try:
        res = subprocess.run([sys.executable, str(ROOT / "tools" / "vllm_baseline.py")], capture_output=True, text=True,
                             timeout=420, env=env)
        lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
        if res.returncode != 0 or not lines:
            return {"error": f"rc={res.returncode}: {(res.stderr or res.stdout)[-300:]}", "wall_s": round(time.time() - t0, 1)}
        out = json.loads(lines[-1])
        out["wall_s"] = round(time.time() - t0, 1)
        return out
    except subprocess.TimeoutExpired:
        return {"error": "timeout after 420 s", "wall_s": round(time.time() - t0, 1)}
    except Exception as e:  # noqa: BLE001
        return {"error": f"{type(e).__name__}: {str(e)[:200]}"}


def bench_components(dev, peak):
    """Trainer-side kernels on Qwen2.5-7B-sized inputs (informational; the headline is the token step)."""
    import torch
    import ctypes as C
    from pipelinerl_b200 import _lib
    lib = _lib.load()
    res = {}
    torch.cuda.empty_cache()
    free = torch.cuda.mem_get_info(dev)[0]
    # fused AdamW: 28 B/param; use as many parameters as fit (7.62e9 needs 122 GB with state)
    n = int(min(7.616e9, (free - 8e9) / 18)) // 4096 * 4096
    try:
        master = torch.zeros(n, device=dev)
        m = torch.zeros(n, device=dev)
        v = torch.zeros(n, device=dev)
        grad = torch.full((n,), 1e-3, dtype=torch.bfloat16, device=dev)
        shadow = torch.zeros(n, dtype=torch.bfloat16, device=dev)
        offs = torch.tensor([0, n], dtype=torch.int64, device=dev)
        nd = torch.zeros(1, dtype=torch.uint8, device=dev)
        ws = torch.zeros(int(lib.prl_adamw_workspace_bytes()), dtype=torch.uint8, device=dev)
        gn = torch.zeros(1, device=dev)
        a = _lib.AdamwArgs()
        a.n, a.master, a.exp_avg, a.exp_avg_sq, a.grad, a.grad_is_bf16 = n, master.data_ptr(), m.data_ptr(), v.data_ptr(), grad.data_ptr(), 1
        a.param_bf16, a.param_bf16_lo, a.tensor_offsets, a.tensor_no_decay, a.n_tensors = shadow.data_ptr(), None, offs.data_ptr(), nd.data_ptr(), 1
        a.lr, a.beta1, a.beta2, a.eps, a.weight_decay, a.max_grad_norm, a.grad_scale = 1e-6, 0.9, 0.999, 1e-8, 0.01, 0.3, 1.0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for i in range(2):
            a.step = i + 1
            _lib.check(lib.prl_adamw_step(C.byref(a), gn.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream_ptr()))
        torch.cuda.synchronize()
        e0.record()
        for i in range(3):
            a.step = i + 3
            _lib.check(lib.prl_adamw_step(C.byref(a), gn.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream_ptr()))
        e1.record()
        torch.cuda.synchronize()
        t = e0.elapsed_time(e1) / 3
        gbs = n * 30 / (t / 1e3) / 1e9  # 28 B/param update + 2 B/param gradient re-read by the norm pass
        res["adamw"] = {"params": n, "ms": round(t, 3), "GBs": round(gbs, 1), "frac_of_hbm_peak": round(gbs / peak, 4),
                        "bytes_per_param": 30, "ms_for_7.616B": round(t * 7.616e9 / n, 2)}
        del master, m, v, grad, shadow
    except RuntimeError as e:  # pragma: no cover
        res["adamw"] = {"error": str(e)[:200]}
    torch.cuda.empty_cache()
    # PG-loss tail on a 4M-token packed row (a step's worth of micro-batches fused): 48 B/token
    T = 1 << 22
    new_lp = -torch.rand(T - 1, device=dev)
    ent = torch.rand(T - 1, device=dev)
    cols = {k: torch.rand(T, device=dev) for k in ("rewards", "advantages", "ref_logprobs", "old_logprobs", "overflow")}
    cols["group_tokens"] = torch.full((T,), 100.0, device=dev)
    cols["num_labels"] = torch.full((T,), 50.0, device=dev)
    labels = torch.randint(0, 1000, (T,), device=dev)
    b = _lib.PgBatch()
    b.T, b.new_logprobs, b.entropy, b.labels, b.num_sequences = T, new_lp.data_ptr(), ent.data_ptr(), labels.data_ptr(), 1
    for k, t_ in cols.items():
        setattr(b, k, t_.data_ptr())
    c = _lib.PgConfig()
    c.policy_loss, c.use_advantages, c.epsilon_low, c.epsilon_high, c.clamp_log_ratio_ref_new_value, c.batch_size = 0, 1, 0.02, 0.02, 5.0, 1024.0
    loss = torch.zeros(1, device=dev)
    dlp = torch.zeros(T - 1, device=dev)
    stats = torch.zeros(32, dtype=torch.float64, device=dev)
    flags = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = torch.zeros(int(lib.prl_pg_workspace_bytes(0)), dtype=torch.uint8, device=dev)
    import ctypes as C2
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def call():
        _lib.check(lib.prl_pg_loss_fwd_bwd(C2.byref(b), C2.byref(c), loss.data_ptr(), dlp.data_ptr(), None, stats.data_ptr(),
                                           flags.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream_ptr()))
    flush = torch.zeros(256 << 20, dtype=torch.uint8, device=dev)
    call()
    tt = 0.0
    for _ in range(5):
        flush.add_(1)  # L2 flush between timed iterations
        e0.record()
        call()
        e1.record()
        torch.cuda.synchronize()
        tt += e0.elapsed_time(e1)
    t = tt / 5
    gbs = (T * 48) / (t / 1e3) / 1e9
    res["pg_loss_tail"] = {"tokens": T, "ms": round(t, 4), "GBs": round(gbs, 1), "frac_of_hbm_peak": round(gbs / peak, 4),
                           "bytes_per_token": 48, "l2": "flushed between iterations"}
    return res


# ----------------------------------------------------------------------------------------------
def cpu_port_step_time(args, n_layers_sample: int, threads: int, budget_s: float):
    """Time the oracle port (oracle/decode_oracle.OracleBatchedStep) on the host cores: `n_layers_sample`
    of the 28 identical layers + the lm_head, at the bench's batch and context."""
    import torch
    from oracle.decode_oracle import OracleBatchedStep
    from pipelinerl_b200.model import ModelConfig
    torch.set_num_threads(threads)
    cfg = ModelConfig.qwen2_5_7b()
    B, S = args.batch, args.context
    g = torch.Generator().manual_seed(0)

    def rnd(*shape, std=0.02):
        return (torch.randn(*shape, generator=g) * std).to(torch.bfloat16).float()
    H, I = cfg.hidden_size, cfg.intermediate_size
    layers, kv = [], []
    for _ in range(n_layers_sample):
        layers.append({"input_layernorm.weight": torch.ones(H), "qkv_proj.weight": rnd(cfg.qkv_size, H),
                       "qkv_proj.bias": torch.zeros(cfg.qkv_size), "o_proj.weight": rnd(H, cfg.q_size),
                       "post_attention_layernorm.weight": torch.ones(H), "gate_up_proj.weight": rnd(2 * I, H),
                       "down_proj.weight": rnd(H, I)})
        kv.append((rnd(B, S, cfg.num_kv_heads, cfg.head_dim, std=0.5), rnd(B, S, cfg.num_kv_heads, cfg.head_dim, std=0.5)))
    embed = rnd(4096, H)  # only the gathered rows matter
    head = rnd(cfg.vocab_size, H)
    tokens = torch.randint(0, 4096, (B,), generator=g)
    pos = torch.full((B,), S)
    body = OracleBatchedStep(cfg, embed, layers, torch.ones(H), head[:1], kv)  # head timed separately below
    t0 = time.perf_counter()
    body.step(tokens, pos)
    t_body = time.perf_counter() - t0
    x = embed[tokens]
    t0 = time.perf_counter()
    lp = torch.log_softmax(x @ head.t(), -1)
    ids = lp.argmax(-1)
    _ = lp.gather(1, ids[:, None])
    t_head = time.perf_counter() - t0
    step_s = t_body / n_layers_sample * cfg.num_layers + t_head
    return step_s, t_body, t_head


def cpu_baseline(args, budget_s=25.0):
    threads = os.cpu_count() or 1
    step_s, t_body, t_head = cpu_port_step_time(args, 1, threads, budget_s)
    return {"value": round(args.batch / step_s, 3), "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"oracle/decode_oracle.OracleBatchedStep (torch fp32 CPU): 1 of 28 identical layers timed "
                      f"({t_body:.2f} s) x28 + fp32 lm_head/logprob/argmax ({t_head:.2f} s), batch {args.batch}, "
                      f"context {args.context}", "s_per_step": round(step_s, 3)}


def run_reference(args):
    """Reference arm for this tier: the reference's CPU implementation of the path = the oracle port (the
    reference itself delegates the token step to vLLM on a GPU and cannot run on host cores); all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    vals = []
    for _ in range(max(1, min(args.steps, 2))):
        step_s, t_body, t_head = cpu_port_step_time(args, 1, threads, 25.0)
        vals.append(step_s)
    step_s = sum(vals) / len(vals)
    value = args.batch / step_s
    out = {"metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": len(vals),
           "warmup": 0, "ms_per_step": round(step_s * 1e3, 1), "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args, world),
           "impl": "reference",
           "cpu_baseline": {"value": round(value, 3), "unit": UNIT, "cores": threads, "kind": "port",
                            "sample": "oracle port, 1 of 28 layers x28 + lm_head per step; each step a bounded sample"},
           "e2e": {"value": round(value, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
