"""Headline benchmark: GRPO episodes/s on Qwen2.5-1.5B (BASELINE.json config 2).

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference ...                      (the unmodified reference; see DESIGN.md)
  python bench.py ... --dump-outputs DIR                    (also write the last timed update's outputs; see dump_outputs)

Batch: the default is ``--mini-batches 8`` = 4 x 8 x 8 = 256 prompts (x 4 samples = 1024 sequences) per rank per update
-- the reference's arithmetic with ``num_mini_batches`` halved from 16 -- so that the driver's ``--steps 20 --warmup 5`` (25 full
updates) finishes inside its per-run limit at every N; ``global_batch`` in ``config`` says what was run and is the same for
the 1-GPU bench and the 1/2/4/8 scaling runs.  ``--mini-batches 16`` is the reference's own 512 prompts per rank
(BASELINE.md has that number too).

One *step* = one full GRPO update through the public API (``GRPOTrainer.train_one_update``): in-process
rollout of ``prompts_per_rank x 4`` samples with up to 1500 response tokens on the sm_100a sampler,
DeBERTa-v3-large reward scoring, policy+ref log-prob pass, advantage estimation, and the
mini-batch x micro-batch optimisation phase with the LoRA(r=64)+embed+lm_head AdamW step -- nothing is
skipped or cached.  ``value`` = global episodes (prompts) per second, device-timed with CUDA events
between barriers, max over ranks.  ``e2e`` is the same quantity timed on the host around the same calls,
including the pinned-host -> device copy of each step's prompts and the device -> host read of the
step's metrics.  Weights are random-init of the named architectures and prompts are synthetic
hh-rlhf-shaped token ids (no network on the benchmark box); with random weights no sequence emits EOS, so
every response runs to the full ``response_length``.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# The only throughput the reference publishes: README.md:36 "~1 s/episode" on 1 x A100-40G with real weights (BASELINE.md
# section 1).  Different hardware, real (EOS-terminated, shorter) responses: context, not a like-for-like ratio.
BASELINE_EPISODES_PER_S = 1.0


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mini-batches", type=int, default=8,
                    help="num_mini_batches: prompts per rank per update = 4 x 8 x this (8 -> 256; the reference's 16 -> 512)")
    ap.add_argument("--response-length", type=int, default=1500)
    ap.add_argument("--samples", type=int, default=4)
    ap.add_argument("--model", default="1.5b", choices=["tiny", "1.5b", "7b"])
    ap.add_argument("--comm", default="fused", choices=["fused", "nccl"])
    ap.add_argument("--rollout-dtype", default="bf16")
    ap.add_argument("--kv-dtype", default="fp8", choices=["bf16", "fp8"],
                    help="sampler KV pages: fp8 = e4m3 + per-token scales (the engine's default; every GEMM and the whole training / "
                         "log-prob / reward math stay bf16), bf16 = the round-1 setting")
    ap.add_argument("--reward", default="deberta-large", choices=["deberta-large", "deberta-tiny"])
    ap.add_argument("--grad-checkpointing", type=int, default=0,
                    help="1 = recompute activations like the reference (A100-40G memory saver); 0 = keep them (B200: 180 GB)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed update computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# Per-token arrays of the dump keep at most this many elements each (a seeded sample of rows beyond it), so that the four of
# them plus the weight sample stay under 64 MB at any batch or response length.
DUMP_TOKENS_PER_ARRAY = 2_500_000
DUMP_SAMPLES_PER_WEIGHT = 2048


def dump_outputs(out_dir, metrics, rollout, policy):
    """Write what one update computed as ``out_dir/<name>.npy`` (float32 / float64) so that two builds can be compared on the
    same seeded inputs: its metrics without timings (``metrics.*``, 0-d float64); the rollout it trained on -- ``responses``
    (token ids), ``logprobs`` / ``ref_logprobs`` (policy / reference log-probs of those tokens), ``advantages``, ``scores``
    (reward-model score) and ``normalized_scores`` (group-normalised), one row per sequence, the same seeded rows in each
    when the batch is larger than the limit; and ``trainable_weights_sample``, a fixed seeded sample of every trainable
    tensor of the updated policy, in name order."""
    import numpy as np
    import torch

    out = {"metrics." + k.replace("/", "."): np.float64(v) for k, v in sorted(metrics.items())
           if not k.startswith(("time/", "throughput/", "mem/"))}
    n, t = rollout["responses"].shape
    keep = max(1, DUMP_TOKENS_PER_ARRAY // t)
    rows = torch.arange(n) if n <= keep else torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].sort().values
    for name, key in (("responses", "responses"), ("logprobs", "logprobs"), ("ref_logprobs", "ref_logprobs"),
                      ("advantages", "advantages"), ("scores", "log_scores"), ("normalized_scores", "scores")):
        x = rollout[key]
        out[name] = x[rows.to(x.device)].float().cpu().numpy()
    g = torch.Generator().manual_seed(0)
    parts = []
    for _, p in sorted(policy.named_parameters(), key=lambda kv: kv[0]):
        if p.requires_grad:
            flat = p.detach().reshape(-1)
            idx = torch.randint(0, flat.numel(), (min(flat.numel(), DUMP_SAMPLES_PER_WEIGHT),), generator=g)
            parts.append(flat[idx.to(flat.device)].float().cpu())
    out["trainable_weights_sample"] = torch.cat(parts).numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)
    total = sum(a.nbytes for a in out.values())
    print(f"[bench] wrote {len(out)} arrays ({total / 1e6:.1f} MB) to {out_dir}", file=sys.stderr, flush=True)


def reference_arm(args):
    """The reference cannot be installed or run offline: it is not a package (no setup.py / pyproject),
    imports trl / peft / accelerate (absent from the image and the wheelhouse) and downloads
    Qwen2.5-1.5B-Instruct, the DeBERTa reward model and hh-rlhf from the HF hub at import (no network)."""
    why = ("reference is not pip-installable (no setup.py/pyproject.toml) and needs trl+peft+accelerate "
           "(not in image/wheelhouse) plus HF-hub downloads of models/datasets (no network)")
    if int(os.environ.get("RANK", "0")) == 0:
        print(json.dumps({"impl": "reference", "unavailable": why}))
    return 0


def main():
    args = parse()
    if args.impl == "reference":
        return reference_arm(args)

    import torch

    from nanorlhf_b200.config import RLConfig
    from nanorlhf_b200.models.deberta_v3 import DebertaV3Config, DebertaV3ForSequenceClassification
    from nanorlhf_b200.models.lora import LoraConfig, get_peft_model
    from nanorlhf_b200.models.qwen2 import Qwen2Config, Qwen2ForCausalLM
    from nanorlhf_b200.ops import native
    from nanorlhf_b200.parallel.comm import Comm
    from nanorlhf_b200.reward.model_reward import ModelReward
    from nanorlhf_b200.trainer import GRPOTrainer
    from nanorlhf_b200.utils.clocks import ClockSampler
    from nanorlhf_b200.utils.data import synthetic_token_dataset
    from nanorlhf_b200.utils.tokenizer import ByteTokenizer
    from dataclasses import dataclass

    comm = Comm.from_env()
    dev = comm.device
    assert dev.type == "cuda", "bench.py needs a GPU"
    native.load()
    torch.manual_seed(0)

    shape = {"tiny": Qwen2Config(vocab_size=4096, hidden_size=256, intermediate_size=512, num_hidden_layers=2,
                                 num_attention_heads=2, num_key_value_heads=1, head_dim=128),
             "1.5b": Qwen2Config.qwen2_5_1_5b(), "7b": Qwen2Config.qwen2_5_7b()}[args.model]
    tok = ByteTokenizer(vocab_size=shape.vocab_size - 1)
    tok.add_special_tokens({"pad_token": "[PAD]"}) if False else None
    # reserve the last two embedding rows for eos / pad so random prompt ids never collide with them
    tok.special_tokens["<|im_end|>"] = shape.vocab_size - 2
    tok.special_tokens["[PAD]"] = shape.vocab_size - 1
    tok.id_to_special = {v: k for k, v in tok.special_tokens.items()}
    tok.eos_token_id, tok.pad_token_id, tok.vocab_size = shape.vocab_size - 2, shape.vocab_size - 1, shape.vocab_size

    policy = Qwen2ForCausalLM.from_config(shape, torch.bfloat16, dev, seed=0)
    ref_policy = Qwen2ForCausalLM.from_config(shape, torch.bfloat16, dev, seed=0)
    policy = get_peft_model(policy, LoraConfig(r=64, lora_alpha=16, modules_to_save=["embed_tokens", "lm_head", "score"]))
    rm_cfg = DebertaV3Config.large() if args.reward == "deberta-large" else DebertaV3Config.tiny(vocab_size=1024)
    rm = DebertaV3ForSequenceClassification.from_config(rm_cfg, torch.bfloat16, dev, seed=1)
    reward = ModelReward(rm, None, reward_batch_size=16, device=dev, token_budget=65536)

    @dataclass
    class GRPOConfig(RLConfig):
        grpo_sample_N: int = 4

    prompts_per_rank = 4 * 8 * args.mini_batches
    total_updates = args.steps + args.warmup
    out_dir = f"/tmp/nanorlhf_bench_{os.getpid()}"
    cfg = GRPOConfig(exp_name="bench-grpo", output_dir=out_dir, response_length=args.response_length, temperature=0.9,
                     kl_coef=0.01, cliprange=0.2, per_device_train_batch_size=4, gradient_accumulation_steps=8,
                     num_mini_batches=args.mini_batches, num_ppo_epochs=1,
                     total_episodes=prompts_per_rank * comm.world_size * total_updates, learning_rate=6e-6,
                     gradient_checkpointing=bool(args.grad_checkpointing), save_strategy="no", report_to="none", sampler="native",
                     rollout_dtype=args.rollout_dtype, kv_cache_dtype=args.kv_dtype, comm=args.comm, resume="never", grpo_sample_N=args.samples,
                     watchdog_timeout_s=0)
    cfg.quiet = True
    dataset = synthetic_token_dataset(prompts_per_rank * comm.world_size * 2, shape.vocab_size - 2, 24, 160, seed=1)
    trainer = GRPOTrainer(cfg, tok, policy, ref_policy, dataset, reward_func=reward, comm=comm)
    it = iter(trainer.dataloader)
    rollout = {}
    if args.dump_outputs:
        # keep a reference to each update's rollout batch; it is copied to the host only after the timed region
        algo_advantages = trainer.advantages

        def advantages(R):
            adv, ret = algo_advantages(R)
            rollout.update(R, advantages=adv)
            return adv, ret
        trainer.advantages = advantages

    def one_update(u):
        batch = next(it)                                    # host tensors (collated, pinned by the trainer)
        return trainer.train_one_update(u, batch)

    for u in range(1, args.warmup + 1):
        m = one_update(u)
        if comm.is_main:
            print(f"[bench] warmup {u}: {m['throughput/episodes_per_s']:.2f} episodes/s/rank-group "
                  f"rollout {m.get('time/rollout_s', 0):.2f}s reward {m.get('time/reward_s', 0):.2f}s "
                  f"logprob {m.get('time/logprob_s', 0):.2f}s train {m.get('time/train_s', 0):.2f}s", file=sys.stderr, flush=True)

    # ---- timed region -------------------------------------------------------------------------------
    clocks = ClockSampler(dev.index or 0, period_ms=500)
    comm.barrier()
    torch.cuda.synchronize()
    if comm.is_main:
        clocks.start()
    launches0 = native.launches()
    h2d0, d2h0 = trainer.io_bytes["h2d"], trainer.io_bytes["d2h"]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record()
    phase = {}
    trainer.optimizer.pop_comm_ms()
    opt_steps0 = trainer.optimizer._step
    for u in range(args.warmup + 1, args.warmup + args.steps + 1):
        m = one_update(u)
        for k, v in m.items():
            if k.startswith("time/") and k.endswith("_s") and "wall" not in k:
                phase[k] = phase.get(k, 0.0) + v
        if comm.is_main:
            g = getattr(trainer, "_graphed", None)
            print(f"[bench] step {u}: rollout {m.get('time/rollout_s', 0):.2f}s reward {m.get('time/reward_s', 0):.2f}s "
                  f"logprob {m.get('time/logprob_s', 0):.2f}s train {m.get('time/train_s', 0):.2f}s "
                  f"(micro-steps so far: {getattr(g, 'replays', 0)} graph replays, {getattr(g, 'eager', 0)} eager)", file=sys.stderr, flush=True)
    ev1.record()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    comm.barrier()
    dev_ms = ev0.elapsed_time(ev1)
    clock_info = clocks.stop() if comm.is_main else None
    n_opt = max(1, trainer.optimizer._step - opt_steps0)
    comm_ms, wait_ms = (x / n_opt for x in trainer.optimizer.pop_comm_ms(split=True))
    times = torch.tensor([dev_ms, (t1 - t0) * 1e3, comm_ms, wait_ms] + [phase.get(k, 0.0) for k in sorted(phase)], dtype=torch.float64, device=dev)
    comm.all_reduce_(times, "max")
    dev_ms, wall_ms, comm_ms, wait_ms = times.tolist()[:4]
    phase = dict(zip(sorted(phase), times.tolist()[4:]))          # max over ranks, like the headline
    episodes = prompts_per_rank * comm.world_size * args.steps
    value = episodes / (dev_ms / 1e3)
    e2e = episodes / (wall_ms / 1e3)
    roll_tokens = prompts_per_rank * args.samples * args.response_length * args.steps
    if comm.is_main:
        line = {
            "metric": "episodes_per_sec", "value": value, "unit": "episodes/s", "n_gpus": comm.world_size,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": value / BASELINE_EPISODES_PER_S,
            "vs_baseline_note": "denominator = the reference README's ~1 episode/s on 1 x A100-40G with real weights (its only "
                                "published throughput); not a same-box ratio -- see BASELINE.md section 2 for same-box anchors",
            "dtype": "bf16",
            "data": "synthetic hh-rlhf-shaped token prompts; random-init weights (no network)",
            "impl": "ours",
            "config": {"model": {"1.5b": "Qwen2.5-1.5B (random init)", "7b": "Qwen2.5-7B (random init)", "tiny": "tiny"}[args.model],
                       "algorithm": "GRPO", "reward_model": args.reward + " (random init)", "lora": "r=64 + embed/lm_head",
                       "global_batch": prompts_per_rank * comm.world_size, "prompts_per_rank": prompts_per_rank,
                       "sequences_per_rank": prompts_per_rank * args.samples, "samples_per_prompt": args.samples,
                       "seq_len": args.response_length, "prompt_len": "24-160", "parallelism": f"dp{comm.world_size}",
                       "comm": args.comm if comm.world_size > 1 else "none", "rollout_dtype": args.rollout_dtype, "kv_cache_dtype": args.kv_dtype,
                       "gradient_checkpointing": bool(args.grad_checkpointing),
                       "l2_policy": "working set (3 GB weights + KV pages + activations) exceeds the 126 MB L2 every step"},
            "e2e": {"value": e2e, "unit": "episodes/s", "h2d_bytes_per_step": (trainer.io_bytes["h2d"] - h2d0) / args.steps,
                    "d2h_bytes_per_step": (trainer.io_bytes["d2h"] - d2h0) / args.steps},
            "gpu_launches": native.launches() - launches0,
            "clocks": clock_info,
            "phases_s_per_step": {k[5:-2]: v / args.steps for k, v in sorted(phase.items())},
            "rollout_tok_per_s_per_gpu": roll_tokens / max(phase.get("time/rollout_s", 1e-9), 1e-9),
            "rollout_tok_per_s": comm.world_size * roll_tokens / max(phase.get("time/rollout_s", 1e-9), 1e-9),
            # device time of the gradient collective per optimizer step (K-AR kernel + its two barriers; runs after the
            # last micro-step's backward, so all of it is exposed), max over ranks; 0 on one GPU
            "exposed_comm_ms_per_step": comm_ms,
            # time a rank spends in the opening barrier of K-AR waiting for the slowest rank's backward (data-dependent load
            # imbalance of the whole update surfaces at its first optimizer step); max over ranks; not communication
            "straggler_wait_ms_per_step": wait_ms,
            "optimizer_steps_per_update": args.mini_batches,
            # micro-steps (forward + loss + backward) since start-up: replayed as CUDA graphs vs run eagerly (first sight of a
            # shape bucket, or everything if capture is disabled / failed)
            "train_micro_steps": {"graph_replays": getattr(getattr(trainer, "_graphed", None), "replays", 0),
                                  "eager": getattr(getattr(trainer, "_graphed", None), "eager", 0),
                                  "capture_failures": getattr(getattr(trainer, "_graphed", None), "capture_failures", 0)},
        }
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, m, rollout, trainer.policy)
    trainer.heartbeat.close()
    comm.barrier()
    comm.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
