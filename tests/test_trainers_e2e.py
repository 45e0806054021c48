"""T1: every algorithm end to end on CPU with the PyTorch sampler (plumbing config of BASELINE.json)."""
import os

import pytest
import torch

from nanorlhf_b200.config import RLConfig
from nanorlhf_b200.models.lora import LoraConfig, get_peft_model
from nanorlhf_b200.models.qwen2 import Qwen2Config, Qwen2ForCausalLM, Qwen2ForSequenceClassification
from nanorlhf_b200.reward.api import ConstantReward, LengthReward
from nanorlhf_b200.trainer import (GRPOTrainer, PPOTrainer, RAFTTrainer, ReinforceTrainer, RemaxTrainer, RLOOTrainer,
                                   SparseGRPOTrainer)
from nanorlhf_b200.utils.data import synthetic_hh_dataset
from nanorlhf_b200.utils.tokenizer import ByteTokenizer

GRPO_KEYS = {"objective/kl_old", "objective/entropy_old", "objective/non_score_reward_old", "eval_objective/rlhf_reward_old",
             "eval_objective/scores_old", "policy/approxkl_avg_new", "policy/clipfrac_avg_new", "loss/policy_avg_new",
             "policy/entropy_avg_new", "val/ratio_new", "val/ratio_var_new", "val/num_eos_tokens_old", "lr", "episode"}


def build(cls, tmp_path, extra=None, reward=None, lora=True, **kw):
    tok = ByteTokenizer()
    cfg = Qwen2Config.tiny(vocab_size=tok.vocab_size)
    policy = Qwen2ForCausalLM.from_config(cfg, torch.float32, seed=1)
    ref = Qwen2ForCausalLM.from_config(cfg, torch.float32, seed=1)
    if lora:
        policy = get_peft_model(policy, LoraConfig(r=4, lora_alpha=8, modules_to_save=["embed_tokens", "lm_head"]))
    base = dict(output_dir=str(tmp_path), response_length=10, per_device_train_batch_size=2, gradient_accumulation_steps=2,
                num_mini_batches=2, total_episodes=16, learning_rate=1e-3, sampler="torch", report_to="none")
    base.update(kw)
    a = RLConfig(**base)
    for k, v in (extra or {}).items():
        setattr(a, k, v)
    ds = synthetic_hh_dataset(tok, 32, max_prompt_tokens=24)
    kwargs = {}
    if cls is PPOTrainer:
        vm = Qwen2ForSequenceClassification.from_causal_lm(ref)
        kwargs["value_model"] = get_peft_model(vm, LoraConfig(r=4, lora_alpha=8, modules_to_save=["score"]))
    # the PyTorch plumbing path on every machine, a GPU present or not (the CUDA runs are in test_trainers_gpu.py)
    return cls(a, tok, policy, ref, ds, reward_func=reward or LengthReward(6), device=torch.device("cpu"), **kwargs)


@pytest.mark.parametrize("cls,extra,kw", [
    (ReinforceTrainer, None, dict(advantage_whiten=True)),
    (GRPOTrainer, {"grpo_sample_N": 4}, {}),
    (RLOOTrainer, {"rloo_sample_N": 4}, {}),
    (RemaxTrainer, None, {}),
    (RAFTTrainer, {"raft_sample_K": 4}, {}),
    (PPOTrainer, {"policy_learning_rate": 1e-3, "value_learning_rate": 2e-3}, dict(vf_coef=1.0)),
    (SparseGRPOTrainer, {"grpo_sample_N": 4}, {}),
])
def test_algorithm_runs_two_updates(cls, extra, kw, tmp_path):
    t = build(cls, tmp_path, extra, **kw)
    before = [p.detach().clone() for p in t.policy.parameters() if p.requires_grad]
    m = t.train()
    assert t.state.global_step == 2 and t.state.episode == 16
    after = [p for p in t.policy.parameters() if p.requires_grad]
    assert any(not torch.equal(a, b) for a, b in zip(before, after)), "no parameter moved"
    assert all(torch.isfinite(p).all() for p in after)
    want = set(GRPO_KEYS)
    if cls is RAFTTrainer:
        want -= {"policy/approxkl_avg_new", "policy/clipfrac_avg_new", "val/ratio_new", "val/ratio_var_new"}
    if cls is PPOTrainer:
        want |= {"loss/value_avg_new", "val/clipfrac_avg_new", "eval_accuracy_new"}
    assert want <= set(m), want - set(m)
    ck = os.path.join(str(tmp_path), "checkpoint-2")
    for f in ("adapter_model.safetensors", "adapter_config.json", "optimizer.pt", "scheduler.pt", "rng_state.pth",
              "trainer_state.json", "training_args.bin"):
        assert os.path.exists(os.path.join(ck, f)), f
    if cls is PPOTrainer:
        assert os.path.exists(os.path.join(ck, "value_model", "adapter_model.safetensors"))
        assert len(t.optimizer.param_groups) >= 2 and t.optimizer.param_groups[0]["lr"] != t.optimizer.param_groups[-1]["lr"]


def test_full_finetune_checkpoint_layout(tmp_path):
    t = build(ReinforceTrainer, tmp_path, lora=False, reward=ConstantReward(1.0))
    t.train()
    ck = os.path.join(str(tmp_path), "checkpoint-2")
    assert os.path.exists(os.path.join(ck, "model.safetensors")) and os.path.exists(os.path.join(ck, "config.json"))


def test_resume_is_bit_identical(tmp_path):
    """save -> load -> next update equals an uninterrupted run (the reference cannot resume at all)."""
    from nanorlhf_b200.sampler import engine
    engine.reseed_stream(42)
    full = build(GRPOTrainer, tmp_path / "a", {"grpo_sample_N": 2}, total_episodes=24)
    full.train()
    ref_params = [p.detach().clone() for p in full.policy.parameters() if p.requires_grad]

    engine.reseed_stream(42)
    first = build(GRPOTrainer, tmp_path / "b", {"grpo_sample_N": 2}, total_episodes=24)
    first.args.num_total_batches = 2           # stop after two of the three updates
    first.train()
    second = build(GRPOTrainer, tmp_path / "b", {"grpo_sample_N": 2}, total_episodes=24)
    second.train()                              # resume=auto picks checkpoint-2 and runs update 3
    assert second.state.global_step == 3
    got = [p for p in second.policy.parameters() if p.requires_grad]
    for a, b in zip(ref_params, got):
        assert torch.equal(a, b)


def test_rotation_and_best_checkpoint(tmp_path):
    t = build(ReinforceTrainer, tmp_path, total_episodes=40, save_total_limit=2)
    t.train()
    cks = sorted(d for d in os.listdir(tmp_path) if d.startswith("checkpoint-"))
    assert len(cks) <= 3 and "checkpoint-5" in cks
    assert t.state.best_model_checkpoint is not None and os.path.isdir(t.state.best_model_checkpoint)


def test_value_initializer(tmp_path):
    from nanorlhf_b200.config import ValueFinetuneConfig
    from nanorlhf_b200.trainer.value_initializer import finetuned_value_model
    t = build(PPOTrainer, tmp_path, {"policy_learning_rate": 1e-3, "value_learning_rate": 1e-3})
    vm = t.model.value_model
    fa = ValueFinetuneConfig(train_data_size=16, num_train_epochs=3, per_device_train_batch_size=4,
                             gradient_accumulation_steps=1, learning_rate=5e-3, per_device_eval_batch_size=8)
    before = [p.detach().clone() for p in vm.parameters() if p.requires_grad]
    out = finetuned_value_model(vm, t.policy, t.ref_policy, LengthReward(6), t.train_dataset, t.tokenizer, t.args, fa,
                                verbose=False)
    hist = out.value_init_history
    assert len(hist) >= 2 and min(h["eval_loss"] for h in hist) <= hist[0]["eval_loss"]
    assert any(not torch.equal(a, b) for a, b in zip(before, [p for p in vm.parameters() if p.requires_grad]))


def test_train_on_all_samples_keeps_step_count(tmp_path):
    """``train_samples_per_prompt = N`` (train on every sample): N x the rows, the same number of optimizer steps, no
    out-of-range stats slot (ADVICE round 1)."""
    t = build(GRPOTrainer, tmp_path, {"grpo_sample_N": 4}, train_samples_per_prompt=4)
    steps0 = t.optimizer._step
    m = t.train()
    assert t.state.global_step == 2
    assert t.optimizer._step - steps0 == 2 * t.args.num_mini_batches
    assert all(k in m for k in GRPO_KEYS)


def test_top_p_consistent_scoring_switch(tmp_path):
    """``logprob_top_p_consistent=True``: policy and reference log-probs come from the truncated, renormalised softmax the
    sampler draws from (models/qwen2.py token_logprobs -> ops/reference.py lmhead_logprob_top_p); training still steps."""
    t = build(GRPOTrainer, tmp_path, {"grpo_sample_N": 4}, logprob_top_p_consistent=True, top_p=0.9)
    lm = getattr(t.policy, "base_model", t.policy)
    assert lm.logprob_top_p == 0.9 and getattr(t.ref_policy, "logprob_top_p", None) == 0.9
    m = t.train()
    assert t.state.global_step == 2
    assert all(v == v for v in m.values() if isinstance(v, float))
    # with the switch the old / new log-probs are >= their full-softmax values, so the recorded KL to the reference stays finite
    assert abs(m["objective/kl_old"]) < 1e3
