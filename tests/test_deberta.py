import os

import numpy as np
import torch

from nanorlhf_b200.models.deberta_v3 import DebertaV3Config, DebertaV3ForSequenceClassification

# HF transformers' DebertaV2ForSequenceClassification at the tiny shape: its weights, a padded batch of ids and the
# logits HF computed for them (transformers 5.5, fp32, CPU).  ``python -m tests.test_deberta`` regenerates it where transformers is installed.
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "deberta_v2_tiny_hf.npz")


def _write_hf_golden(path=GOLDEN):
    from transformers import DebertaV2Config, DebertaV2ForSequenceClassification
    hf_cfg = DebertaV2Config(vocab_size=200, hidden_size=64, num_hidden_layers=2, num_attention_heads=4,
                             intermediate_size=128, relative_attention=True, position_buckets=16, norm_rel_ebd="layer_norm",
                             share_att_key=True, pos_att_type=["p2c", "c2p"], position_biased_input=False,
                             max_position_embeddings=64, max_relative_positions=-1, pooler_hidden_size=64,
                             num_labels=1, layer_norm_eps=1e-7, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0,
                             pooler_dropout=0.0, type_vocab_size=0, pad_token_id=0)
    torch.manual_seed(0)
    hf = DebertaV2ForSequenceClassification(hf_cfg).eval()
    ids = torch.randint(3, 200, (3, 40))
    ids[0, 30:] = 0
    ids[2, 12:] = 0
    with torch.no_grad():
        logits = hf(input_ids=ids, attention_mask=(ids != 0).long()).logits
    arrays = {"sd/" + k: v.numpy() for k, v in hf.state_dict().items()}
    np.savez(path, input_ids=ids.numpy(), logits=logits.float().numpy(), **arrays)


def test_matches_hf_deberta_v2():
    g = np.load(GOLDEN)
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd/")}
    mine = DebertaV3ForSequenceClassification(DebertaV3Config.tiny(vocab_size=200)).eval()
    missing, unexpected = mine.load_state_dict(sd, strict=False)
    assert not missing, missing
    ids = torch.from_numpy(g["input_ids"])
    mask = ids != 0
    want = torch.from_numpy(g["logits"])
    with torch.no_grad():
        got = mine(ids, mask)
    assert torch.allclose(got, want, atol=1e-4, rtol=1e-4), (got, want)


def test_model_reward_id_path():
    from nanorlhf_b200.reward.model_reward import ModelReward
    from nanorlhf_b200.utils.tokenizer import ByteTokenizer
    tok = ByteTokenizer()
    rm = DebertaV3ForSequenceClassification.from_config(DebertaV3Config.tiny(vocab_size=300), torch.float32, seed=0)
    r = ModelReward(rm, None, reward_batch_size=4)
    q = torch.randint(0, 250, (6, 10))
    resp = torch.randint(0, 250, (6, 12))
    resp[1, 5:] = tok.pad_token_id
    s = r(q, resp, tok)
    assert s.shape == (6,) and torch.isfinite(s).all()
    # batching must not change scores
    r2 = ModelReward(rm, None, reward_batch_size=1)
    assert torch.allclose(s, r2(q, resp, tok), atol=1e-5)


if __name__ == "__main__":
    _write_hf_golden()
