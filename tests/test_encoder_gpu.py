"""GPU parity: BERT encoder / cross-encoder through the C ABI vs the goldens (HF transformers) and
the oracle.  Tolerance 1e-3 on embeddings and logits (BASELINE.json)."""
from dataclasses import asdict

import numpy as np
import pytest
import torch

from oracle import bert_ref
from ragmeup_b200.weights import PRESETS, BertConfig, synthetic_bert_weights

pytestmark = pytest.mark.gpu
TOL = 1e-3
ENC_CASES = [("tiny", 0, 1.0), ("all-MiniLM-L6-v2", 0, 1.0), ("all-MiniLM-L6-v2", 1, 4.0), ("bge-base-en-v1.5", 0, 1.0)]
CE_CASES = [("tiny", 3, 4.0), ("ms-marco-MiniLM-L-6-v2", 0, 1.0), ("ms-marco-MiniLM-L-6-v2", 2, 6.0)]


def _ragged(ids, mask, typ):
    lens = mask.sum(1)
    cu = np.r_[0, np.cumsum(lens)].astype(np.int32)
    rid = np.concatenate([ids[b, :n] for b, n in enumerate(lens)]).astype(np.int32)
    rty = np.concatenate([typ[b, :n] for b, n in enumerate(lens)]).astype(np.int32)
    return rid, rty, cu, int(lens.max())


@pytest.mark.parametrize("preset,seed,scale", ENC_CASES)
def test_embeddings_match_hf_golden(cuda, golden_dir, preset, seed, scale):
    from ragmeup_b200.encoder import BertEncoder
    g = np.load(f"{golden_dir}/encoder.npz")
    key = f"enc_{preset}_{seed}_{scale}"
    cfg = BertConfig(**asdict(PRESETS[preset][0]))
    enc = BertEncoder(cfg, synthetic_bert_weights(cfg, seed=seed, scale=scale), with_head=False)
    ids, typ, cu, mx = _ragged(g[key + "_ids"].astype(np.int64), g[key + "_mask"].astype(np.int64), g[key + "_typ"].astype(np.int64))
    mean = enc.embed_tokens(ids, typ, cu, mx, "mean", True).cpu().numpy()
    cls = enc.embed_tokens(ids, typ, cu, mx, "cls", True).cpu().numpy()
    assert np.abs(mean - g[key + "_mean"]).max() < TOL
    assert np.abs(cls - g[key + "_cls"]).max() < TOL
    h = enc.hidden_tokens(ids, typ, cu, mx).cpu().numpy()
    assert np.abs(h[cu[:-1]] - g[key + "_h_first"]).max() < 5e-3
    assert np.abs(h[cu[1:] - 1] - g[key + "_h_last"]).max() < 5e-3
    # host-buffer entry point returns the same numbers
    assert np.abs(enc.embed_host(ids, typ, cu, "mean", True) - mean).max() < 1e-6
    # unnormalised mean pooling
    raw = enc.embed_tokens(ids, typ, cu, mx, "mean", False).cpu().numpy()
    assert np.abs(raw / np.linalg.norm(raw, axis=1, keepdims=True) - mean).max() < 1e-5


@pytest.mark.parametrize("preset,seed,scale", CE_CASES)
def test_logits_match_hf_golden(cuda, golden_dir, preset, seed, scale):
    from ragmeup_b200.encoder import BertEncoder
    g = np.load(f"{golden_dir}/cross_encoder.npz")
    key = f"ce_{preset}_{seed}_{scale}"
    cfg = BertConfig(**asdict(PRESETS[preset][0]))
    enc = BertEncoder(cfg, synthetic_bert_weights(cfg, seed=seed, with_head=True, scale=scale), with_head=True)
    ids, typ, cu, mx = _ragged(g[key + "_ids"].astype(np.int64), g[key + "_mask"].astype(np.int64), g[key + "_typ"].astype(np.int64))
    lg = enc.classify_tokens(ids, typ, cu, mx).cpu().numpy()
    assert np.abs(lg - g[key + "_logits"]).max() < TOL
    assert np.abs(enc.classify_host(ids, typ, cu) - lg).max() < 1e-6


def _ragged_batch_vs_oracle(preset, head, lens, alone):
    """one ragged batch through the encoder vs the oracle (logits with the classifier head, else normalised mean
    embeddings), then the sequences `alone` re-run one at a time"""
    from ragmeup_b200.encoder import BertEncoder
    cfg = BertConfig(**asdict(PRESETS[preset][0]))
    ocfg = bert_ref.BertCfg(**asdict(cfg))
    w = synthetic_bert_weights(cfg, seed=5, with_head=head, scale=4.0)
    enc = BertEncoder(cfg, w, with_head=head)
    rng = np.random.default_rng(9)
    ids = np.concatenate([np.r_[101, rng.integers(104, cfg.vocab_size, n - 2), 102] for n in lens]).astype(np.int32)
    typ = np.concatenate([np.r_[np.zeros(n // 3, np.int32), np.ones(n - n // 3, np.int32)] for n in lens])
    cu = np.r_[0, np.cumsum(lens)].astype(np.int32)

    def run(i, t, c, mx):
        return (enc.classify_tokens(i, t, c, mx) if head else enc.embed_tokens(i, t, c, mx, "mean", True)).cpu()

    out = run(ids, typ, cu, max(lens))
    S = max(lens)
    I = np.zeros((len(lens), S), np.int64); M = np.zeros_like(I); T = np.zeros_like(I)
    for b, n in enumerate(lens):
        I[b, :n] = ids[cu[b]:cu[b + 1]]; T[b, :n] = typ[cu[b]:cu[b + 1]]; M[b, :n] = 1
    with torch.no_grad():
        h = bert_ref.bert_encoder_forward(w, ocfg, torch.from_numpy(I), torch.from_numpy(M), torch.from_numpy(T))
        ref = bert_ref.classifier_head(w, h) if head else bert_ref.l2_normalize(bert_ref.pool(h, torch.from_numpy(M), "mean"))
    assert float((out - ref).abs().max()) < TOL
    # batch-composition invariance: each sequence alone gives the same result
    for b in alone:
        one = run(ids[cu[b]:cu[b + 1]], typ[cu[b]:cu[b + 1]], np.array([0, lens[b]], np.int32), lens[b])
        assert float((one[0] - out[b]).abs().max()) < 1e-5


def test_ragged_batch_vs_oracle_long_sequences(cuda):
    """S up to 512 (truncation limit), 150-token rerank-shaped pairs, single-token edge"""
    _ragged_batch_vs_oracle("ms-marco-MiniLM-L-6-v2", True, [512, 147, 147, 2, 300, 31], (1, 3))


# The longest sequence picks the attention kernel: MiniLM (d_h = 32) takes the per-head tcgen05 kernel at 161-224
# keys, bge-base (d_h = 64, embeddings) the mma.sync kernel past 192 keys.
@pytest.mark.parametrize("preset,head,lens,alone", [
    ("ms-marco-MiniLM-L-6-v2", True, [200, 147, 31, 2], (1, 3)),
    ("bge-base-en-v1.5", False, [300, 64, 5], (1, 2)),
], ids=["minilm-200-keys", "bge-base-300-keys"])
def test_ragged_batch_vs_oracle_attention_kernels(cuda, preset, head, lens, alone):
    _ragged_batch_vs_oracle(preset, head, lens, alone)
