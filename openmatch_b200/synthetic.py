"""Seeded synthetic weights and inputs of the shapes BASELINE.json names (no checkpoints, datasets or
network on the build / GPU boxes).  Weights follow HuggingFace's default initialisation statistics
(N(0, 0.02) matrices and embeddings, LayerNorm weight 1 / bias 0, zero biases perturbed slightly so that
bias paths are exercised); token ids follow SURVEY.md section 8(d)."""
from __future__ import annotations

import json
from typing import Dict, Tuple

import numpy as np
import torch

BERT_BASE = dict(arch="bert", layers=12, hidden=768, heads=12, ffn=3072, vocab=30522, max_pos=512, type_vocab=2,
                 ln_eps=1e-12)
BERT_LARGE = dict(arch="bert", layers=24, hidden=1024, heads=16, ffn=4096, vocab=30522, max_pos=512, type_vocab=2,
                  ln_eps=1e-12)
T5_BASE = dict(arch="t5", layers=12, hidden=768, heads=12, ffn=3072, vocab=32128, ln_eps=1e-6, rel_buckets=32,
               rel_max_distance=128)


def bert_state_dict(spec: Dict, seed: int = 0, std: float = 0.02) -> Dict[str, torch.Tensor]:
    g = torch.Generator().manual_seed(seed)
    H, F = spec["hidden"], spec["ffn"]

    def w(*shape):
        return torch.randn(*shape, generator=g) * std

    def ln():
        return 1.0 + 0.05 * torch.randn(H, generator=g), 0.02 * torch.randn(H, generator=g)

    sd = {"embeddings.word_embeddings.weight": w(spec["vocab"], H),
          "embeddings.position_embeddings.weight": w(spec["max_pos"], H),
          "embeddings.token_type_embeddings.weight": w(spec["type_vocab"], H)}
    sd["embeddings.LayerNorm.weight"], sd["embeddings.LayerNorm.bias"] = ln()
    shapes = {"attention.self.query": (H, H), "attention.self.key": (H, H), "attention.self.value": (H, H),
              "attention.output.dense": (H, H), "intermediate.dense": (F, H), "output.dense": (H, F)}
    for i in range(spec["layers"]):
        p = f"encoder.layer.{i}."
        for name, (o, k) in shapes.items():
            sd[p + name + ".weight"], sd[p + name + ".bias"] = w(o, k), w(o)
        sd[p + "attention.output.LayerNorm.weight"], sd[p + "attention.output.LayerNorm.bias"] = ln()
        sd[p + "output.LayerNorm.weight"], sd[p + "output.LayerNorm.bias"] = ln()
    return sd


def t5_state_dict(spec: Dict, seed: int = 0) -> Dict[str, torch.Tensor]:
    g = torch.Generator().manual_seed(seed)
    H, F, nh = spec["hidden"], spec["ffn"], spec["heads"]
    inner = nh * 64

    def w(o, k, std):
        return torch.randn(o, k, generator=g) * std

    sd = {"shared.weight": torch.randn(spec["vocab"], H, generator=g),
          "encoder.final_layer_norm.weight": 1.0 + 0.05 * torch.randn(H, generator=g),
          "encoder.block.0.layer.0.SelfAttention.relative_attention_bias.weight":
              torch.randn(spec.get("rel_buckets", 32), nh, generator=g)}
    for i in range(spec["layers"]):
        p = f"encoder.block.{i}.layer."
        sd[p + "0.SelfAttention.q.weight"] = w(inner, H, (H * 64) ** -0.5)
        sd[p + "0.SelfAttention.k.weight"] = w(inner, H, H ** -0.5)
        sd[p + "0.SelfAttention.v.weight"] = w(inner, H, H ** -0.5)
        sd[p + "0.SelfAttention.o.weight"] = w(H, inner, inner ** -0.5)
        sd[p + "0.layer_norm.weight"] = 1.0 + 0.05 * torch.randn(H, generator=g)
        sd[p + "1.DenseReluDense.wi.weight"] = w(F, H, H ** -0.5)
        sd[p + "1.DenseReluDense.wo.weight"] = w(H, F, F ** -0.5)
        sd[p + "1.layer_norm.weight"] = 1.0 + 0.05 * torch.randn(H, generator=g)
    return sd


def _splitmix64(seed: int, n: int) -> np.ndarray:
    z = np.uint64(seed) + np.arange(1, n + 1, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def recipe_state_dict(recipe) -> Dict[str, torch.Tensor]:
    """Weights rebuilt from a recipe: a JSON list (or the list itself) of [name, shape, mean, std, seed] entries, each
    tensor mean + std * U with U uniform on [-sqrt 3, sqrt 3) at 24-bit resolution, drawn from a splitmix64 stream.
    Integer arithmetic and correctly rounded float operations only, so the weights are bit-identical on every platform
    and library version; tests/golden stores such recipes instead of the weights themselves."""
    if isinstance(recipe, (str, np.ndarray)):
        recipe = json.loads(str(recipe))
    sd = {}
    for name, shape, mean, std, seed in recipe:
        n = int(np.prod(shape, dtype=np.int64))
        u = (_splitmix64(seed, n) >> np.uint64(40)).astype(np.int64) - (1 << 23)  # [-2^23, 2^23): exact in float64
        sd[name] = torch.from_numpy((mean + u * (std * 3.0 ** 0.5 / (1 << 23))).astype(np.float32).reshape(shape))
    return sd


def token_batch(B: int, L: int, vocab: int, seed: int = 1234, ragged: bool = False, bert: bool = True,
                device="cpu") -> Tuple[torch.Tensor, torch.Tensor]:
    """ids uniform in [1000, vocab), [CLS]=101 first and [SEP]=102 (BERT) / </s>=1 (T5) last; ``ragged``
    draws lengths ~ clip(N(0.55 L, 0.2 L), 8, L) with zero padding after the end token."""
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(1000, vocab, (B, L), generator=g)
    mask = torch.ones(B, L, dtype=torch.long)
    lens = torch.full((B,), L, dtype=torch.long)
    if ragged:
        lens = (torch.randn(B, generator=g) * 0.2 * L + 0.55 * L).round().clamp(min(8, L), L).long()
    end = 102 if bert else 1
    for b in range(B):
        n = int(lens[b])
        ids[b, n - 1] = end
        ids[b, n:] = 0
        mask[b, n:] = 0
    if bert:
        ids[:, 0] = 101
    return ids.to(device), mask.to(device)
