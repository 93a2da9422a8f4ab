"""Shared helpers for the golden-fixture tests (no reference import: fixtures + synthetic weights only)."""
import json
import os

import numpy as np
import torch

from voicecraft_b200 import synthetic

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SILENCE = [1388, 1898, 131]


def load_cases():
    with open(os.path.join(GOLDEN, "lm_cases.json")) as f:
        return json.load(f)


def build_case(name, case):
    """Re-create config / weights exactly as tests/golden/make_golden.py::build_case did."""
    cfg = synthetic.make_config(case["cfg"], **case.get("over", {}))
    sd = synthetic.make_state_dict(cfg, seed=case["seed"])
    if case.get("eos_bias"):
        end = cfg.eos if cfg.eos > 0 else cfg.eog
        sd["predict_layer.0.2.bias"][end] += case["eos_bias"]
    if case.get("eog_bias"):
        sd["predict_layer.0.2.bias"][cfg.eog] += case["eog_bias"]
    if case.get("silence_bias"):
        sd["predict_layer.0.2.bias"][SILENCE[0]] += 9.0
    g = np.load(os.path.join(GOLDEN, f"lm_{name}.npz"))
    x = torch.from_numpy(g["x"])
    x_lens = torch.from_numpy(g["x_lens"])
    y = torch.from_numpy(g["y"])
    # inputs are also reproducible from the seed; the fixture copy is authoritative
    x2, xl2, y2 = synthetic.synthetic_utterance(cfg, 1000 + case["seed"], case["text_len"], case["prompt"])
    assert torch.equal(x, x2) and torch.equal(y, y2)
    return cfg, sd, x, x_lens, y, g


def cpu_noise_fn(seed):
    """Exp(1) noise from a private CPU generator seeded like the golden run (torch.manual_seed(seed))."""
    gen = torch.Generator(device="cpu").manual_seed(seed)

    def fn(shape, device=None):
        q = torch.empty(shape, dtype=torch.float32).exponential_(1, generator=gen)
        return q if device is None else q.to(device)
    return fn


# ---- headline shape (giga830M, 32 independent utterances): tests/golden/make_golden_830m.py ---------------------------
# The bf16-policy logit trace is stored as its bit pattern minus that of the fp32-policy trace (mod 2^32), split into byte
# planes: the two traces differ by ~1e-3, so the difference deflates 40 % smaller than the raw floats -- losslessly --
# which keeps the fixture under 1 MB.
def pack_logits_delta(base, logits):
    d = logits.astype("<f4").view("<u4") - base.astype("<f4").view("<u4")
    return np.ascontiguousarray(d.reshape(-1).view(np.uint8).reshape(-1, 4).T)


def unpack_logits_delta(base, planes):
    d = np.ascontiguousarray(planes.T).view("<u4").reshape(base.shape)
    return (base.astype("<f4").view("<u4") + d).view("<f4")


def headline_fixture():
    with open(os.path.join(GOLDEN, "lm_830m_b32.json")) as f:
        meta = json.load(f)
    g = dict(np.load(os.path.join(GOLDEN, "lm_830m_b32.npz")))
    g["logits_bf16"] = unpack_logits_delta(g["logits_fp32"], g.pop("logits_bf16_planes"))
    return meta, g


def suppress_end_tokens(cfg, sd):
    """only the reference's length cap ends generation (bench.py does the same)"""
    for k in range(cfg.n_codebooks):
        sd[f"predict_layer.{k}.2.bias"][cfg.eos] = -1e4
        sd[f"predict_layer.{k}.2.bias"][cfg.eog] = -1e4
    return sd


def headline_checkpoint(seed):
    cfg = synthetic.make_config("830M")
    return cfg, suppress_end_tokens(cfg, synthetic.make_state_dict(cfg, seed=seed))


def headline_utterance(cfg, meta, i):
    return synthetic.synthetic_utterance(cfg, 100 + i, meta["text_len"], meta["prompts"][i % len(meta["prompts"])])
