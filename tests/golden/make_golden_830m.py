"""Golden fixtures at the HEADLINE shape (BASELINE.json configs[1]: giga830M, B=32 independent utterances, K=4).

Run in the build container only (imports /root/reference):
    python tests/golden/make_golden_830m.py            # ~20 min on 8 cores

Part A (reference-pinned): two utterances whose generation ends by the reference's own length cap
(voicecraft.py:1041-1045) are run through the UNMODIFIED reference (fp32, CPU, torch.manual_seed(s)) and through
oracle/lm_oracle.py; tokens must be identical.  Stored: inputs, the reference's `res`.
Part B (batch of 32): the bench checkpoint (synthetic seed 0, end tokens suppressed) and 32 utterances with prompt
lengths chosen so that, within N = 64 decode steps, contexts cross KV-page boundaries (64), 256 and 512.  Every
utterance is decoded by the oracle with its own CPU generator (seed 1 + i, SURVEY.md section 8d config 2) under both KV
policies (fp32 = the reference's arithmetic; bf16 = the engine's default pages, `kv_round_bf16=True`).  Stored per
policy: the sampled rows [32, N, K], the SENSITIVITY of every sample and a thin logit trace.  Sensitivity = the smallest
delta such that moving every logit by at most +-delta could change the sampled token: min of (a) half the log-score gap
to the best other kept token, (b) half the gap between the winner's logit and the (k+1)-th largest logit (the winner is
filtered out by top-k), (c) over excluded tokens, the larger of half its distance to the top-k threshold and half its
log-score gap to the winner (it enters the top-k and wins).  A CUDA-path token may differ from the oracle's only where
this is below the logit tolerance.
The -m gpu tests rebuild weights / inputs from the seeds and compare the CUDA path with these rows.
"""
import json
import os
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

import golden_util  # noqa: E402

N_STEPS = 64
PROMPTS = [150, 170, 400, 420, 230, 330, 110, 460]       # ctx = 80 + p + 1: 231, 251, 481, 501, 311, 411, 191, 541
TEXT_LEN = 80
KW = dict(top_k=40, top_p=1.0, temperature=1.0, stop_repetition=3)
SILENCE = [1388, 1898, 131]
TRACE_UTTS = [0, 3, 13, 31]
TRACE_STEPS = [0, 1, 31, 63]


def bench_checkpoint():
    from voicecraft_b200 import synthetic
    cfg = synthetic.make_config("830M")
    sd = synthetic.make_state_dict(cfg, seed=0)
    for k in range(cfg.n_codebooks):        # only the length cap ends generation (same as bench.py)
        sd[f"predict_layer.{k}.2.bias"][cfg.eos] = -1e4
        sd[f"predict_layer.{k}.2.bias"][cfg.eog] = -1e4
    return cfg, sd


def utterance(cfg, i):
    from voicecraft_b200 import synthetic
    return synthetic.synthetic_utterance(cfg, 100 + i, TEXT_LEN, PROMPTS[i % len(PROMPTS)])


def cpu_noise(seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return lambda shape: torch.empty(shape, dtype=torch.float32).exponential_(1, generator=g)


def main():
    torch.set_num_threads(8)
    from make_golden import import_reference, ref_model
    from oracle import lm_oracle
    from voicecraft_b200 import synthetic
    out = {}
    t0 = time.time()

    # ---------------- Part A: the real reference at 830M, natural (length-cap) termination ----------------
    prev = os.path.join(HERE, "lm_830m_b32.npz")
    if "--keep-part-a" in sys.argv and os.path.exists(prev):
        old = np.load(prev)
        out.update({k: old[k] for k in old.files if k.startswith("pin")})
        return part_b(out, t0)
    voicecraft, _ = import_reference()
    cfg = synthetic.make_config("830M")
    sd = synthetic.make_state_dict(cfg, seed=3)
    for k in range(cfg.n_codebooks):
        sd[f"predict_layer.{k}.2.bias"][cfg.eos] = -1e4
        sd[f"predict_layer.{k}.2.bias"][cfg.eog] = -1e4
    model = ref_model(voicecraft, cfg, sd)
    oracle = lm_oracle.OracleLM(cfg, sd)
    pinned = [dict(seed=41, text_len=26, prompt=200), dict(seed=42, text_len=33, prompt=292)]
    for j, pc in enumerate(pinned):
        x, xl, y = synthetic.synthetic_utterance(cfg, 7000 + j, pc["text_len"], pc["prompt"])
        torch.manual_seed(pc["seed"])
        res, gen = model.inference_tts(x, xl, y, silence_tokens=SILENCE, kvcache=1, **KW)
        ores, ogen = oracle.inference_tts(x, xl, y, silence_tokens=SILENCE, noise_fn=cpu_noise(pc["seed"]), **KW)
        assert torch.equal(res, ores), f"pinned utterance {j}: oracle tokens differ from the reference"
        print(f"part A utt {j}: reference == oracle, generated {gen.shape[-1]} frames, ctx {pc['text_len'] + pc['prompt'] + 1}+ "
              f"({time.time() - t0:.0f}s)", flush=True)
        out[f"pin{j}_res"] = res.numpy().astype(np.int16)
    del model, oracle
    return part_b(out, t0)


def part_b(out, t0):
    from oracle import lm_oracle
    pinned = [dict(seed=41, text_len=26, prompt=200), dict(seed=42, text_len=33, prompt=292)]
    # ---------------- Part B: 32 utterances x 64 steps, both KV policies -----------------------------------
    cfg, sd = bench_checkpoint()
    state = {}
    orig = lm_oracle.sample_rows

    def spy(logits, top_k, top_p, temperature, noise_fn):
        """sample_rows + the smallest per-logit perturbation that could change the sampled token (see module docstring)"""
        assert top_p >= 1.0 and temperature == 1.0 and top_k > 0
        raw = logits.clone()
        lg = lm_oracle.filter_top_k_top_p(logits.clone(), top_k=top_k, top_p=top_p)
        p = F.softmax(lg, dim=-1)
        q = noise_fn(tuple(p.shape))
        sc = p / q
        win = torch.argmax(sc, dim=-1)
        sens = []
        for row in range(raw.shape[0]):
            L = raw[row].double()
            s = L - torch.log(q[row].double())                    # log-domain score (the softmax normaliser cancels)
            k = min(top_k, L.numel())
            srt = torch.sort(L, descending=True)[0]
            kth, nxt = srt[k - 1], (srt[k] if k < L.numel() else torch.tensor(-1e30, dtype=torch.float64))
            kept = L >= kth
            w = int(win[row])
            s_w = s[w]
            others = s.clone()
            others[~kept] = -1e30
            others[w] = -1e30
            d1 = (s_w - others.max()) / 2                          # another kept token overtakes the winner
            d2 = (L[w] - nxt) / 2                                  # the winner drops below the top-k threshold (lower bound)
            exc = ~kept
            d3 = torch.tensor(1e30, dtype=torch.float64)
            if exc.any():                                          # an excluded token enters the top-k AND beats the winner
                d3 = torch.maximum((kth - L[exc]) / 2, (s_w - s[exc]) / 2).min()
            sens.append(float(torch.minimum(torch.minimum(d1, d2), d3).clamp(min=0)))
        state["margins"].append(np.array(sens))
        return win.unsqueeze(-1)
    lm_oracle.sample_rows = spy
    for pol, rb in (("fp32", False), ("bf16", True)):
        oracle = lm_oracle.OracleLM(cfg, sd, kv_round_bf16=rb)
        rows_all, marg_all, traces = [], [], {}
        for i in range(32):
            x, xl, y = utterance(cfg, i)
            state["margins"] = []
            rows = oracle.inference_tts(x, xl, y, silence_tokens=SILENCE, noise_fn=cpu_noise(1 + i), max_steps=N_STEPS,
                                        trace_logits=True, **KW)
            assert rows.shape == (N_STEPS, cfg.n_codebooks)
            rows_all.append(rows.numpy())
            marg_all.append(np.stack(state["margins"]))           # [N, K]
            if i in TRACE_UTTS:
                traces[i] = np.stack([oracle.logit_trace[s].numpy() for s in TRACE_STEPS])
            print(f"part B {pol} utt {i}: ctx {TEXT_LEN + PROMPTS[i % 8] + 1} ({time.time() - t0:.0f}s)", flush=True)
        out[f"rows_{pol}"] = np.stack(rows_all).astype(np.int16)
        out[f"sens_{pol}"] = np.stack(marg_all).astype(np.float32)
        out[f"logits_{pol}"] = np.stack([traces[i] for i in TRACE_UTTS]).astype(np.float32)   # [utt, step, K, V]
        del oracle
    lm_oracle.sample_rows = orig
    out["logits_bf16_planes"] = golden_util.pack_logits_delta(out["logits_fp32"], out.pop("logits_bf16"))
    np.savez_compressed(os.path.join(HERE, "lm_830m_b32.npz"), **out)
    meta = dict(n_steps=N_STEPS, prompts=PROMPTS, text_len=TEXT_LEN, kw=KW, trace_utts=TRACE_UTTS, trace_steps=TRACE_STEPS,
                pinned=pinned, pinned_ckpt_seed=3, ckpt_seed=0, noise_seed="1 + i", data_seed="100 + i")
    with open(os.path.join(HERE, "lm_830m_b32.json"), "w") as f:
        json.dump(meta, f, indent=1, sort_keys=True)
    print("written", time.time() - t0)


if __name__ == "__main__":
    main()
