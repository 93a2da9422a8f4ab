"""bench.py contract checks: the reference arm (CPU oracle port) prints the one JSON result line, the product arm refuses
to run without a CUDA device (no CPU fallback), --steps is honoured exactly or refused, and (-m gpu) --dump-outputs writes
what the timed path returns."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = ["--model", "tiny", "--batch", "2", "--steps", "2", "--warmup", "1", "--text-len", "8", "--prompt", "10"]
SAMPLING = dict(top_k=40, top_p=1.0, temperature=1.0)


def _run(extra, base=SMALL):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + base + extra, cwd=ROOT, capture_output=True,
                          text=True, timeout=600)


def _line(p):
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, "exactly one JSON line on stdout"
    return json.loads(lines[0])


def test_reference_arm_prints_the_contract_line():
    p = _run(["--impl", "reference"])
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, "exactly one JSON line on stdout"
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="needs a machine without a GPU")
def test_product_arm_has_no_cpu_fallback():
    p = _run(["--no-cpu", "--no-e2e"])
    assert p.returncode != 0
    assert not [l for l in p.stdout.splitlines() if l.startswith("{")], "no bench line may be printed without a GPU"


def test_reference_arm_times_exactly_the_requested_steps():
    """--steps K on the reference arm is K timed CPU decode steps after --warmup W untimed ones (no silent cap)."""
    d = _line(_run(["--impl", "reference", "--steps", "70", "--warmup", "3", "--text-len", "12"]))
    assert d["steps"] == 70 and d["warmup"] == 3
    assert "70 decode steps" in d["cpu_baseline"]["sample"] and "3 warm-up steps" in d["cpu_baseline"]["sample"]


@pytest.mark.parametrize("extra", [["--impl", "reference", "--steps", "100"],          # more than a generation holds
                                   ["--steps", "1000", "--no-cpu", "--no-e2e"],          # the same on the CUDA arm
                                   ["--workload", "edit", "--no-cpu"]])                  # edit times whole sessions
def test_steps_that_cannot_be_honoured_are_refused(extra):
    """Refused up front, before any GPU work, with a message that names --steps; no bench line."""
    p = _run(extra)
    assert p.returncode != 0 and "--steps" in p.stderr, p.stderr[-2000:]
    assert not [l for l in p.stdout.splitlines() if l.startswith("{")]


def _tiny_model(args):
    import bench
    from voicecraft_b200.voicecraft import VoiceCraft
    cfg, sd = bench.make_model(args)
    m = VoiceCraft(cfg)
    m.load_state_dict(sd)
    return bench, cfg, m.cuda().eval()


@pytest.mark.gpu
def test_dump_outputs_are_reproducible_and_steps_are_exact(tmp_path):
    """--dump-outputs (tts) writes, as float32, every utterance's token rows up to the last timed step and that step's
    logits: identical across two runs with the same arguments, and equal to the same decode re-run here through the public
    session API (bench.py's engine configuration, seeds 1 + i)."""
    dumps = []
    for run in ("a", "b"):
        d = _line(_run(["--no-cpu", "--no-e2e", "--dump-outputs", str(tmp_path / run)]))
        assert d["steps"] == 2
        dumps.append({n: np.load(tmp_path / run / f"{n}.npy") for n in ("tokens", "logits")})
    a, b = dumps
    assert all(a[n].dtype == np.float32 and np.array_equal(a[n], b[n]) for n in a)
    B, K, n_rows = 2, 4, 1 + d["warmup"] + 2
    assert a["tokens"].shape == (B, n_rows, K) and a["logits"].shape[:2] == (B, K)

    from voicecraft_b200 import _lib
    args = argparse.Namespace(model="tiny", codebooks=4, batch=B, text_len=8, prompt=10)
    bench, cfg, m = _tiny_model(args)
    utts = bench.make_utterances(args, cfg, range(B))
    cap = args.text_len * (cfg.encodec_sr // 5)
    m.configure_engine(max_slots=B, max_seq_len=(args.text_len + cap + 64 + 255) // 256 * 256, kv_dtype="bf16",
                       max_new_tokens=cap + 64)
    sess = m.open_tts_session([u[0].cuda() for u in utts], [u[2].cuda() for u in utts], seeds=[1 + i for i in range(B)],
                              stop_repetition=3, **SAMPLING)
    try:
        sess.sample()
        for _ in range(n_rows - 1):
            sess.step()
        rows = np.stack([sess.raw_tokens(i) for i in range(B)])
        logits = torch.empty(B * K, sess.V, device="cuda")
        _lib.check(sess.lib.vcb_debug_logits(sess.eng, logits.data_ptr(), B * K))
        logits = logits.view(B, K, sess.V).cpu().numpy()
    finally:
        sess.close()
    assert np.array_equal(a["tokens"], rows)
    assert np.allclose(a["logits"], logits, rtol=0, atol=1e-5)
    assert not np.array_equal(logits[:, 0], logits[:, 1]), "codebooks must have their own logits"


@pytest.mark.gpu
def test_edit_dump_holds_the_edited_token_matrices(tmp_path):
    """--dump-outputs (edit) writes each utterance's edited token matrix, padded with -1, and its length: equal to
    inference_many on the same inputs, span and seeds."""
    base = ["--model", "tiny", "--batch", "2", "--text-len", "8", "--prompt", "420"]
    _line(_run(["--workload", "edit", "--no-cpu", "--e2e-repeats", "1", "--dump-outputs", str(tmp_path)], base=base))
    tokens, lengths = np.load(tmp_path / "tokens.npy"), np.load(tmp_path / "lengths.npy")
    assert tokens.dtype == np.float32 and lengths.dtype == np.float32

    args = argparse.Namespace(model="tiny", codebooks=4, batch=2, text_len=8, prompt=420)
    bench, cfg, m = _tiny_model(args)
    utts = bench.make_utterances(args, cfg, range(2))
    m.configure_engine(max_slots=2, max_seq_len=2048, max_new_tokens=1400, kv_dtype="bf16")
    res = m.inference_many([u[0].cuda() for u in utts], [u[2].cuda() for u in utts], [torch.tensor([[[300, 400]]])] * 2,
                           poll_every=8, seeds=[1, 2], stop_repetition=-1, **SAMPLING)
    assert lengths.tolist() == [r.shape[-1] for r in res]
    assert tokens.shape == (2, cfg.n_codebooks, max(lengths))
    for i, r in enumerate(res):
        L = r.shape[-1]
        assert np.array_equal(tokens[i, :, :L], r[0].cpu().numpy()) and (tokens[i, :, L:] == -1).all()
