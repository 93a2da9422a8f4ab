#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (BASELINE.json metric: codec tokens/s at 830M decode).

Workloads (BASELINE.json configs, SURVEY.md section 8d), random-init bf16-representable weights of the giga830M shape
(d=2048, 16 heads, 16 layers, K=4 codebooks, vocab 2048+4), end tokens suppressed so only the reference's length cap stops
generation:
  --workload tts  (default, configs[1]): B=32 independent utterances PER GPU (80 phoneme ids, 150-frame / 3 s prompt ->
                  800 frames / 16 s), every rank decodes DIFFERENT utterances (data seed 100 + global id, one random stream
                  per utterance: seed 1 + global id); weak scaling.  A "step" is one decode step of the whole batch:
                  B frames = B*K codec tokens through every layer, the logit heads and the fused sampler.
  --workload edit (configs[2]): 16 speech-editing utterances in TOTAL (T=800 frames, 160 phonemes, span [300,400)),
                  partitioned over the ranks (voicecraft_b200.distributed.partition), results exchanged with one padded
                  all_gather over NCCL; strong scaling.

    python bench.py [--gpus N] [--steps K] [--warmup W]              our CUDA path (one JSON line on rank 0)
    python bench.py --impl reference ...                            the CPU reference arm (oracle port, all host threads)
    python bench.py --dump-outputs DIR ...                          also write what the timed path returned as DIR/<name>.npy

--steps K times exactly K decode steps after the warm-up, or is refused when one generation cannot hold them; the edit
workload times whole sessions, whose length the workload sets, and takes no --steps.
--dump-outputs: inputs, weights and random streams are fixed by seeds, so two builds run with the same arguments can be
compared output for output.  tts: `tokens` [B, steps so far, K] (every utterance's delayed token rows up to and including
the last timed step) and `logits` [B, K, V] (the logits that step sampled from).  edit: `tokens` [N, K, T'max] (each
edited token matrix, padded with -1) and `lengths` [N].  float32 (token ids are exact), at most 64 MB (beyond that, a
fixed seeded sample of the utterances, their indices in `utterances`); with N > 1 GPUs every rank writes its own
utterances, the names suffixed with _rank<r>.  DIR = bench_outputs/ inside the tree is ignored by git.

value    = whole-job codec tokens/s, device-timed (CUDA events on the launching stream, max over ranks), inputs resident
           in HBM.  tts: K timed steps form a window CENTRED on the mean context of the 16 s generation (ctx 231 -> 881,
           mean 556), so a short --steps run is timed at the same context as a long one; the steps before the window
           (>= W) are warm-up.  edit: the whole session (prefill + all decode steps) of this rank's utterances.
e2e      = the same metric through the public API (VoiceCraft.inference_tts_many / inference_many) from pinned HOST
           inputs to HOST outputs: prefill + every decode step + H2D/D2H (+ the NCCL gather when N > 1) inside the timed
           region; one untimed warm-up call, then the median of 3.
roofline = dominant kernel by device time (event-per-launch pass over further steps): algorithmic bytes per launch over
           its average launch duration in the timed region, against MEASURED_PEAKS.json; step_roofline = whole step.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

DUMP_LIMIT = 64 << 20


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed decode steps, exactly (600; reference arm: 64); the edit workload times whole sessions")
    ap.add_argument("--warmup", type=int, default=None, help="untimed decode steps before them (10; reference arm: 2)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="tts", choices=["tts", "edit"])
    ap.add_argument("--model", default="830M")
    ap.add_argument("--batch", type=int, default=None, help="tts: utterances per GPU (32); edit: utterances in total (16)")
    ap.add_argument("--codebooks", type=int, default=4)
    ap.add_argument("--text-len", type=int, default=None)
    ap.add_argument("--prompt", type=int, default=None)
    ap.add_argument("--kv", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--cpu-steps", type=int, default=4, help="decode steps of the bounded CPU baseline sample")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-repeats", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the timed path returned as DIR/<name>.npy")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    if a.impl == "ours" and a.workload == "edit" and a.steps is not None:
        ap.error("--steps: the edit workload times whole editing sessions, whose length the workload sets")
    if a.steps is None:
        a.steps = 64 if a.impl == "reference" else 600
    if a.warmup is None:
        a.warmup = 2 if a.impl == "reference" else 10
    if a.warmup < 0:
        ap.error("--warmup must be >= 0")
    if a.batch is None:
        a.batch = 32 if a.workload == "tts" else 16
    if a.text_len is None:
        a.text_len = 80 if a.workload == "tts" else 160
    if a.prompt is None:
        a.prompt = 150 if a.workload == "tts" else 800
    return a


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def make_model(args):
    from voicecraft_b200 import synthetic
    over = {}
    if args.codebooks != 4:
        over["n_codebooks"] = args.codebooks
    cfg = synthetic.make_config(args.model, **over)
    sd = synthetic.make_state_dict(cfg, seed=0)
    end = cfg.eos if cfg.eos > 0 else cfg.eog
    for k in range(cfg.n_codebooks):            # only the length cap ends generation (SURVEY.md section 8c)
        sd[f"predict_layer.{k}.2.bias"][end] = -1e4
        sd[f"predict_layer.{k}.2.bias"][cfg.eog] = -1e4
    return cfg, sd


def make_utterances(args, cfg, ids):
    """utterance with GLOBAL id i: data seed 100 + i (SURVEY.md section 8d) -- every rank of a multi-GPU run decodes
    different utterances"""
    from voicecraft_b200 import synthetic
    return [synthetic.synthetic_utterance(cfg, 100 + i, args.text_len, args.prompt) for i in ids]


def make_model_inputs(args, device=None):          # kept for scripts/
    cfg, sd = make_model(args)
    return cfg, sd, make_utterances(args, cfg, range(args.batch))


class ClockSampler:
    """SM clock and throttle reasons sampled in-process through NVML every few ms DURING the timed region
    (B200_PROFILING.md: a run that saw hw_slowdown / thermal slowdown, or clocks stuck low for no reason, is rejected)."""

    def __init__(self, index, period=0.003):
        self.index, self.period, self.rows, self.stop_flag, self.th, self.err = index, period, [], False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # pragma: no cover
            self.nv, self.err = None, repr(e)

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((sm, rs))
            except Exception as e:  # pragma: no cover
                self.err = repr(e)
                return
            time.sleep(self.period)

    def start(self):
        if self.nv is None:
            return
        self.stop_flag = False
        self.th = threading.Thread(target=self._loop, daemon=True)
        self.th.start()

    def stop(self):
        self.stop_flag = True
        if self.th:
            self.th.join(timeout=1.0)
        if self.nv is None or not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "error": self.err}
        nv = self.nv
        sm = sorted(r[0] for r in self.rows)
        bits = 0
        for _, rs in self.rows:
            bits |= int(rs)
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_sm, "reasons": sorted(n for n, b in names.items() if bits & b),
                "samples": len(sm), "source": "NVML in-process, %.0f ms period, sampled during the timed region" % (self.period * 1e3)}


def algorithmic_bytes(cfg, B, S_mean, kv_bytes):
    """SURVEY.md section 8d: bf16 weights + KV read (B*S tokens) + KV write (B tokens), per decode step."""
    d, L, K = cfg.d_model, cfg.num_decoder_layers, cfg.n_codebooks
    V = 2048 + cfg.n_special
    per_layer = 3 * d * d + d * d + 8 * d * d
    heads = K * ((1024 * d) + V * 1024)
    W = 2 * (L * per_layer + heads)
    kv_tok = L * 2 * d * kv_bytes
    return W, B * S_mean * kv_tok, B * kv_tok


def host_threads():
    """Usable host cores: affinity mask, cgroup CPU quota, capped at 64 (fp32 GEMV-like steps stop scaling earlier)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(p))))
    except Exception:
        pass
    env = os.environ.get("BENCH_CPU_THREADS")
    return int(env) if env else max(1, min(n, 64))


def decode_steps(args, cfg):
    """decode steps of one utterance until the reference's length cap (y_len > x_len * encodec_sr / 5) ends it"""
    return args.text_len * (cfg.encodec_sr // 5) - (args.prompt + 1) - 2


def check_steps(args):
    """--steps is exactly the number of timed decode steps: refuse, before any work, a count one generation cannot hold
    after the warm-up (the CUDA arm also keeps a few steps after the window for its profiled pass)."""
    from voicecraft_b200 import synthetic
    W = args.warmup if args.impl == "reference" else max(3, args.warmup)
    top = decode_steps(args, synthetic.make_config(args.model)) - W - 10
    if not 1 <= args.steps <= top:
        raise SystemExit(f"--steps {args.steps}: a --text-len {args.text_len}, --prompt {args.prompt} generation holds 1 to "
                         f"{top} timed steps after {W} warm-up steps")


def cpu_baseline(args, cfg, sd, utts, steps, threads=None, warm=0):
    """The oracle port of the reference's own batched decode (inference_tts_batch, B copies of one prompt ==
    the compute of B independent utterances of that length) timed on the host cores, bounded sample: `steps` decode
    steps after `warm` untimed ones."""
    from oracle import lm_oracle
    threads = threads or host_threads()
    torch.set_num_threads(threads)
    oracle = lm_oracle.OracleLM(cfg, sd)
    x, x_lens, y = utts[0]
    marks = []
    torch.manual_seed(1)
    B = 32 if args.workload == "tts" else args.batch
    oracle.inference_tts_batch(x, x_lens, y, top_k=40, top_p=1.0, temperature=1.0, stop_repetition=3,
                               batch_size=B, max_steps=warm + steps + 1, on_step=lambda c: marks.append(time.perf_counter()))
    dt = marks[-1] - marks[warm]                   # decode steps only (the first mark is after prefill + first sample)
    n = len(marks) - 1 - warm
    assert n == steps, (n, steps)
    tok_s = B * cfg.n_codebooks * n / dt
    return dict(value=tok_s, unit="codec tokens/s", cores=threads, kind="port",
                sample=f"oracle inference_tts_batch B={B}, {n} decode steps after a {args.text_len + args.prompt + 1}-token "
                       f"prefill and {warm} warm-up steps, fp32, {threads} threads, {dt / n * 1e3:.0f} ms/step"), dt / n


def workload_config(args, cfg, world=1):
    if args.workload == "edit":
        return {"workload": f"giga{args.model} speech-editing infill, {args.batch} independent utterances in total over {world} GPU(s), "
                            f"K={cfg.n_codebooks}, T={args.prompt} frames, text {args.text_len}, span [300,400), generation to the "
                            f"reference's length cap",
                "batch_total": args.batch, "n_codebooks": cfg.n_codebooks, "kv_cache": args.kv,
                "sampling": "top_k=40, top_p=1.0, temperature=1.0, one Philox stream per utterance (seed 1 + id)",
                "l2": "per-step working set (1.65 GB weights + KV) >> 126 MB L2: no flush needed"}
    return {"workload": f"giga{args.model} TTS decode, B={args.batch}/GPU independent utterances (different on every rank), "
                        f"K={cfg.n_codebooks}, text {args.text_len}, prompt {args.prompt} frames, 16 s ctx "
                        f"({args.text_len + args.prompt + 1} -> {args.text_len + args.text_len * 10 + 1})",
            "batch_per_gpu": args.batch, "n_codebooks": cfg.n_codebooks, "kv_cache": args.kv,
            "l2": "per-step working set (1.65 GB weights + >=0.9 GB KV) >> 126 MB L2: no flush needed",
            "sampling": "top_k=40, top_p=1.0, temperature=1.0, one Philox stream per utterance (seed 1 + global id), generated "
                        "inside the sampler kernel"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg, sd = make_model(args)
    utts = make_utterances(args, cfg, range(1))
    steps, warm = args.steps, args.warmup
    cb, ms = cpu_baseline(args, cfg, sd, utts, steps, warm=warm)
    line = {"impl": "reference", "metric": "codec tokens/s (830M TTS decode)", "value": cb["value"], "unit": "codec tokens/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": ms * 1e3, "higher_is_better": True,
            "scaling": "weak" if args.workload == "tts" else "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, cfg, args.gpus), "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "codec tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def dump_outputs(path, arrays, rank, world):
    """--dump-outputs: one float32 DIR/<name>.npy per array (see the module docstring).  Every array is indexed by utterance
    first; above DUMP_LIMIT bytes in all, a fixed seeded sample of the utterances is written, their indices in `utterances`."""
    arrays = {k: np.asarray(v, dtype=np.float32) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        keep = np.sort(np.random.default_rng(0).choice(n, size=max(1, n * DUMP_LIMIT // total - 1), replace=False))
        arrays = {k: a[keep] for k, a in arrays.items()}
        arrays["utterances"] = keep.astype(np.float32)
    os.makedirs(path, exist_ok=True)
    suffix = f"_rank{rank}" if world > 1 else ""
    for name, a in arrays.items():
        np.save(os.path.join(path, name + suffix + ".npy"), a)


def traffic_record(kernel_name):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture of THIS build (profiles/r02_ncu_traffic.json,
    written by scripts/ncu_traffic.py from `ncu --set full`); None when no capture of this kernel is committed."""
    p = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
    if not os.path.exists(p):
        return None
    try:
        rec = json.load(open(p))
    except Exception:
        return None
    for k, v in rec.items():
        if k.split("(")[0].strip() and k.split("(")[0].strip() in kernel_name:
            return v
    return None


class Dist:
    def __init__(self):
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)
            self.dist = dist

    def barrier(self):
        torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            torch.cuda.synchronize()

    def max(self, v):
        if self.world == 1:
            return v
        t = torch.tensor([v], device=self.dev, dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum(self, v):
        if self.world == 1:
            return v
        t = torch.tensor([v], device=self.dev, dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def close(self):
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


def profile_pass(lib, eng, sess, nprof):
    """event-per-launch pass (serialises launches: only the SHARES are used)"""
    import ctypes as C
    lib.vcb_set_option(eng, b"profile", 1)
    for _ in range(nprof):
        sess.step()
    msb = (C.c_double * 7)()
    cnt = (C.c_int64 * 7)()
    lib.vcb_profile_read(eng, msb, cnt, 7)
    lib.vcb_set_option(eng, b"profile", 0)
    return list(msb), list(cnt)


KERNEL_NAMES = ["gemm_w_xT_cluster(tcgen05, cluster split-K)", "attn_rows_kernel(paged KV, TMA bulk, split ctx)",
                "ln_rows_kernel", "(unused)", "sampler_kernel", "step_prep_kernel",
                "mega_step_kernel(persistent decode step: TMA weight/KV ring, tcgen05, stream-K)"]


def run_tts(args, D):
    from voicecraft_b200 import _lib, distributed as vdist
    from voicecraft_b200.voicecraft import VoiceCraft
    rank, world, dev = D.rank, D.world, D.dev
    cfg, sd = make_model(args)
    K, B = cfg.n_codebooks, args.batch
    ids = [rank * B + i for i in range(B)]
    utts = make_utterances(args, cfg, ids)
    seeds = [1 + i for i in ids]
    model = VoiceCraft(cfg)
    model.load_state_dict(sd)
    model = model.to(dev).eval()
    cap = args.text_len * (cfg.encodec_sr // 5)
    S_total = decode_steps(args, cfg)
    W = max(3, args.warmup)
    Ksteps = args.steps                                    # in range: check_steps()
    start = max(W, (S_total - Ksteps) // 2)                # window centred on the mean context of the generation
    model.configure_engine(max_slots=B, max_seq_len=(args.text_len + cap + 64 + 255) // 256 * 256, kv_dtype=args.kv,
                           max_new_tokens=cap + 64)
    xs = [u[0] for u in utts]
    ys = [u[2] for u in utts]
    kw = dict(top_k=40, top_p=1.0, temperature=1.0, stop_repetition=3)
    lib = _lib.load()

    # ------------------------------------------------------------------ value: device-timed decode steps
    sess = model.open_tts_session([x.to(dev) for x in xs], [y.to(dev) for y in ys], seeds=seeds, **kw)
    eng = sess.eng
    sess.sample()
    for _ in range(start):
        sess.step()
    ctx0 = args.text_len + args.prompt + 1 + start
    clocks = ClockSampler(D.local)
    launches0 = lib.vcb_counter(eng, b"launches")
    D.barrier()
    clocks.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(Ksteps):
        sess.step()
    ev1.record()
    D.barrier()
    clk = clocks.stop()
    ms = D.max(ev0.elapsed_time(ev1))
    launches = lib.vcb_counter(eng, b"launches") - launches0
    st = sess.poll()
    assert all(s.n_steps == 1 + start + Ksteps for s in st), [s.n_steps for s in st]
    assert not any(s.done for s in st)
    if args.dump_outputs:
        logits = torch.empty(B * K, sess.V, device=dev)
        _lib.check(lib.vcb_debug_logits(eng, logits.data_ptr(), B * K))
        dump_outputs(args.dump_outputs, {"tokens": np.stack([sess.raw_tokens(i) for i in range(B)]),
                                         "logits": logits.view(B, K, sess.V).cpu()}, rank, world)
    tok_s = world * B * K * Ksteps / (ms * 1e-3)
    ctx1 = ctx0 + Ksteps

    # ------------------------------------------------------------------ roofline: profiled pass (same engine state)
    roof = step_roof = None
    peak, peak_src = peaks()
    kvb = 4 if args.kv == "fp32" else 2
    S_mean = (ctx0 + ctx1) / 2.0
    Wb, KVr, KVw = algorithmic_bytes(cfg, B, S_mean, kvb)
    step_bytes = Wb + KVr + KVw
    step_gbs = step_bytes / (ms / Ksteps * 1e-3) / 1e9
    step_roof = {"bound": "hbm", "achieved": step_gbs, "peak": peak, "unit": "GB/s", "frac": step_gbs / peak,
                 "algorithmic_bytes_per_step": step_bytes, "weights_bytes": Wb, "kv_read_bytes": KVr,
                 "peak_source": peak_src, "ctx_mean": S_mean}
    nprof = min(8, S_total - (start + Ksteps) - 2)
    if rank == 0 and nprof > 0:
        msb, cnt = profile_pass(lib, eng, sess, nprof)
        total = sum(msb)
        shares = {KERNEL_NAMES[i]: {"ms_per_step": msb[i] / nprof, "launches_per_step": cnt[i] / nprof, "share": msb[i] / total}
                  for i in range(7) if cnt[i]}
        S_prof = ctx1 + nprof / 2.0
        dom = max(range(7), key=lambda i: msb[i])
        if dom == 6:
            # the whole step is one launch of the persistent kernel: its algorithmic bytes are the step's (at the MEAN
            # context of the timed window, which is where its average duration is taken)
            bytes_per_launch, ctx_used = step_bytes, S_mean
        elif dom == 1:
            bytes_per_launch, ctx_used = B * (S_mean + 1) * 2 * cfg.d_model * kvb, S_mean
        else:
            bytes_per_launch, ctx_used = Wb / (cnt[0] / nprof), S_mean
        # average launch duration over the TIMED region: the kernel's share of the step (from the event-per-launch pass,
        # which serialises launches, so only the share is used) x the timed step / launches per step
        dur = (msb[dom] / total) * (ms / Ksteps * 1e-3) / (cnt[dom] / nprof)
        ach = bytes_per_launch / dur / 1e9
        tr = traffic_record(KERNEL_NAMES[dom])
        roof = {"bound": "hbm", "kernel": KERNEL_NAMES[dom], "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": tr["dram_bytes_per_launch"] if tr else None,
                "traffic_source": (tr.get("source") if tr else "no ncu --set full capture of this kernel committed under profiles/"),
                "traffic_capture": tr,
                "algorithmic_bytes_per_launch": bytes_per_launch, "avg_launch_us": dur * 1e6,
                "isolated_launch_us": msb[dom] / cnt[dom] * 1e3, "peak_source": peak_src, "ctx": ctx_used, "by_kernel": shares,
                "note": "avg_launch_us = share of the step (event-per-launch pass at ctx %.0f) x timed step / launches per step; "
                        "isolated_launch_us = raw per-launch event time of that pass" % S_prof}
    sess.close()

    # ------------------------------------------------------------------ e2e: public API, host in / host out (+ NCCL gather)
    e2e = None
    if not args.no_e2e:
        xs_h = [x.pin_memory() for x in xs]
        ys_h = [y.pin_memory() for y in ys]
        times, comm = [], 0
        gen_frames = steps_e2e = d2h = 0
        for rep in range(1 + max(1, args.e2e_repeats)):
            D.barrier()
            t0 = time.perf_counter()
            out = model.inference_tts_many(xs_h, ys_h, poll_every=8, seeds=seeds, **kw)
            local = [r[0][0] for r in out]                                  # [K, T_i] on the device
            full = vdist.gather_token_lists(local, ids, world * B)          # padded all_gather over NCCL when N > 1
            res_h = [t.cpu() for t in (full if rank == 0 else local)]
            torch.cuda.synchronize()
            times.append(D.max(time.perf_counter() - t0))
            comm = vdist.last_gather_bytes
            gen_frames = sum(int(r[1].shape[-1]) for r in out)
            steps_e2e = gen_frames // B + K
            d2h = sum(t.numel() * 8 for t in res_h)
        timed = sorted(times[1:])
        dt = timed[len(timed) // 2]
        gen_total = D.sum(gen_frames)
        h2d = sum(x.numel() * 8 for x in xs_h) + sum(y.numel() * 8 for y in ys_h)
        e2e = {"value": gen_total * K / dt, "unit": "codec tokens/s", "h2d_bytes_per_step": h2d / max(steps_e2e, 1),
               "d2h_bytes_per_step": d2h / max(steps_e2e, 1), "seconds": dt, "seconds_first_call": times[0],
               "seconds_all": times[1:], "generated_frames": int(gen_total), "comm_bytes_per_rank": int(comm),
               "note": "median of %d calls after one untimed warm-up call (first-call allocations); prefill + all decode steps + "
                       "polling + H2D of prompts + D2H of tokens%s inside the timed region" %
                       (len(timed), " + all_gather of the token lists over NCCL" if world > 1 else "")}
    cb = None
    if rank == 0 and not args.no_cpu:
        cb, _ = cpu_baseline(args, cfg, sd, utts, args.cpu_steps)
    if rank != 0:
        return None
    frames_s = tok_s / K
    return {"metric": "codec tokens/s (830M TTS decode)", "value": tok_s, "unit": "codec tokens/s", "n_gpus": world,
            "steps": Ksteps, "warmup": start, "ms_per_step": ms / Ksteps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": dict(workload_config(args, cfg, world), ctx_start=ctx0, ctx_end=ctx1,
                           timed_window="steps [%d, %d) of %d: centred on the mean context of the 16 s generation" % (start, start + Ksteps, S_total)),
            "rtf_per_stream": frames_s / (world * B) / cfg.encodec_sr, "frames_per_s": frames_s,
            "clocks": clk, "e2e": e2e, "gpu_launches": int(launches), "decode_path": {"persistent_kernel_grid": int(lib.vcb_counter(eng, b"mega_grid"))},
            "roofline": roof, "step_roofline": step_roof, "cpu_baseline": cb}


def run_edit(args, D):
    """BASELINE.json configs[2]: `args.batch` utterances in total, partitioned over the ranks, gathered with NCCL."""
    from voicecraft_b200 import _lib, distributed as vdist
    from voicecraft_b200.voicecraft import VoiceCraft
    rank, world, dev = D.rank, D.world, D.dev
    cfg, sd = make_model(args)
    K, N = cfg.n_codebooks, args.batch
    utts = make_utterances(args, cfg, range(N))
    mine = vdist.partition([args.prompt] * N, world, rank)
    model = VoiceCraft(cfg)
    model.load_state_dict(sd)
    model = model.to(dev).eval()
    model.configure_engine(max_slots=max(1, N), max_seq_len=2048, max_new_tokens=1400, kv_dtype=args.kv)
    kw = dict(top_k=40, top_p=1.0, temperature=1.0, stop_repetition=-1)
    span = lambda: torch.tensor([[[300, 400]]])
    lib = _lib.load()

    def decode(idx, host):
        if not idx:
            return []
        xs = [utts[i][0].pin_memory() if host else utts[i][0].to(dev) for i in idx]
        ys = [utts[i][2].pin_memory() if host else utts[i][2].to(dev) for i in idx]
        return model.inference_many(xs, ys, [span() for _ in idx], poll_every=8, seeds=[1 + i for i in idx], **kw)

    # ---- value: device-timed session of this rank's share (prefill + decode), inputs resident
    decode(mine[:1] or [0], False)                       # warm-up: engine build, first-call allocations
    clocks = ClockSampler(D.local)
    D.barrier()
    clocks.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = lib.vcb_counter(model._eng, b"launches")
    ev0.record()
    res = decode(mine, False)
    ev1.record()
    D.barrier()
    clk = clocks.stop()
    launches = lib.vcb_counter(model._eng, b"launches") - l0
    ms = D.max(ev0.elapsed_time(ev1))
    # generated frames replace the 100-frame span: T' = T - 100 + generated
    gen_frames_total = D.sum(sum(int(r.shape[-1]) - (args.prompt - 100) for r in res))
    tok_s = gen_frames_total * K / (ms * 1e-3)
    if args.dump_outputs:
        lengths = [int(r.shape[-1]) for r in res]
        tokens = torch.full((len(res), K, max(lengths, default=0)), -1, dtype=torch.int64)
        for i, r in enumerate(res):
            tokens[i, :, : lengths[i]] = r[0].cpu()
        dump_outputs(args.dump_outputs, {"tokens": tokens, "lengths": lengths}, rank, world)

    # ---- e2e: host in -> inference_many -> NCCL gather -> host out
    times, comm, full = [], 0, None
    for rep in range(1 + max(1, args.e2e_repeats)):
        D.barrier()
        t0 = time.perf_counter()
        out = decode(mine, True)
        full = vdist.gather_token_lists([r[0] for r in out], mine, N)
        res_h = [t.cpu() for t in full]
        torch.cuda.synchronize()
        times.append(D.max(time.perf_counter() - t0))
        comm = vdist.last_gather_bytes
    timed = sorted(times[1:])
    dt = timed[len(timed) // 2]
    same = None
    if rank == 0 and world > 1:                       # the gathered result must equal a single-GPU decode of all N utterances
        ref = decode(list(range(N)), False)
        same = all(torch.equal(a[0].cpu(), b.cpu()) for a, b in zip(ref, full))
    if rank != 0:
        return None
    h2d = sum(u[0].numel() * 8 + u[2].numel() * 8 for u in utts)
    d2h = sum(t.numel() * 8 for t in res_h)
    steps = max(1, int(gen_frames_total // max(1, N)))
    return {"metric": "codec tokens/s (830M speech-editing infill)", "value": tok_s, "unit": "codec tokens/s", "n_gpus": world,
            "steps": steps, "warmup": 1, "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": workload_config(args, cfg, world),
            "session_ms": ms, "utterances_per_rank": [len(vdist.partition([args.prompt] * N, world, r)) for r in range(world)],
            "clocks": clk, "gpu_launches": int(launches), "matches_single_gpu": same,
            "e2e": {"value": gen_frames_total * K / dt, "unit": "codec tokens/s", "h2d_bytes_per_step": h2d / steps,
                    "d2h_bytes_per_step": d2h / steps, "seconds": dt, "seconds_first_call": times[0], "seconds_all": times[1:],
                    "comm_bytes_per_rank": int(comm),
                    "note": "median of %d calls after one warm-up; H2D prompts, prefill, decode to the length cap, all_gather of the "
                            "edited token matrices over NCCL, D2H" % len(timed)}}


def main():
    args = parse()
    if args.impl == "reference" or args.workload == "tts":
        check_steps(args)
    if args.impl == "reference":
        return run_reference(args)
    D = Dist()
    line = run_tts(args, D) if args.workload == "tts" else run_edit(args, D)
    D.close()
    if line is not None:
        print(json.dumps(line))


if __name__ == "__main__":
    main()
