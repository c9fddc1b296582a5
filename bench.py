#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200-native Qwen3-TTS decode engine.

Metric (BASELINE.json): xRealTime (RTF = audio seconds / wall seconds) and p50 TTFA, Qwen3-TTS-12Hz-1.7B streaming,
chunk_size=8, on 1/2/4/8 B200 (independent replicas, no collective on this path).

A "step" is one streaming voice-clone request of SURVEY.md section 8(d) config 3: an ICL prompt of P=232 positions
(a 30-word reference transcript + a 17-word text + 174 reference codec frames = 13.9 s of reference audio, assembled
by the package's own prompt builder), 128 frames (10.24 s of audio) generated in chunks of 8, every chunk decoded to
24 kHz PCM with the reference's two-phase window policy.  min_new_tokens = max_new_tokens pins the work per step.
Weights are random-init at the real 1.7B geometry, inputs synthetic (no checkpoint / tokenizer exists offline).

  value        RTF with the prompt embeddings already resident in HBM, CUDA-event timed, max over ranks
  e2e          RTF through the public API FasterQwen3TTS.generate_voice_clone_streaming(text, language, ref_audio,
               ref_text): tokenisation, voice-clone prompt, prompt assembly, prefill, decode, codec inside the timed
               region; the reference audio is copied host->device from pinned memory every step (what the upstream
               speaker / codec encoders would consume; those encoders themselves are absent offline and answered by
               stand-ins) and every PCM chunk is read back to the host
  roofline     persistent decode kernel, algorithmic bytes per launch (SURVEY.md 8(d) B_alg) / CUDA-event launch time
               against the MEASURED HBM copy bandwidth in MEASURED_PEAKS.json
  config4      BASELINE config 4 on the same GPU(s): `--batch` (32) concurrent requests per GPU decoded by the batched
               persistent kernel (all requests share every pass over the weight tape), aggregate RTF with and without
               the per-request codec decode, and its own roofline (weights once per step, KV per row)
  gpu_reference the reference's METHOD (static KV + mask table + CUDA graphs + per-frame eager glue,
               baseline/reference_method.py) on the same GPU, same synthetic weights, same request -- the stand-in
               SURVEY 8(d)(ii) prescribes because upstream qwen_tts cannot be installed offline
  cpu_baseline / --impl reference: the CPU oracle (torch eager fp32, dynamic KV) on a bounded sample, host threads
  --sweep      chunk (BASELINE config 5: chunk_size in {1,2,4,8,16}) / prompt (TTFA over P in {10,40,96,232} split
               into prefill, first chunk, first window) ; --size 0.6B = config 2
  --dump-outputs DIR  what the last timed step returned: its PCM (pcm.npy, float32, with the chunk lengths in
               chunk_samples.npy), or its codes with --no-codec (codes.npy); seeded inputs, so two builds can be compared
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "faster-qwen3-tts_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

FRAME_S = 0.08  # 1920 samples @ 24 kHz (ggml_backend.py:22)
METRIC = "xRealTime (RTF) Qwen3-TTS-1.7B streaming chunk_size=8 (p50 TTFA in config)"
WORDS = ("the quick brown fox jumps over a lazy dog and then runs far away into the deep green forest where nobody "
         "can find it again").split()


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--size", default="1.7B", choices=["1.7B", "0.6B"])
    ap.add_argument("--prompt", type=int, default=232)
    ap.add_argument("--frames", type=int, default=128)
    ap.add_argument("--chunk", type=int, default=8)
    ap.add_argument("--ref-frames", type=int, default=174, help="ICL reference codec frames (13.9 s of reference audio)")
    ap.add_argument("--no-codec", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true")
    ap.add_argument("--no-stateful", action="store_true", help="skip the extra legs with the stateful streaming codec")
    ap.add_argument("--batch", type=int, default=32, help="config 4: concurrent requests per GPU (0/1 disables the leg)")
    ap.add_argument("--batch-prompt", type=int, default=40)
    ap.add_argument("--batch-steps", type=int, default=2)
    ap.add_argument("--sweep", default="none", choices=["none", "chunk", "prompt", "all"])
    ap.add_argument("--num-ctas", type=int, default=0)
    ap.add_argument("--cpu-frames", type=int, default=64)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (PCM, or codes with --no-codec) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    return args


DUMP_BUDGET = 64 << 20   # bytes, all dumped arrays together


def dump_outputs(out_dir, arrays):
    """Save each array as out_dir/<name>.npy.  Above DUMP_BUDGET in all, each array is replaced by the same fixed, seeded
    sample of its flattened elements (in order), so that two runs with the same arguments stay comparable."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_BUDGET:
            keep = a.size * DUMP_BUDGET // total
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ----------------------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md recipe)
# ----------------------------------------------------------------------------------------------------------------
class Clocks:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle on host cores
# ----------------------------------------------------------------------------------------------------------------
def cpu_oracle_run(args, frames: int):
    """prefill(P) + `frames` decode frames on the CPU oracle (fp32 eager -- torch CPU bf16 GEMV is ~50x slower than
    fp32 on this host -- dynamic KV).  Returns (rtf, seconds, threads, description)."""
    from oracle import qwen3_tts_oracle as O
    # torch-eager GEMV chains stop scaling (and collapse under OpenMP oversubscription) -- use at most 16 threads and
    # report the number used
    nthreads = min(os.cpu_count() or 1, 16)
    torch.set_num_threads(nthreads)
    cfg = O.cfg_1p7b() if args.size == "1.7B" else O.cfg_0p6b()
    t0 = time.time()
    W = {}
    g = torch.Generator().manual_seed(0)

    def fill(shape, std):
        return (torch.empty(shape, dtype=torch.float32).normal_(0.0, std, generator=g))

    def stack(prefix, c):
        qd, kd = c.num_attention_heads * 128, c.num_key_value_heads * 128
        for li in range(c.num_hidden_layers):
            p = f"{prefix}.layers.{li}."
            for n, sh in (("self_attn.q_proj", (qd, c.hidden_size)), ("self_attn.k_proj", (kd, c.hidden_size)),
                          ("self_attn.v_proj", (kd, c.hidden_size)), ("self_attn.o_proj", (c.hidden_size, qd)),
                          ("mlp.gate_proj", (c.intermediate_size, c.hidden_size)),
                          ("mlp.up_proj", (c.intermediate_size, c.hidden_size)),
                          ("mlp.down_proj", (c.hidden_size, c.intermediate_size))):
                W[p + n + ".weight"] = fill(sh, 0.02)
            for n, k in (("input_layernorm", c.hidden_size), ("post_attention_layernorm", c.hidden_size),
                         ("self_attn.q_norm", 128), ("self_attn.k_norm", 128)):
                W[p + n + ".weight"] = torch.ones(k, dtype=torch.float32)
        W[prefix + ".norm.weight"] = torch.ones(c.hidden_size, dtype=torch.float32)

    Ht, Hp = cfg.talker.hidden_size, cfg.predictor.hidden_size
    stack("talker.model", cfg.talker)
    W["talker.model.codec_embedding.weight"] = fill((cfg.talker.vocab_size, Ht), 1.0)
    W["talker.codec_head.weight"] = fill((cfg.talker.vocab_size, Ht), 0.08)
    stack("talker.code_predictor.model", cfg.predictor)
    for i in range(15):
        W[f"talker.code_predictor.model.codec_embedding.{i}.weight"] = fill((cfg.predictor.vocab_size, Ht), 1.0)
        W[f"talker.code_predictor.lm_head.{i}.weight"] = fill((cfg.predictor.vocab_size, Hp), 0.08)
    if cfg.has_mtp_projection:
        W["talker.code_predictor.small_to_mtp_projection.weight"] = fill((Hp, Ht), 0.02)
        W["talker.code_predictor.small_to_mtp_projection.bias"] = fill((Hp,), 0.02)
    om = O.OracleModel(cfg, W, max_pos=args.prompt + frames + 8)
    tie, tth, tpe = O.make_inputs(cfg, args.prompt, 1, seed=0, dtype=torch.float32)
    import numpy as np
    u = np.random.default_rng(0).random((frames + 1, 16), dtype=np.float32)
    t_build = time.time() - t0
    with torch.inference_mode():
        t1 = time.time()
        codes = O.generate(om, tie, tth, tpe, max_new_tokens=frames, min_new_tokens=frames, uniforms=u,
                           max_seq_len=2048)
        dt = time.time() - t1
    n = int(codes.shape[0])
    desc = (f"CPU oracle (torch eager FP32, dynamic KV): prefill P={args.prompt} + {n} frames of the {args.size} "
            f"workload, {nthreads} threads, {dt:.1f}s (weights built in {t_build:.0f}s, untimed); NO codec decode, "
            f"fp32 not bf16 -- a reported baseline on a bounded sample, not a like-for-like arm")
    return n * FRAME_S / dt, dt, nthreads, desc


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals = []
    for i in range(args.warmup + args.steps):
        rtf, dt, nth, desc = cpu_oracle_run(args, args.cpu_frames)
        if i >= args.warmup:
            vals.append((rtf, dt))
        if i == 0 and args.warmup > 0 and dt > 60:  # keep the whole run within minutes
            args.warmup = 0
            vals.append((rtf, dt))
            break
    v = statistics.mean(x[0] for x in vals)
    ms = statistics.mean(x[1] for x in vals) * 1000
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "x realtime", "n_gpus": args.gpus,
        "steps": len(vals), "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, P=args.prompt, sample=f"prefill + {args.cpu_frames} frames per step, no codec decode",
                                  same_config=False,
                                  note="CPU oracle port in fp32 on <=16 host threads, ONE process whatever --gpus says: "
                                       "a reported baseline, not the reference's CUDA-graph backend (see gpu_reference in "
                                       "the b200 line for that method on the GPU)"),
        "cpu_baseline": {"value": v, "unit": "x realtime", "cores": nth, "kind": "port", "sample": desc},
        "e2e": {"value": v, "unit": "x realtime", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def workload_config(args, P=None, **extra):
    c = {"workload": f"Qwen3-TTS-12Hz-{args.size} streaming voice-clone (SURVEY 8(d) config 3): ICL prompt P={P or args.prompt} "
                     f"({args.ref_frames} reference frames), {args.frames} frames, chunk_size={args.chunk}, "
                     f"T=0.9 top_k=50 top_p=1.0 penalty=1.05, min_new_tokens=max_new_tokens (fixed work)",
         "batch_per_gpu": 1, "parallelism": f"replicas x{args.gpus} (no collective)",
         "l2_policy": "per-step weight stream (3.2 GB tape) exceeds the 126 MB L2; no explicit flush needed",
         "codec_policy": "reference window policy (model.py:1052-1135), sample-identical; Phase 1 of a request with an ICL "
                         "reference runs on a copy of that reference's warmed decoder stream (cached per voice like the voice "
                         "prompt; the e2e leg clears both caches every step, so it pays the reference decode each time)"}
    c.update(extra)
    return c


# ----------------------------------------------------------------------------------------------------------------
# B200 arm
# ----------------------------------------------------------------------------------------------------------------
def craft_request(model, P_target: int, ref_frames: int):
    """(text, ref_text, ref_audio, prepared tuple) whose ICL prompt (non_streaming_mode=True: text first, then the
    reference frames, model.py:704-716) has exactly P_target positions when reachable."""
    import numpy as np
    ref_text = " ".join((WORDS * 3)[:30])
    audio = (np.zeros(int(round(ref_frames / 12.5 * 24000)), dtype=np.float32), 24000)
    best = None
    for nw in range(2, 60):
        text = " ".join((WORDS * 4)[:nw])
        prep = model._prepare_generation(text, ref_audio=audio, ref_text=ref_text, language="English",
                                         non_streaming_mode=True)
        P = int(prep[3].shape[1])
        if best is None or abs(P - P_target) < abs(best[0] - P_target):
            best = (P, text, prep)
        if P >= P_target:
            break
    P, text, prep = best
    return text, ref_text, audio, prep, P


def run_b200(args):
    import numpy as np
    import torch.distributed as dist
    from faster_qwen3_tts import synthetic
    from faster_qwen3_tts.model import FasterQwen3TTS

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = synthetic.make_config(args.size)
    B4 = args.batch if args.batch > 1 else 0
    model = FasterQwen3TTS.from_synthetic(args.size, device=f"cuda:{local}", dtype=torch.bfloat16, max_seq_len=2048,
                                          seed=1234 + rank, num_ctas=args.num_ctas, with_codec=not args.no_codec,
                                          max_batch=max(B4, 1))
    eng = model.engine
    eng.time_kernels = True
    tcfg = cfg.talker_config
    text, ref_text, ref_audio, prep, P = craft_request(model, args.prompt, args.ref_frames)
    _, _, _, tie, tam, tth, tpe, ref_codes = prep
    if args.no_codec:
        ref_codes = None
    pinned_audio = torch.from_numpy(ref_audio[0]).pin_memory()
    kw = dict(max_new_tokens=args.frames, min_new_tokens=args.frames, chunk_size=args.chunk)
    chunk_ms, ttfa_ms = [], []

    def step_resident(timed: bool, chunk=None, prompt=None, keep=None):
        """prompt resident in HBM; codes -> PCM per chunk on device.  Returns frames.  `keep`: a list that receives a
        device copy of every chunk the caller gets (PCM, or codes without the codec)."""
        torch.manual_seed(rank * 1000 + len(ttfa_ms))
        e0 = torch.cuda.Event(enable_timing=True)
        e0.record()
        first = None
        n = 0
        k2 = dict(kw)
        if chunk is not None:
            k2["chunk_size"] = chunk
        a = prompt or (tie, tam, tth, tpe)
        gen = model.stream_from_embeds(*a, ref_codes=ref_codes if prompt is None else None, to_host=False, **k2)
        for pcm, sr, t in gen:
            if first is None:
                first = torch.cuda.Event(enable_timing=True)
                first.record()
            n += t["chunk_steps"]
            if keep is not None:
                keep.append(pcm.clone())
            if timed and "kernel_ms" in t:
                chunk_ms.append(t["kernel_ms"])
        if timed and first is not None:
            first.synchronize()
            ttfa_ms.append(e0.elapsed_time(first))
        return n

    def step_e2e():
        """public API with HOST inputs: text + reference audio in, PCM chunks out (H2D / D2H inside the timed region)"""
        h2d = d2h = 0
        t0 = time.perf_counter()
        a_dev = pinned_audio.to(dev, non_blocking=True)   # what the upstream speaker / codec encoders would read
        h2d += pinned_audio.numel() * pinned_audio.element_size()
        n = 0
        t_first = None
        for pcm, sr, t in model.generate_voice_clone_streaming(
                text, "English", ref_audio=ref_audio, ref_text=ref_text, non_streaming_mode=True,
                max_new_tokens=args.frames, min_new_tokens=args.frames, chunk_size=args.chunk):
            if t_first is None:
                t_first = time.perf_counter() - t0
            d2h += pcm.nbytes
            n += t["chunk_steps"]
        del a_dev
        return n, h2d, d2h, t_first

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_resident(False)
    clocks = Clocks(local)
    if rank == 0:
        clocks.start()
    barrier()
    l0 = eng.launch_count + model.codec_launches()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    frames = 0
    last = [] if args.dump_outputs and rank == 0 else None
    for i in range(args.steps):
        frames += step_resident(True, keep=last if i == args.steps - 1 else None)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    launches = eng.launch_count + model.codec_launches() - l0
    clk = clocks.stop() if rank == 0 else None
    if last is not None:
        if args.no_codec:   # codes [frames, 16] per chunk
            dump_outputs(args.dump_outputs, {"codes": torch.cat(last).cpu().double().numpy()})
        else:               # 24 kHz PCM per chunk: the samples in order, and where the chunks split them
            dump_outputs(args.dump_outputs, {"pcm": torch.cat(last).float().cpu().numpy(),
                                             "chunk_samples": np.array([c.numel() for c in last], dtype=np.float64)})
    # ---- extra leg: the same request with the STATEFUL streaming codec (SURVEY 8(f) item 2; not the headline: its
    # Phase-2 audio is the non-streaming decode rather than the reference's 25-frame-context windows)
    sc = None
    if not args.no_codec and not args.no_stateful:
        model.streaming_codec = "stateful"
        step_resident(False)
        n0, k0 = len(ttfa_ms), len(chunk_ms)
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        fr_s = sum(step_resident(True) for _ in range(args.steps))
        s1.record()
        barrier()
        sc = {"ms": s0.elapsed_time(s1), "frames": fr_s, "ttfa_ms_p50": statistics.median(ttfa_ms[n0:])}
        del ttfa_ms[n0:], chunk_ms[k0:]
        model.streaming_codec = "window"
    # ---- e2e leg
    model._voice_prompt_cache.clear()
    step_e2e()   # one untimed pass (lazy allocations of the prompt path)
    barrier()
    t0 = time.perf_counter()
    e_frames = h2d = d2h = 0
    e_ttfa = []
    for _ in range(args.steps):
        model._voice_prompt_cache.clear()   # every step pays the voice-clone prompt, like a new speaker ...
        if hasattr(model.model.model.speech_tokenizer, "clear_reference_cache"):
            model.model.model.speech_tokenizer.clear_reference_cache()   # ... and the codec-side warm-up of its reference
        n, a, b, tf = step_e2e()
        e_frames += n
        h2d, d2h = a, b
        e_ttfa.append(tf * 1000)
    torch.cuda.synchronize()
    e_s = time.perf_counter() - t0
    # the reference's own TTFA recipe repeats requests with ONE voice (prompt cache hit, benchmarks/throughput.py:29-75):
    # the same public call without clearing the caches, outside the timed region of `e2e`
    e_ttfa_cached = [step_e2e()[3] * 1000 for _ in range(3)]
    # ---- config 4: B concurrent requests per GPU through the batched kernel
    c4 = None
    if B4:
        c4 = run_config4(args, model, cfg, dev, rank, barrier)
    from faster_qwen3_tts.replicas import aggregate
    vals = [ms, e_s * 1000] + ([c4["ms_decode"], c4["ms_codec"], c4["ms_stateful"]] if c4 else [0.0, 0.0, 0.0]) + [sc["ms"] if sc else 0.0]
    cnts = [frames, e_frames] + ([c4["frames_decode"], c4["frames_codec"], c4["frames_stateful"]] if c4 else [0, 0, 0]) + [sc["frames"] if sc else 0]
    mx, sm = aggregate(vals, cnts, device=dev)
    ms, e_ms = mx[0], mx[1]
    frames, e_frames = sm[0], sm[1]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    value = frames * FRAME_S / (ms / 1000)
    e2e = e_frames * FRAME_S / (e_ms / 1000)
    # ---- roofline of the persistent decode kernel
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_kind = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    t_bytes, p_bytes = eng.tape_bytes()
    esz = 2
    Lt, nKV = tcfg.num_hidden_layers, tcfg.num_key_value_heads
    pbar = P + (args.frames - 1) / 2.0
    kv_row = Lt * 2 * nKV * 128 * esz
    kv_bytes = kv_row * (pbar + 1)
    from faster_qwen3_tts.weights import stack_config
    pc = stack_config(cfg.code_predictor_config)
    pred_layers = pc["num_hidden_layers"] * (2 * pc["hidden_size"] * (pc["num_attention_heads"] + pc["num_key_value_heads"]) * 128
                                             + 3 * pc["hidden_size"] * pc["intermediate_size"]) * esz
    pred_heads = 15 * pc["vocab_size"] * pc["hidden_size"] * esz
    mtp = (tcfg.hidden_size * pc["hidden_size"] * esz) if cfg.has_mtp else 0
    w_alg = t_bytes + pred_layers + pred_heads + mtp      # every distinct weight byte once per frame (SURVEY 8(d))
    b_alg = w_alg + kv_bytes
    b_stream = t_bytes + kv_bytes + p_bytes
    k_ms = statistics.mean(chunk_ms) if chunk_ms else None
    traffic, traffic_file = None, None
    for f in ("r2_decode_kernel_ncu.csv", "r1c_decode_kernel_ncu.csv"):
        if os.path.exists(os.path.join(ROOT, "profiles", f)):
            traffic_file = f
            break
    try:  # DRAM bytes of one launch from the committed ncu capture of this kernel (profiles/)
        for line in open(os.path.join(ROOT, "profiles", traffic_file)):
            f = line.strip().split(",")
            if len(f) == 4 and f[0] == "0" and f[1] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                traffic = (traffic or 0.0) + float(f[3]) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[f[2]]
    except Exception:
        traffic = None
    talker = None
    try:
        ppos = int(pbar)
        xh = torch.randn(tcfg.hidden_size, device=dev).to(torch.bfloat16)
        for _ in range(3):
            eng.talker_step(xh, ppos)
        torch.cuda.synchronize()
        t0e, t1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0e.record()
        for _ in range(20):
            eng.talker_step(xh, ppos)
        t1e.record(); t1e.synchronize()
        ts_ms = t0e.elapsed_time(t1e) / 20
        ts_bytes = t_bytes - tcfg.vocab_size * tcfg.hidden_size * esz + kv_row * (ppos + 1)
        talker = {"position": ppos, "ms": ts_ms, "bytes": ts_bytes, "achieved": ts_bytes / (ts_ms / 1000) / 1e9,
                  "frac": ts_bytes / (ts_ms / 1000) / 1e9 / peak,
                  "note": "one launch per step here (launch + pipeline fill included); inside the fused loop the step is shorter"}
    except Exception as ex:  # never let the extra measurement break the bench line
        talker = {"error": str(ex)[:120]}
    roof = None
    if k_ms:
        ach = b_alg * args.chunk / (k_ms / 1000) / 1e9
        roof = {"bound": "hbm", "kernel": "fq3_decode_kernel<bf16> (one launch = one %d-frame chunk)" % args.chunk,
                "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                "traffic_source": ("ncu --set full capture of one 8-frame launch, profiles/" + traffic_file) if traffic_file else None,
                "peak_source": peak_kind, "alg_bytes_per_frame": b_alg, "launch_ms": k_ms,
                "streamed_bytes_per_frame": b_stream, "streamed_frac": b_stream * args.chunk / (k_ms / 1000) / 1e9 / peak,
                "ms_per_frame": k_ms / args.chunk, "talker_step": talker}
    out = {
        "metric": METRIC, "value": value, "unit": "x realtime", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(args, P=P, ttfa_ms_p50=statistics.median(ttfa_ms) if ttfa_ms else None,
                                  ttfa_ms_e2e_p50=statistics.median(e_ttfa) if e_ttfa else None,
                                  ttfa_ms_e2e_cached_voice_p50=statistics.median(e_ttfa_cached) if e_ttfa_cached else None,
                                  codec=not args.no_codec, ctas=eng.num_ctas, ref_frames=args.ref_frames,
                                  e2e_path="FasterQwen3TTS.generate_voice_clone_streaming(text, language, ref_audio, "
                                           "ref_text, non_streaming_mode=True): tokeniser + voice prompt + prompt "
                                           "assembly + prefill inside TTFA; speaker/codec ENCODERS are stand-ins"),
        "e2e": {"value": e2e, "unit": "x realtime", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": int(launches), "clocks": clk, "roofline": roof,
    }
    if c4:
        fd, fc = sm[2], sm[3]
        md, mc = mx[2], mx[3]
        kms = c4["kernel_ms"]
        pb4 = c4["P"] + (args.frames - 1) / 2.0
        bytes_step = w_alg + B4 * kv_row * (pb4 + 1)     # weights once per step, KV per row (SURVEY 8(d))
        ach4 = bytes_step * args.chunk / (kms / 1000) / 1e9 if kms else None
        out["config4"] = {
            "workload": f"BASELINE config 4: {B4} concurrent requests per GPU, P={c4['P']} (left-padded batch, mixed lengths "
                        f"{c4['lens'][0]}..{c4['lens'][1]}), {args.frames} frames each, chunk_size={args.chunk}, independent "
                        f"uniforms per request; batched persistent kernel (one launch per chunk for all requests)",
            "requests_per_gpu": B4, "n_gpus": world,
            "rtf_aggregate_decode": fd * FRAME_S / (md / 1000), "rtf_aggregate_with_codec": fc * FRAME_S / (mc / 1000) if mc else None,
            "rtf_aggregate_with_stateful_codec": sm[4] * FRAME_S / (mx[4] / 1000) if mx[4] else None,
            "ms_per_frame_step": kms / args.chunk if kms else None,
            "speedup_vs_batch1_decode": (fd * FRAME_S / (md / 1000)) / (value * 1.0) if value else None,
            "roofline": {"bound": "hbm", "kernel": "fq3_decode_batch_kernel<bf16> (one launch = one chunk of all requests)",
                         "achieved": ach4, "peak": peak, "unit": "GB/s", "frac": ach4 / peak if ach4 else None,
                         "alg_bytes_per_step": bytes_step, "launch_ms": kms,
                         "note": "weights once per step + KV of every row; frac measures HBM use, aggregate RTF the gain"},
        }
    if sc:
        out["stateful_codec"] = {
            "what": "same request, streaming_codec='stateful' (fq3_codec_stream_decode: every chunk costs its own 8 frames; "
                    "audio = the non-streaming decode; the ICL reference frames warm the stream state before the first chunk)",
            "rtf": sm[5] * FRAME_S / (mx[5] / 1000) if mx[5] else None, "ttfa_ms_p50_rank0": sc["ttfa_ms_p50"]}
    if not args.no_gpu_reference and not args.no_codec:
        try:
            out["gpu_reference"] = run_gpu_reference(args, model, cfg, dev, (tie, tam, tth, tpe), ref_codes)
            gr = out["gpu_reference"]
            out["gpu_reference"]["engine_over_reference_method"] = {
                "rtf": value / gr["rtf"] if gr.get("rtf") else None,
                "ttfa": gr["ttfa_ms_p50"] / statistics.median(ttfa_ms) if gr.get("ttfa_ms_p50") and ttfa_ms else None}
        except Exception as ex:
            out["gpu_reference"] = {"error": repr(ex)[:300]}
    if args.sweep != "none":
        out["sweeps"] = run_sweeps(args, model, cfg, dev, step_resident, chunk_ms, ttfa_ms)
    if not args.no_cpu_baseline and world == 1:
        try:
            rtf, dt, nth, desc = cpu_oracle_run(args, args.cpu_frames)
            out["cpu_baseline"] = {"value": rtf, "unit": "x realtime", "cores": nth, "kind": "port", "sample": desc}
        except Exception as ex:  # the bench line must still print
            out["cpu_baseline"] = {"value": None, "unit": "x realtime", "cores": os.cpu_count(), "kind": "port",
                                   "sample": f"failed: {ex!r}"}
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def run_config4(args, model, cfg, dev, rank, barrier):
    """B concurrent requests on this GPU: decode-only timing (CUDA events) and decode + per-request codec."""
    from faster_qwen3_tts import synthetic
    B = args.batch
    H = cfg.talker_config.hidden_size
    g = torch.Generator().manual_seed(77 + rank)
    Pm = args.batch_prompt
    lens = [int(x) for x in torch.randint(max(4, Pm - 12), Pm + 1, (B,), generator=g)]
    lens[0] = Pm
    tie = torch.zeros(B, Pm, H, dtype=torch.bfloat16)
    tam = torch.zeros(B, Pm, dtype=torch.long)
    for b, L in enumerate(lens):
        tie[b, Pm - L:] = torch.randn(L, H, generator=g).to(torch.bfloat16)
        tam[b, Pm - L:] = 1
    tpe = torch.randn(H, generator=g).to(torch.bfloat16)
    tth = tpe[None, None].expand(B, 1, H).contiguous()
    tie, tam, tth, tpe = tie.to(dev), tam.to(dev), tth.to(dev), tpe[None, None].to(dev)
    kw = dict(max_new_tokens=args.frames, min_new_tokens=args.frames, chunk_size=args.chunk)
    eng = model.engine
    kms = []

    def run(decode_audio):
        n = 0
        for items in model.stream_batch_from_embeds(tie, tam, tth, tpe, to_host=False, decode_audio=decode_audio, **kw):
            n += sum(t["chunk_steps"] for _, _, _, t in items)
            if eng.last_kernel_ms is not None and not decode_audio:
                kms.append(eng.last_kernel_ms)
        return n

    run(False)
    kms.clear()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fd = 0
    for _ in range(args.batch_steps):
        fd += run(False)
    e1.record()
    barrier()
    ms_d = e0.elapsed_time(e1)
    ms_c, fc = 0.0, 0
    if not args.no_codec:
        run(True)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.batch_steps):
            fc += run(True)
        e1.record()
        barrier()
        ms_c = e0.elapsed_time(e1)
    ms_s, fs = 0.0, 0
    if not args.no_codec and not args.no_stateful:
        model.streaming_codec = "stateful"
        run(True)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.batch_steps):
            fs += run(True)
        e1.record()
        barrier()
        ms_s = e0.elapsed_time(e1)
        model.streaming_codec = "window"
    return {"ms_decode": ms_d, "frames_decode": fd, "ms_codec": ms_c, "frames_codec": fc, "ms_stateful": ms_s,
            "frames_stateful": fs, "kernel_ms": statistics.mean(kms) if kms else None, "P": Pm, "lens": (min(lens), max(lens))}


def run_gpu_reference(args, model, cfg, dev, prompt, ref_codes):
    """The reference's method (CUDA-graphed torch modules + eager glue) on the same weights, same request."""
    from baseline.reference_method import build_reference_method, ref_generate_streaming
    from faster_qwen3_tts.codec import SpeechTokenizer
    m = model.model.model
    talker = m.talker
    tie, tam, tth, tpe = prompt
    t0 = time.time()
    pg, tg = build_reference_method(talker, cfg, device=str(dev), dtype=torch.bfloat16, max_seq_len=2048,
                                    prefill_len=tie.shape[1])
    capture_s = time.time() - t0
    st = SpeechTokenizer(m.speech_tokenizer.decoder, backend="torch")   # upstream's own codec path: torch modules / cuDNN
    kw = dict(max_new_tokens=args.frames, min_new_tokens=args.frames, chunk_size=args.chunk)

    def one():
        talker.rope_deltas = None
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        first = None
        n = 0
        chunks = ref_generate_streaming(talker, tie, tam, tth, tpe, m.config.talker_config, pg, tg, **kw)
        for pcm, sr, t in model._stream_audio(chunks, st, ref_codes, args.chunk, to_host=False):
            if first is None:
                torch.cuda.synchronize()
                first = time.perf_counter() - t0
            n += t["chunk_steps"]
        torch.cuda.synchronize()
        return n, time.perf_counter() - t0, first

    one()
    res = [one() for _ in range(max(2, min(args.steps, 3)))]
    n = sum(r[0] for r in res)
    s = sum(r[1] for r in res)
    del pg, tg
    torch.cuda.empty_cache()
    return {"label": "reference-method stand-in (synthetic weights): static KV + mask table + torch.cuda.CUDAGraph of the "
                     "talker step and of the 15-pass predictor loop + the reference's per-frame eager glue + torch/cuDNN codec "
                     "(baseline/reference_method.py restating talker_graph.py / predictor_graph.py / streaming.py)",
            "rtf": n * FRAME_S / s, "ttfa_ms_p50": statistics.median(r[2] for r in res) * 1000,
            "ms_per_frame": s / n * 1000, "runs": len(res), "graph_capture_s": capture_s}


def run_sweeps(args, model, cfg, dev, step_resident, chunk_ms, ttfa_ms):
    from faster_qwen3_tts import synthetic
    out = {}
    if args.sweep in ("chunk", "all"):   # BASELINE config 5 (benchmarks/chunk_sweep.py:24-99)
        rows = []
        for ch in (1, 2, 4, 8, 16):
            step_resident(False, chunk=ch)
            n0 = len(ttfa_ms)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fr = sum(step_resident(True, chunk=ch) for _ in range(3))
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            rows.append({"chunk_size": ch, "rtf": fr * FRAME_S / dt, "ttfa_ms_p50": statistics.median(ttfa_ms[n0:])})
        out["chunk"] = rows
    if args.sweep in ("prompt", "all"):  # TTFA over P with its three terms (SURVEY 8(d))
        eng = model.engine
        rows = []
        for P in (10, 40, 96, 232):
            pr = synthetic.make_prompt(cfg, P, 25, seed=P, dtype=torch.bfloat16, device=dev)
            step_resident(False, prompt=pr)
            n0 = len(ttfa_ms)
            for _ in range(5):
                step_resident(True, prompt=pr)
            # split: prefill / first chunk / first window, each timed alone with CUDA events
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            from faster_qwen3_tts.generate import begin_fused
            m = model.model.model
            parts = []
            for _ in range(5):
                ev[0].record()
                begin_fused(eng, m.talker, pr[0], pr[1], pr[2], pr[3], m.config.talker_config, model.predictor_graph,
                            model.talker_graph, max_new_tokens=args.frames, min_new_tokens=args.frames, temperature=0.9,
                            top_k=50, top_p=1.0, do_sample=True, repetition_penalty=1.05, uniforms=None)
                ev[1].record()
                codes, res = eng.decode_chunk(args.chunk)
                ev[2].record()
                if m.speech_tokenizer is not None:
                    m.speech_tokenizer.decode({"audio_codes": codes.unsqueeze(0)})
                ev[3].record()
                ev[3].synchronize()
                parts.append([ev[i].elapsed_time(ev[i + 1]) for i in range(3)])
            med = [statistics.median(p[i] for p in parts) for i in range(3)]
            rows.append({"P": P, "ttfa_ms_p50": statistics.median(ttfa_ms[n0:]), "prefill_ms": med[0],
                         "first_chunk_ms": med[1], "first_window_ms": med[2]})
        out["prompt"] = rows
    return out


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
