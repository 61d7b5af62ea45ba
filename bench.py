"""Benchmark of the SONAR text-embedding hot path (BASELINE.json metric: sentences/sec -> 1024-d).

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a engine
    python bench.py --impl reference --gpus N --steps K ...   # the CPU restatement of the reference path
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's embeddings as .npy

Workload (BASELINE.json configs[1]): text_sonar_basic_encoder architecture (24 layers, d=1024,
16 heads, FFN 8192, vocab 256206, random-init weights), batch 4096 sentences x 128 tokens of
synthetic ids per GPU per step.  A "step" is one pass of the hot path over one batch:
embed -> 24 encoder layers -> final LN -> mean-pool -> [4096,1024] fp32.

* `value`  : whole-job sentences/s with the ids already resident in HBM (CUDA events, max over ranks)
* `e2e`    : same metric through the reference-facing model call with HOST (pinned) ids in and
             HOST embeddings out, copies inside the timed region
* `roofline`: the dominant kernel (tcgen05 GEMM, FFN inner-projection instantiation) timed alone
             with CUDA events on its launch stream, against MEASURED_PEAKS.json
* `cpu_baseline`: the fp32 PyTorch restatement of the fairseq2 op sequence (oracle/, "port") on the
             host cores, on a bounded sample of the same workload (rank 0, N=1 only)
* `predict` : (N=1) the same metric through `TextToEmbeddingModelPipeline.predict(batch_size=4096)` on 65 536
             synthetic strings -- tokenise, length-sort, bucket, collate, H2D, model, D2H -- the public call
* `speech`, `decoder`, `xsim` : (N=1) BASELINE.json configs 3 / 4 / 5 on this GPU (value, roofline fraction, parity
             against the CPU oracle measured in the same run)
* `config5` : (N>1) BASELINE.json config 5 end to end: every rank encodes its shard of 1M/8 synthetic sentences,
             ONE NCCL all-gather assembles [N,1024], `xsim_distributed` mines it (ratio margin, k=4); predictions are
             checked against the fp64 oracle on rows of a 64K x 64K slice
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

BATCH, SEQ, D, FFN, LAYERS, HEADS, VOCAB = 4096, 128, 1024, 8192, 24, 16, 256206
FALLBACK_PEAKS = {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0}


def flops_per_sentence(s: int) -> float:
    """SURVEY §8(d): F(S) = L*S*(2*(4d^2 + 2df) + 4*S*d)."""
    return LAYERS * s * (2.0 * (4 * D * D + 2 * D * FFN) + 4.0 * s * D)


def kernel_source_digest() -> str:
    """sha256 of the sources the dominant kernel is compiled from (ties an ncu capture to the code it measured)."""
    import hashlib

    h = hashlib.sha256()
    for name in ("gemm_tcgen05.cu", "common.cuh", "sonar_b200_internal.h"):
        with open(os.path.join(ROOT, "sonar_b200", "csrc", name), "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


DUMP_BYTES = 64 << 20


def dump_outputs(path: str, name: str, t: torch.Tensor) -> None:
    """Write `t` as `path/<name>.npy` in float32.  An output larger than 64 MB is cut to a fixed sample of its rows (seed 0,
    sorted), the same rows from run to run, so that dumps of two builds compare row for row."""
    import numpy as np

    a = t.detach().float().cpu()
    keep = DUMP_BYTES // (a[0].numel() * 4)
    if a.shape[0] > keep:
        a = a[torch.randperm(a.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values]
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, name + ".npy"), a.numpy())


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return dict(FALLBACK_PEAKS), "fallback"


def synthetic_state_dict(device, layers=LAYERS, vocab=VOCAB, seed=1, std=0.02):
    """Seeded random-init weights of the `basic` architecture under the fairseq2 state-dict names
    (SURVEY §8(d) distributions), generated directly on `device`."""
    g = torch.Generator(device=device).manual_seed(seed)

    def rn(*shape, s=std):
        return torch.randn(*shape, generator=g, device=device, dtype=torch.float32) * s

    sd = {"encoder_frontend.embed.weight": rn(vocab, D, s=D ** -0.5)}
    for i in range(layers):
        p = f"encoder.layers.{i}."
        for name in ("q_proj", "k_proj", "v_proj", "output_proj"):
            sd[p + f"self_attn.{name}.weight"] = rn(D, D)
            sd[p + f"self_attn.{name}.bias"] = rn(D)
        sd[p + "self_attn_layer_norm.weight"] = 1.0 + rn(D)
        sd[p + "self_attn_layer_norm.bias"] = rn(D)
        sd[p + "ffn.inner_proj.weight"] = rn(FFN, D)
        sd[p + "ffn.inner_proj.bias"] = rn(FFN)
        sd[p + "ffn.output_proj.weight"] = rn(D, FFN)
        sd[p + "ffn.output_proj.bias"] = rn(D)
        sd[p + "ffn_layer_norm.weight"] = 1.0 + rn(D)
        sd[p + "ffn_layer_norm.bias"] = rn(D)
    sd["layer_norm.weight"] = 1.0 + rn(D)
    sd["layer_norm.bias"] = rn(D)
    return sd


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap,power.limit")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, pw, plim = [], None, set(), [], None
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            try:  # board power next to the clocks: the step runs under sw_power_cap, this says how close to the limit
                pw.append(float(f[3]))
                if len(f) > 8:
                    plim = float(f[8])
            except ValueError:
                pass
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        pw.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "power_w": pw[len(pw) // 2] if pw else None, "power_limit_w": plim}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def calibrate_cpu_threads() -> int:
    """Pick the torch intra-op thread count that runs an encoder-layer-shaped fp32 GEMM fastest on this host
    (more threads than physical cores / NUMA-local memory can be slower); a few seconds."""
    cores = os.cpu_count() or 1
    cands = sorted({c for c in (cores, cores // 2, cores // 4, 32, 16, 8) if 1 <= c <= cores}, reverse=True)
    a = torch.randn(8192, 1024)
    w = torch.randn(8192, 1024)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        torch.nn.functional.linear(a, w)
        t0 = time.perf_counter()
        for _ in range(3):
            torch.nn.functional.linear(a, w)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def cpu_port_throughput(state_dict_cpu, target_seconds: float, sentences_per_step: int = 64):
    """Time the CPU restatement of the reference path (oracle) on a bounded sample of the workload."""
    from oracle.text_encoder import OracleEncoderConfig, OracleTextEncoder

    torch.set_float32_matmul_precision("high")  # reference precision_context for fp32 (text.py:36-54,255)
    cfg = OracleEncoderConfig(vocab_size=state_dict_cpu["encoder_frontend.embed.weight"].shape[0],
                              num_layers=LAYERS)
    enc = OracleTextEncoder(cfg, state_dict_cpu)
    g = torch.Generator().manual_seed(0)
    ids = torch.randint(4, cfg.vocab_size, (sentences_per_step, SEQ), generator=g)
    enc(ids[:2], None)  # warm-up
    n, t0 = 0, time.perf_counter()
    while True:
        emb, _ = enc(ids, None)
        n += sentences_per_step
        dt = time.perf_counter() - t0
        if dt >= target_seconds:
            break
    return n / dt, n, dt, emb, ids


def run_reference(args):
    """`--impl reference`: the reference's own (CPU, fp32) path -- fairseq2 cannot be installed here, so
    this is the oracle port of its op sequence -- on all host threads.  Rank 0 only."""
    rank, world, _ = dist_env()
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    calibrate_cpu_threads()
    layers, vocab = args.layers or LAYERS, args.vocab or VOCAB  # overrides exist for the CPU test-suite only
    sd = synthetic_state_dict("cpu", layers=layers, vocab=vocab)
    from oracle.text_encoder import OracleEncoderConfig, OracleTextEncoder

    torch.set_float32_matmul_precision("high")
    enc = OracleTextEncoder(OracleEncoderConfig(vocab_size=vocab, num_layers=layers), sd)
    per_step = 16
    ids = torch.randint(4, vocab, (per_step, SEQ), generator=torch.Generator().manual_seed(0))
    for _ in range(max(args.warmup, 1) if args.warmup < 3 else 3):
        enc(ids, None)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        emb, _ = enc(ids, None)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, "sentence_embeddings", emb)
    val = per_step * args.steps / dt
    line = {
        "impl": "reference", "metric": "sentences/sec->1024-d", "value": val, "unit": "sentences/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"text_sonar_basic_encoder arch, batch {BATCH} x seq_len {SEQ} per GPU "
                               f"(each CPU step = a bounded sample of {per_step} sentences x {SEQ} tokens)"
                               + ("" if (layers, vocab) == (LAYERS, VOCAB) else
                                  f" -- REDUCED MODEL ({layers} layers, vocab {vocab}): test-suite smoke run, not a measurement")},
        "cpu_baseline": {"value": val, "unit": "sentences/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": f"{per_step} sentences x {SEQ} tokens x {layers} layers per step, fp32, "
                                   f"host cpu_count={cores}"},
        "e2e": {"value": val, "unit": "sentences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)



# ======================================================================================================
# Secondary configurations (BASELINE.json configs 3, 4, 5) -- extra keys on the same JSON line
# ======================================================================================================
def _timed_ms(fn, iters=3, warm=1):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def synthetic_sentences(n: int, words: int, seed: int = 11):
    """n strings of `words` whitespace words each (drawn from a 50k-word pool) -> SyntheticTokenizer makes
    [lang] + words + [eos] = words + 2 tokens of each."""
    import numpy as np

    rng = np.random.default_rng(seed)
    pool = np.array([f"w{i:x}" for i in range(50000)])
    idx = rng.integers(0, len(pool), size=(n, words))
    return [" ".join(row) for row in pool[idx]]


def bench_predict(model, dev, peaks, n_sent=65536, batch=BATCH, seq=SEQ):
    """The public call: TextToEmbeddingModelPipeline.predict on host strings (reference text.py:173-269)."""
    from sonar_b200.batching import collate, dynamic_bucket
    from sonar_b200.inference_pipelines import TextToEmbeddingModelPipeline
    from sonar_b200.tokenizer import SyntheticTokenizer

    tok = SyntheticTokenizer(vocab_size=VOCAB)
    pipe = TextToEmbeddingModelPipeline(model, tok, device=dev)
    sents = synthetic_sentences(n_sent, seq - 2)
    pipe.predict(sents[: 2 * batch], "eng_Latn", batch_size=batch, target_device="cpu")  # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = pipe.predict(sents, "eng_Latn", batch_size=batch, target_device="cpu")
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    # the host stages alone (tokenise + bucket + collate into pinned memory), same thread model minus the GPU
    enc = tok.create_encoder(lang="eng_Latn")
    t1 = time.perf_counter()
    for group in dynamic_bucket((enc(x) for x in sents), 2 ** 31, len, max_num_examples=batch):
        collate(group, 0, pin_memory=True)
    host = time.perf_counter() - t1
    return {"api": "TextToEmbeddingModelPipeline.predict(list[str], 'eng_Latn', batch_size=4096, target_device='cpu')",
            "sentences": n_sent, "tokens_per_sentence": seq, "value": n_sent / wall, "unit": "sentences/s",
            "wall_s": wall, "host_stages_alone_s": host, "host_share_if_serial": host / wall,
            "output_shape": list(out.shape),
            "note": "wall clock around the whole call; tokenise/bucket/collate run in the prefetch thread and overlap the GPU"}


def bench_speech(dev, peaks):
    """BASELINE config 3: 256 x 10 s synthetic waveforms -> fbank -> 24 Conformer layers -> attention pooler."""
    from oracle.speech_encoder import OracleSpeechConfig, OracleSpeechEncoder, make_synthetic_speech_state_dict
    from oracle.speech_frontend import collate_fbank, waveform_to_fbank
    from sonar_b200 import B200SpeechEncoderModel, PaddingMask, SequenceBatch, sonar_speech_encoder_config
    from sonar_b200.speech_frontend import WaveformToFbank

    n = 256
    ocfg = OracleSpeechConfig()
    sd = make_synthetic_speech_state_dict(ocfg, seed=3)
    model = B200SpeechEncoderModel(sonar_speech_encoder_config("english"), sd, dev)
    g = torch.Generator().manual_seed(0)
    waves = [(torch.randn(160000, generator=g) * 0.05).clamp(-1, 1) for _ in range(n)]  # SURVEY §8(d) config 3
    wd = [w.to(dev) for w in waves]
    conv = WaveformToFbank(dev)

    def run():
        fb, fr = conv(wd)
        return model(SequenceBatch(fb, PaddingMask(torch.tensor(fr), fb.shape[1], fr))).sentence_embeddings

    ms = _timed_ms(run, iters=3, warm=2)
    # same-run A/B of the other relative-position attention kernel (tcgen05: attention_relpos_tc.cu)
    other = "tcgen05" if model.attn_impl == "mma_sync" else "mma_sync"
    model_b = B200SpeechEncoderModel(sonar_speech_encoder_config("english"), sd, dev, attn_impl=other)

    def run_b():
        fb, fr = conv(wd)
        return model_b(SequenceBatch(fb, PaddingMask(torch.tensor(fr), fb.shape[1], fr))).sentence_embeddings

    ms_b = _timed_ms(run_b, iters=3, warm=2)
    ab_rel = float(((run_b() - run()).norm(dim=1) / run().norm(dim=1)).max())
    attn_ab = {"default": model.attn_impl, "utterances_per_s": {model.attn_impl: n / ms * 1e3, other: n / ms_b * 1e3},
               "rel_l2_between_kernels_max": ab_rel}
    del model_b
    # e2e: pinned host waveforms in, host embeddings out
    wp = [w.pin_memory() for w in waves]
    out_host = torch.empty((n, 1024), dtype=torch.float32).pin_memory()

    def run_e2e():
        fb, fr = conv(wp)
        out_host.copy_(model(SequenceBatch(fb, PaddingMask(torch.tensor(fr), fb.shape[1], fr))).sentence_embeddings,
                       non_blocking=True)

    ms_e2e = _timed_ms(run_e2e, iters=2, warm=1)
    flop_per_utt = 499 * 24 * 52.38e6 + 7e9  # SURVEY §8(d)
    peak = float(peaks["bf16_tflops_sustained"])
    val = n / ms * 1e3
    calibrate_cpu_threads()
    oracle = OracleSpeechEncoder(ocfg, sd)
    t0 = time.perf_counter()
    fb, fl = collate_fbank([waveform_to_fbank(w) for w in waves[:2]])
    ref, _, _ = oracle(fb, fl)
    dt = time.perf_counter() - t0
    got = run()[:2].cpu().double()
    cos = torch.nn.functional.cosine_similarity(got, ref.double(), dim=1)
    rel = (got - ref.double()).norm(dim=1) / ref.double().norm(dim=1)
    del model
    return {"workload": "sonar_speech_encoder_eng arch (random init): 256 x 10 s 16 kHz synthetic waveforms, "
                        "fbank + 24 Conformer layers + 3 pooler layers",
            "metric": "utterances/sec->1024-d", "value": val, "unit": "utterances/s", "ms_per_step": ms,
            "e2e": {"value": n / ms_e2e * 1e3, "unit": "utterances/s", "h2d_bytes_per_step": n * 160000 * 4,
                    "d2h_bytes_per_step": n * 1024 * 4},
            "ab_relpos_attention": attn_ab,
            "roofline": {"bound": "tensor", "achieved": val * flop_per_utt / 1e12, "peak": peak, "unit": "TFLOP/s",
                         "frac": val * flop_per_utt / 1e12 / peak,
                         "algorithmic_flop_per_utterance": flop_per_utt},
            "cpu_baseline": {"value": 2 / dt, "unit": "utterances/s", "cores": torch.get_num_threads(), "kind": "port",
                             "sample": f"2 utterances in {dt:.1f}s (fp32 torch oracle incl. fbank)",
                             "parity_vs_gpu": {"one_minus_cos_max": float((1 - cos).max()),
                                               "rel_l2_max": float(rel.max())}}}


def synthetic_decoder_state_dict(dev, layers=24, vocab=VOCAB, seed=3):
    g = torch.Generator(device=dev).manual_seed(seed)

    def rn(*shape, s=0.02):
        return torch.randn(*shape, generator=g, device=dev) * s

    sd = {"decoder_frontend.embed.weight": rn(vocab, D, s=1 / 32)}
    for i in range(layers):
        p = f"decoder.layers.{i}."
        for a in ("self_attn", "encoder_decoder_attn"):
            for nme in ("q_proj", "k_proj", "v_proj", "output_proj"):
                sd[p + f"{a}.{nme}.weight"], sd[p + f"{a}.{nme}.bias"] = rn(D, D), rn(D)
            sd[p + f"{a}_layer_norm.weight"], sd[p + f"{a}_layer_norm.bias"] = 1 + rn(D), rn(D)
        sd[p + "ffn.inner_proj.weight"], sd[p + "ffn.inner_proj.bias"] = rn(FFN, D), rn(FFN)
        sd[p + "ffn.output_proj.weight"], sd[p + "ffn.output_proj.bias"] = rn(D, FFN), rn(D)
        sd[p + "ffn_layer_norm.weight"], sd[p + "ffn_layer_norm.bias"] = 1 + rn(D), rn(D)
    sd["decoder.layer_norm.weight"], sd["decoder.layer_norm.bias"] = 1 + rn(D), rn(D)
    return sd


def bench_decoder(dev, peaks):
    """BASELINE config 4: 512 embeddings, beam 5, max_seq_len 128 through the beam-search generator."""
    import math

    from oracle.text_decoder import OracleDecoderConfig, OracleTextDecoder
    from sonar_b200 import B200TextDecoderModel, sonar_text_decoder_config
    from sonar_b200.generation import BeamSearchSeq2SeqGenerator

    sd = synthetic_decoder_state_dict(dev)
    model = B200TextDecoderModel(sonar_text_decoder_config("basic"), sd, dev)
    n, beam, max_seq_len = 512, 5, 128  # SURVEY §8(d) config 4
    emb = torch.randn((n, D), device=dev, generator=torch.Generator(device=dev).manual_seed(5)) * 0.25 / math.sqrt(D) * 32
    prompt = torch.tensor([3, 256100])
    runs = {}
    out = None
    for label, flag, calls in (("eager", False, 2), ("cuda_graphs", True, 3)):
        gen = BeamSearchSeq2SeqGenerator(model, beam_size=beam, max_seq_len=max_seq_len, pad_idx=0, cuda_graphs=flag)
        walls = []
        for _ in range(calls):  # the first call allocates the KV cache / records the graphs
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = gen(emb, None, prompt, None)
            torch.cuda.synchronize()
            walls.append(time.perf_counter() - t0)
        runs[label] = walls
    dt = min(runs["eager"][1:] + runs["cuda_graphs"][1:])
    steps = max(len(h[0].seq) for h in out.hypotheses if h)
    # e2e: host embeddings in, host token sequences out (the generator's own D2H of hypotheses is inside every call)
    emb_host = emb.cpu().pin_memory()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    gen(emb_host.to(dev, non_blocking=True), None, prompt, None)
    torch.cuda.synchronize()
    dt_e2e = time.perf_counter() - t0
    # the pipelines' default batch (5 sentences x beam 5 = 25 hypothesis rows)
    emb5 = emb[:5].contiguous()
    g5 = BeamSearchSeq2SeqGenerator(model, beam_size=beam, max_seq_len=max_seq_len, pad_idx=0, cuda_graphs=True)
    g5(emb5, None, prompt, None)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    o5 = g5(emb5, None, prompt, None)
    torch.cuda.synchronize()
    d5 = time.perf_counter() - t1
    st5 = max(len(h[0].seq) for h in o5.hypotheses if h)
    # in-run parity at config size: teacher-forced steps at R = 2560 rows, 64 of them against the fp32 CPU oracle
    R = n * beam
    tmax = 8
    model.begin(emb, beam, tmax)
    table = torch.arange(R, dtype=torch.int32, device=dev)[:, None].expand(R, tmax).contiguous()
    gt = torch.Generator().manual_seed(9)
    toks = torch.randint(4, 256000, (R, 3), generator=gt)
    rows = torch.arange(0, R, R // 64)[:64]
    ocfg = OracleDecoderConfig()
    sd_cpu = {k: v.float().cpu() for k, v in sd.items()}
    sd_cpu["final_proj.weight"] = sd_cpu["decoder_frontend.embed.weight"]
    oracle = OracleTextDecoder(ocfg, sd_cpu)
    enc_rows = emb.cpu()[rows // beam][:, None, :]
    worst = 0.0
    for t in range(3):
        lp, tk, _ = model.step(toks[:, t].contiguous().to(dev), table, t)
        ref = oracle.step_lprobs(toks[rows, : t + 1], enc_rows)
        got_lp, got_tk = lp[rows.to(dev)].cpu(), tk[rows.to(dev)].cpu().long()
        worst = max(worst, float((got_lp - torch.gather(ref, 1, got_tk)).abs().max()))
    hyp_tokens = n * beam * steps
    peak = float(peaks["bf16_tflops_sustained"])
    # the step is a SERIES of kernels with different bounds: the GEMMs against the tensor peak, the KV-cache attention against
    # HBM (every hypothesis row reads K and V of all earlier positions in all 24 layers: 2 * 2 B * D per position and layer)
    hbm = float(peaks.get("hbm_gbs", FALLBACK_PEAKS.get("hbm_gbs", 6572.2)))
    kv_bytes = n * beam * D * 4.0 * 24 * steps * (steps + 1) / 2.0
    floor_s = hyp_tokens * 1.63e9 / (peak * 1e12) + kv_bytes / (hbm * 1e9)
    del model, oracle, sd_cpu
    return {"workload": f"text_sonar_basic_decoder arch (random init): {n} embeddings, beam {beam}, max_seq_len {max_seq_len} "
                        f"({steps} steps ran: random-weight hypotheses rarely emit EOS early)",
            "metric": "sentences/sec decoded", "value": n / dt, "unit": "sentences/s", "wall_s": dt, "steps": steps,
            "ms_per_step": dt / steps * 1e3, "hypothesis_tokens_per_s": hyp_tokens / dt,
            "wall_s_by_mode": runs,
            "e2e": {"value": n / dt_e2e, "unit": "sentences/s", "h2d_bytes_per_step": n * D * 4,
                    "d2h_bytes_per_step": n * beam * (max_seq_len * 8 + 12)},
            "batch5_beam5": {"wall_s": d5, "steps": st5, "ms_per_step": d5 / st5 * 1e3},
            "roofline": {"bound": "tensor", "achieved": hyp_tokens * 1.63e9 / dt / 1e12, "peak": peak, "unit": "TFLOP/s",
                         "frac": hyp_tokens * 1.63e9 / dt / 1e12 / peak,
                         "algorithmic_flop_per_hypothesis_token": 1.63e9,
                         "serial_floor": {"frac": floor_s / dt, "floor_s": floor_s, "kv_cache_bytes": kv_bytes,
                                          "note": "GEMM flops / sustained bf16 peak + KV-cache bytes / measured HBM bandwidth: "
                                                  "the kernels run one after the other, so their floors add"}},
            "parity_vs_oracle": {"rows": 64, "of_rows": R, "steps": 3, "max_abs_lprob_err": worst,
                                 "tolerance": "2e-2 + 2e-3*|lprob| (tests/test_gpu_decoder.py)"}}


def oracle_xsim_rows(x, y, rows: int, k: int = 4, margin: str = "ratio"):
    """fp64 NumPy oracle predictions for the first `rows` rows of x against ALL of y (the reverse k-NN is only needed for
    the y rows that appear as forward candidates, so the cost is ~5 * rows * len(y) similarities, not len(x) * len(y))."""
    import numpy as np

    from oracle import xsim as ox

    cos_xy, idx_xy = ox.knn(x[:rows], y, k)
    if margin == "absolute":
        return idx_xy[:, 0]
    cand = np.unique(idx_xy)
    cos_yx, _ = ox.knn(y[cand], x, k)
    avg_y = np.zeros(len(y))
    avg_y[cand] = cos_yx.mean(axis=1)
    denom = (cos_xy.mean(axis=1)[:, None] + avg_y[idx_xy]) / 2.0
    score = cos_xy / denom if margin == "ratio" else cos_xy - denom
    return idx_xy[np.arange(rows), np.argmax(score, axis=1)]


def bench_xsim(dev, peaks):
    """BASELINE config 5 on ONE GPU: k-NN (k=4) of [262144,1024] vs noisy copies + margin scoring on a 64K slice."""
    import numpy as np

    from oracle import xsim as ox
    from sonar_b200 import xsim

    n = m = 262144
    g = torch.Generator(device=dev).manual_seed(0)
    y = torch.randn((m, D), generator=g, device=dev)
    x = y + 0.1 * torch.randn((n, D), generator=g, device=dev) * y.norm(dim=1, keepdim=True) / 32.0  # §8(d) config 5
    ms = _timed_ms(lambda: xsim.knn(x, y, 4), iters=2, warm=1)
    bidir_stats = {}
    ms_bidir = _timed_ms(lambda: xsim.knn_bidir(x, y, 4, bidir_stats), iters=2, warm=1)  # both directions from one pass
    err, _, pred = xsim.xsim(x[:65536], y[:65536], margin="ratio", k=4)
    peak = float(peaks["bf16_tflops_sustained"])
    pairs = n * m / ms * 1e3
    xs, ys = x[:65536].cpu().numpy(), y[:65536].cpu().numpy()
    t0 = time.perf_counter()
    ref_pred = oracle_xsim_rows(xs, ys, 2048)
    dt = time.perf_counter() - t0
    rv, ri = ox.knn(xs[:2048], ys[:16384], 4)
    gv, gi = xsim.knn(x[:2048], y[:16384], 4)
    return {"workload": f"xsim k-NN (k=4) of [{n},1024] x [{m},1024] noisy copies on 1 GPU (one direction)",
            "metric": "xsim pairs/sec", "value": pairs, "unit": "pairs/s", "ms_per_step": ms,
            "xsim_error_64k_ratio_margin": err,
            "bidirectional": {"ms": ms_bidir, "value": 2.0 * n * m / ms_bidir * 1e3, "unit": "pairs/s (both directions scored)",
                              "vs_two_passes": 2.0 * ms / ms_bidir, "overflow_rows_redone": bidir_stats.get("overflow_rows"),
                              "roofline_frac": 2.0 * n * m * D * 1.125 / ms_bidir / 1e9 / peak},
            "roofline": {"bound": "tensor", "achieved": 2.0 * n * m * D / ms / 1e9, "peak": peak, "unit": "TFLOP/s",
                         "frac": 2.0 * n * m * D / ms / 1e9 / peak},
            "cpu_baseline": {"value": 5 * 2048 * 65536 / dt, "unit": "pairs/s", "kind": "port",
                             "sample": f"fp64 numpy oracle, ratio-margin predictions of 2048 rows of the 64K x 64K slice in {dt:.1f}s"},
            "parity_vs_oracle": {"margin_predictions_identical": bool(np.array_equal(pred[:2048].cpu().numpy(), ref_pred)),
                                 "rows": 2048, "top4_indices_identical": bool(np.array_equal(gi.cpu().numpy(), ri))}}


def bench_config5(model, dev, dist, rank, world, local, peaks, per_gpu, S=SEQ, B=BATCH):
    """BASELINE config 5 end to end (SURVEY §8(d)/(e)): sharded encode -> ONE all-gather -> distributed xsim."""
    import math

    import numpy as np

    from sonar_b200 import SequenceBatch, xsim
    from sonar_b200.xsim import xsim_distributed

    ns = per_gpu
    g = torch.Generator(device=dev).manual_seed(77 + rank)
    x_shard = torch.empty((ns, D), dtype=torch.float32, device=dev)

    def ev():
        return torch.cuda.Event(enable_timing=True)

    def max_ms(e0, e1):
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def encode():
        for s0 in range(0, ns, B):
            nb = min(B, ns - s0)
            ids = torch.randint(4, VOCAB, (nb, S), generator=g, device=dev, dtype=torch.int64)
            x_shard[s0:s0 + nb] = model(SequenceBatch(ids, None)).sentence_embeddings

    torch.cuda.synchronize()
    dist.barrier()
    e0, e1 = ev(), ev()
    e0.record()
    encode()
    e1.record()
    torch.cuda.synchronize()
    enc_ms = max_ms(e0, e1)

    x_all = torch.empty((world * ns, D), dtype=torch.float32, device=dev)
    dist.all_gather_into_tensor(x_all, x_shard)  # warm the communicator at this size
    torch.cuda.synchronize()
    dist.barrier()
    e0, e1 = ev(), ev()
    e0.record()
    dist.all_gather_into_tensor(x_all, x_shard)
    e1.record()
    torch.cuda.synchronize()
    ag_ms = max_ms(e0, e1)
    # second set: noisy copies, so the true neighbour of x_i is y_i (SURVEY §8(d))
    y_shard = x_shard + 0.1 * torch.randn((ns, D), generator=g, device=dev) * x_shard.norm(dim=1, keepdim=True) / math.sqrt(D)
    parity = None
    if rank == 0:  # fp64 oracle on rows of a 64K x 64K slice of THIS rank's data (needs ns >= 65536, else all of it)
        sl = min(65536, ns)
        err_s, _, pred_s = xsim.xsim(x_shard[:sl], y_shard[:sl], margin="ratio", k=4)
        xs, ys = x_shard[:sl].cpu().numpy(), y_shard[:sl].cpu().numpy()
        t0 = time.perf_counter()
        rows = min(2048, sl)
        ref_pred = oracle_xsim_rows(xs, ys, rows)
        parity = {"slice": f"{sl} x {sl}", "rows_checked": rows, "oracle_seconds": time.perf_counter() - t0,
                  "predictions_identical": bool(np.array_equal(pred_s[:rows].cpu().numpy(), ref_pred)),
                  "gpu_errors_on_slice": err_s}
    del x_all
    torch.cuda.synchronize()
    dist.barrier()
    xsim_distributed(x_shard, y_shard, margin="ratio", k=4)  # warm-up: workspace allocation, communicator at these sizes
    torch.cuda.synchronize()
    dist.barrier()
    e0, e1 = ev(), ev()
    e0.record()
    for _ in range(2):
        err, n_tot, _ = xsim_distributed(x_shard, y_shard, margin="ratio", k=4)
    e1.record()
    torch.cuda.synchronize()
    xs_ms = max_ms(e0, e1) / 2.0
    if rank != 0:
        return None
    peak = float(peaks["bf16_tflops_sustained"])
    sent_s = n_tot / enc_ms * 1e3
    pairs = 2.0 * n_tot * n_tot  # both k-NN directions are scored ...
    gemm_flop = 2.0 * n_tot * n_tot * D * (1.0 + 1.0 / 8.0)  # ... from ONE pass over x.y^T plus the 1/8-sample threshold pass
    return {"workload": f"{n_tot} synthetic sentences x {S} tokens sharded {ns}/GPU over {world} GPUs; one fp32 all-gather; "
                        f"xsim ratio margin k=4 of [{n_tot},1024] vs noisy copies (both k-NN directions, one pass)",
            "encode": {"value": sent_s, "unit": "sentences/s", "ms": enc_ms,
                       "roofline_frac": sent_s * flops_per_sentence(S) / 1e12 / (world * peak)},
            "all_gather": {"bytes_received_per_rank": (world - 1) * ns * D * 4, "ms": ag_ms,
                           "value": (world - 1) * ns * D * 4 / ag_ms / 1e6, "unit": "GB/s per rank (receive)"},
            "xsim": {"value": pairs / xs_ms * 1e3, "unit": "pairs/s", "ms": xs_ms, "errors": err, "n": n_tot,
                     "includes": "the [N,1024] all-gather of y and the [N,k] all-gather of the reverse lists inside "
                                 "xsim_distributed, L2 normalisation, the 1/8-sample threshold GEMM, ONE bf16 GEMM pass with row "
                                 "top-16 + column filter, fp64 re-ranks, margin scoring, error all-reduce",
                     "tensor_tflops": gemm_flop / xs_ms / 1e9,
                     "roofline_frac": gemm_flop / xs_ms / 1e9 / (world * peak)},
            "parity_vs_oracle": parity}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--seq-len", type=int, default=SEQ)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--cta-group", type=int, default=2)
    ap.add_argument("--ln-fold", type=int, default=0, choices=[0, 1, 2],
                    help="0 = separate LayerNorm kernels (default schedule), 1 = LayerNorms folded into the GEMMs, "
                         "2 = only the attention-block LayerNorm folded")
    ap.add_argument("--epi-groups", type=int, default=1, choices=[1, 2], help="epilogue warpgroups per GEMM CTA")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-secondary", action="store_true", help="N=1: skip the predict / speech / decoder / xsim blocks")
    ap.add_argument("--only", default="", help="N=1: comma list of secondary blocks to run (predict,speech,decoder,xsim)")
    ap.add_argument("--skip-config5", action="store_true", help="N>1: skip the config-5 block")
    ap.add_argument("--config5-per-gpu", type=int, default=125000, help="sentences every rank encodes for config 5")
    ap.add_argument("--layers", type=int, default=0, help="--impl reference only: reduced depth for the CPU test-suite")
    ap.add_argument("--vocab", type=int, default=0, help="--impl reference only: reduced vocabulary for the CPU test-suite")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write the sentence embeddings of the last timed step as "
                         "DIR/sentence_embeddings.npy (float32; with N > 1 the all-gathered [N*batch,1024]; above 64 MB "
                         "a fixed seeded sample of rows)")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the sm_100a engine has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)

    import __graft_entry__

    if rank == 0:
        __graft_entry__.build()
    if dist is not None:
        dist.barrier()
    from sonar_b200 import B200TextEncoderModel, SequenceBatch, ops, sonar_text_encoder_config

    B, S = args.batch, args.seq_len
    sd = synthetic_state_dict(dev)
    model = B200TextEncoderModel(sonar_text_encoder_config("basic"), sd, dev, cta_group=args.cta_group,
                                 ln_fold=args.ln_fold, epi_groups=args.epi_groups)
    # same-box A/B of the engine's schedule variants (clock and power state differ box to box by ~10 %, so variants are only
    # comparable inside one run): (ln_fold, epi_groups)
    variants = {}
    if rank == 0 and world == 1 and not args.skip_secondary:
        for lf_, eg_ in ((0, 1), (0, 2), (2, 2), (1, 2)):
            if (lf_, eg_) != (args.ln_fold, args.epi_groups):
                variants[(lf_, eg_)] = B200TextEncoderModel(sonar_text_encoder_config("basic"), sd, dev,
                                                            cta_group=args.cta_group, ln_fold=lf_, epi_groups=eg_)
    sd_cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu_baseline:
        sd_cpu = {k: v.cpu() for k, v in sd.items()}
    del sd
    torch.cuda.empty_cache()

    g = torch.Generator().manual_seed(1000 + rank)
    ids_host = torch.randint(4, VOCAB, (B, S), generator=g, dtype=torch.int64).pin_memory()
    ids_dev = ids_host.to(dev)
    batch_dev = SequenceBatch(ids_dev, None)  # all rows full length -> padding_mask None (utils.py:18-21)
    gather_buf = torch.empty((world * B, D), dtype=torch.float32, device=dev) if world > 1 else None

    def step_resident():
        out = model(batch_dev).sentence_embeddings
        if dist is not None:  # the one exchange step of the path: assemble [N,1024] on every rank
            dist.all_gather_into_tensor(gather_buf, out)
            return gather_buf
        return out

    out_host = torch.empty((B, D), dtype=torch.float32).pin_memory()

    def step_e2e():
        out = model(SequenceBatch(ids_host, None)).sentence_embeddings  # H2D of the ids inside
        if dist is not None:
            dist.all_gather_into_tensor(gather_buf, out)
        out_host.copy_(out, non_blocking=True)  # D2H of the result
        return out

    def timed(fn, steps, warmup, sample_clocks=False):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        sampler = ClockSampler(local) if sample_clocks else None
        if sampler:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = None
        for _ in range(steps):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        clocks = sampler.stop() if sampler else None
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), clocks, out

    # dominant kernel timed INSIDE the real steps: events recorded by the engine around the middle layer's FFN1 GEMM
    k_ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    k_ev[0].record(); k_ev[1].record()  # materialise the handles
    model.profile_ffn1(*k_ev)
    # e2e is timed in two halves AROUND the resident loop so that the slow drift of the power-capped clock hits both
    # measurements alike (round 1 timed them back to back and e2e came out faster than the copy-free value)
    k_a = args.steps // 2
    k_b = args.steps - k_a
    e2e_a = timed(step_e2e, k_a, args.warmup)[0] if k_a else 0.0
    total_ms, clocks, last_out = timed(step_resident, args.steps, args.warmup, sample_clocks=True)
    if args.dump_outputs and rank == 0:  # now: the e2e steps below reuse gather_buf
        dump_outputs(args.dump_outputs, "sentence_embeddings", last_out)
    in_step_kernel_ms = k_ev[0].elapsed_time(k_ev[1])  # the last timed step's launch
    model.profile_ffn1(None, None)
    e2e_b = timed(step_e2e, k_b, 1)[0]
    e2e_ms = e2e_a + e2e_b
    model.check_inputs()
    value = world * B * args.steps / (total_ms / 1e3)
    e2e_value = world * B * args.steps / (e2e_ms / 1e3)

    # ---- dominant kernel alone: tcgen05 GEMM, FFN inner-projection instantiation (bias+ReLU, bf16 out) ----
    peaks, peak_kind = load_peaks()
    roofline = None
    if rank == 0:
        T = B * S
        a = torch.randn((T, D), device=dev, dtype=torch.float32).to(torch.bfloat16)
        w = model._layer_bufs[0]["w1"]
        b1 = model._layer_bufs[0]["b1"]
        f = torch.empty((T, FFN), device=dev, dtype=torch.bfloat16)
        for _ in range(3):
            ops.gemm_bf16(a, w, b1, epilogue="relu", out=f, cta_group=args.cta_group)
        torch.cuda.synchronize()
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 5
        k0.record()
        for _ in range(reps):
            ops.gemm_bf16(a, w, b1, epilogue="relu", out=f, cta_group=args.cta_group)
        k1.record()
        torch.cuda.synchronize()
        kms = k0.elapsed_time(k1) / reps
        flops = 2.0 * T * FFN * D  # algorithmic FLOPs of one launch
        alone_tflops = flops / (kms / 1e3) / 1e12
        achieved = flops / (in_step_kernel_ms / 1e3) / 1e12  # the launch inside the last timed step
        peak = float(peaks.get("bf16_tflops_sustained", FALLBACK_PEAKS["bf16_tflops_sustained"]))
        burst = float(peaks.get("bf16_tflops", FALLBACK_PEAKS["bf16_tflops"]))
        # DRAM bytes per launch of this kernel from an `ncu --set full` capture -- only quoted when the capture was taken
        # on the kernel source being benched (the capture file records kernel_source_digest()), else null
        traffic, traffic_note = None, None
        tp = os.path.join(ROOT, "profiles", "ncu_gemm_ffn1.json")
        if os.path.exists(tp) and (B, S) == (BATCH, SEQ):
            with open(tp) as fh:
                tj = json.load(fh)
            if tj.get("kernel_source_digest") and tj.get("kernel_source_digest") == kernel_source_digest():
                traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
                traffic_note = f"ncu capture {tj.get('capture')} of this kernel source (gemm_tcgen05.cu + common.cuh)"
            else:
                traffic_note = (f"null: the committed capture ({tj.get('capture')}) was taken on a different version of "
                                "gemm_tcgen05.cu")
        roofline = {"bound": "tensor", "kernel": "gemm_bf16_tcgen05_kernel<cta_group,EPI_BIAS_RELU,bf16> "
                    f"M={T} N={FFN} K={D}", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                    "frac": achieved / peak, "traffic": traffic, "traffic_note": traffic_note,
                    "ms_per_launch_in_step": in_step_kernel_ms,
                    "timed_alone": {"achieved": alone_tflops, "peak": burst, "frac": alone_tflops / burst,
                                    "peak_source": f"{peak_kind} bf16_tflops (burst)", "ms_per_launch": kms},
                    "algorithmic_bytes": 2.0 * T * D + 2.0 * FFN * D + 4.0 * FFN + 2.0 * T * FFN,
                    "peak_source": f"{peak_kind} bf16_tflops_sustained (kernel timed inside the long step)",
                    "whole_step_frac": (value / world) * flops_per_sentence(S) / 1e12 / peak}
        del a, f

    # ---- same-box A/B of the schedule variants: alternating 3-step blocks so clock drift hits all of them alike ----
    ab = None
    if variants and (B, S) == (BATCH, SEQ):
        def run_n(m, k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(k):
                m(batch_dev)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / k

        def vname(lf_, eg_):
            return {0: "ln_separate", 1: "ln_folded", 2: "ln1_folded"}[lf_] + f"/epi_groups{eg_}"

        allv = {(args.ln_fold, args.epi_groups): model, **variants}
        for m in variants.values():
            run_n(m, 1)
        times = {k: [] for k in allv}
        for _ in range(3):
            for k, m in allv.items():
                times[k].append(run_n(m, 3))
        ref_out = model(batch_dev).sentence_embeddings[:256].double()
        ab = {"ms_per_step": {vname(*k): v for k, v in times.items()},
              "sentences_per_s": {vname(*k): B / (sum(v) / len(v)) * 1e3 for k, v in times.items()},
              "default": vname(args.ln_fold, args.epi_groups), "rel_l2_vs_default_max": {}}
        for k, m in variants.items():
            got = m(batch_dev).sentence_embeddings[:256].double()
            ab["rel_l2_vs_default_max"][vname(*k)] = float(((got - ref_out).norm(dim=1) / ref_out.norm(dim=1)).max())
        variants.clear()
        allv.clear()
        torch.cuda.empty_cache()

    # ---- ragged variant (SURVEY §8(d)): lengths U{16..128}; the engine packs tokens, the reference would pad to 128 ----
    ragged = None
    if rank == 0 and world == 1 and (B, S) == (BATCH, SEQ):
        from sonar_b200 import PaddingMask

        gl = torch.Generator().manual_seed(7)
        lens = torch.randint(16, 129, (B,), generator=gl)
        lens_list = lens.tolist()
        rb = SequenceBatch(ids_dev, PaddingMask(lens, S, lens_list))
        for _ in range(2):
            model(rb)
        torch.cuda.synchronize()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        for _ in range(3):
            model(rb)
        r1.record()
        torch.cuda.synchronize()
        rms = r0.elapsed_time(r1) / 3
        rflops = sum(flops_per_sentence(n) for n in lens_list)
        peak_s = float(peaks.get("bf16_tflops_sustained", FALLBACK_PEAKS["bf16_tflops_sustained"]))
        ragged = {"lengths": "U{16..128}, seed 7", "tokens": int(lens.sum()), "padded_tokens": B * S,
                  "value": B / rms * 1e3, "unit": "sentences/s", "ms_per_step": rms,
                  "roofline_frac_of_real_flops": rflops / (rms / 1e3) / 1e12 / peak_s}

    cpu_baseline = None
    if sd_cpu is not None:
        calibrate_cpu_threads()
        v, n, dt, emb_cpu, ids_cpu = cpu_port_throughput(sd_cpu, args.cpu_seconds)
        got = model(SequenceBatch(ids_cpu.to(dev), None)).sentence_embeddings.cpu().double()
        ref = emb_cpu.double()
        cos = torch.nn.functional.cosine_similarity(got, ref, dim=1)
        rel = (got - ref).norm(dim=1) / ref.norm(dim=1)
        cpu_baseline = {"value": v, "unit": "sentences/s", "cores": torch.get_num_threads(), "kind": "port",
                        "sample": f"{n} sentences x {S} tokens x {LAYERS} layers in {dt:.1f}s, fp32 torch CPU "
                                  f"restatement of the fairseq2 op sequence (oracle/text_encoder.py), "
                                  f"host cpu_count={os.cpu_count()}",
                        "parity_vs_gpu": {"one_minus_cos_max": float((1 - cos).max()),
                                          "rel_l2_max": float(rel.max()), "sentences": int(len(cos))}}

    # ---- BASELINE config 5 end to end (N > 1), before the text model is released ----
    config5 = None
    if world > 1 and not args.skip_config5 and (B, S) == (BATCH, SEQ):
        try:
            config5 = bench_config5(model, dev, dist, rank, world, local, peaks, args.config5_per_gpu)
        except Exception as e:  # the headline line must survive a failure here
            config5 = {"error": f"{type(e).__name__}: {e}"}

    # ---- N = 1: the public predict() call and BASELINE configs 3 / 4 / 5 on this GPU ----
    extra = {}
    if rank == 0 and world == 1 and not args.skip_secondary and (B, S) == (BATCH, SEQ):
        only = [x for x in args.only.split(",") if x]
        plan = [("predict", lambda: bench_predict(model, dev, peaks))]
        plan += [(nme, (lambda f=f: f(dev, peaks))) for nme, f in (("speech", bench_speech), ("decoder", bench_decoder),
                                                                   ("xsim", bench_xsim))]
        for nme, fn in plan:
            if only and nme not in only:
                continue
            if nme == "speech":  # the text engine (weights + 14 GB workspace) is no longer needed
                model = None
                torch.cuda.empty_cache()
            t0 = time.perf_counter()
            try:
                extra[nme] = fn()
            except Exception as e:
                extra[nme] = {"error": f"{type(e).__name__}: {e}"}
            extra[nme]["block_wall_s"] = time.perf_counter() - t0
            torch.cuda.empty_cache()

    if rank == 0:
        launches_per_step = 1 + LAYERS * {0: 7, 1: 5, 2: 6}[args.ln_fold] + 1  # embed, per layer 4 GEMMs + attention (+ LNs), pool
        line = {
            "metric": "sentences/sec->1024-d", "value": value, "unit": "sentences/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": f"text_sonar_basic_encoder arch (24L, d=1024, 16 heads, FFN 8192, vocab {VOCAB}), "
                                   f"batch {B} x seq_len {S} per GPU, random-init weights, synthetic ids",
                       "l2": "inputs larger than L2 (per-step activations ~15 GB vs 126 MB L2)",
                       "parallelism": f"dp{world}" + (" + all_gather of embeddings" if world > 1 else ""),
                       "cta_group": args.cta_group,
                       "layernorm": {0: "separate kernels", 1: "folded into the QKV / FFN1 GEMMs (statistics from the residual "
                                     "GEMMs' epilogues)", 2: "attention-block LayerNorm folded (FFN2 -> QKV), FFN-block LayerNorm "
                                     "a kernel"}[args.ln_fold],
                       "epi_groups": args.epi_groups},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "sentences/s", "h2d_bytes_per_step": B * S * 8,
                    "d2h_bytes_per_step": B * D * 4, "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": launches_per_step * args.steps,
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "ragged": ragged,
            "ab_schedule_variants": ab,
            **extra,
        }
        if config5 is not None:
            line["config5"] = config5
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
