#!/usr/bin/env python
"""Headline benchmark: audio-seconds/sec (RTF^-1) of Fr-En simultaneous S2ST at chunk = 320 ms (BASELINE.json).

A "step" is one pass of the hot path over one synthetic 10 s / 16 kHz utterance, streamed in 320 ms chunks
(32 policy() calls: fbank -> chunk-Conformer encoder -> 2 CTC heads -> policy gate -> MT decoder -> T2U ->
NAR unit decoder -> CodeHiFiGAN vocoder), batch 1, exactly BASELINE.json configs[1].

  value : audio-seconds / second with the utterance already resident in HBM and results left on the device
  e2e   : the same through the reference-facing agent API (StreamSpeechS2STAgent.pushpop with python-list
          SpeechSegments): host->device copy of every new chunk and device->host read of every emitted waveform
  N > 1 : one process per GPU (torchrun), utterances sharded over ranks, no data-path collective; the synthetic
          checkpoint is NCCL-broadcast from rank 0 once before timing (weak scaling: every rank streams K utterances)

  --impl reference : the CPU restatement of the reference agent (oracle/, kind "port": the reference itself cannot be
          installed here, see DESIGN.md) with all host threads, same utterance, same metric.
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

UTT_SECONDS = 10.0
CHUNK_MS = 320
SAMPLE_RATE = 16000
METRIC = "audio-seconds/sec (RTF^-1) Fr-En simul S2ST @chunk=320ms"
WORKLOAD = "Fr-En simultaneous S2ST, chunk_size=320ms, batch=1, synthetic 10 s 16 kHz audio (BASELINE.json configs[1])"


def shard_utterances(n_utts: int, rank: int, world: int):
    """utterance ids of this rank: round-robin, no collective on the data path"""
    return [i for i in range(n_utts) if i % world == rank]


def agent_args(device_index=0, encoder_mode="cached"):
    return argparse.Namespace(model_path="synthetic", vocoder="synthetic", vocoder_cfg=None, data_bin=".", config_yaml=None,
                              multitask_config_yaml=None, sample_rate=SAMPLE_RATE, max_len=200, force_finish=False,
                              dur_prediction=True, lagging_k1=0, lagging_k2=0, segment_size=CHUNK_MS, stride_n=1, stride_n2=1,
                              unit_per_subword=15, source_segment_size=CHUNK_MS, vocoder_context="receptive-field",
                              device_index=device_index, encoder_mode=encoder_mode)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
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
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def host_threads() -> int:
    """threads for the CPU arm: the host cores this process may use (affinity mask when the platform has one), capped at 64 --
    the path is a chain of small fp32 ops (batch 1, <= 250 x 256 activations) that stops scaling long before that, and
    oversubscribing OpenMP on bigger hosts only slows it down"""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    return max(1, min(n, 64))


def note(msg: str):
    """progress marker on stderr (a run killed by a timeout shows where it was)"""
    print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def dump_outputs(out_dir, calls):
    """--dump-outputs: what the last timed step returned to its caller, one policy() call after the other, as float npy files:
    wav (every emitted waveform chunk, concatenated), write and samples_per_call (the action and chunk length of each call), and the
    latest asr_tokens / st_tokens / mt_tokens / units / dur of the step (the complete hypotheses of the utterance)."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    wavs = [wav.float().cpu().numpy() for w, wav, _ in calls if w and wav is not None]
    arrays = {"wav": np.concatenate(wavs) if wavs else np.zeros(0, dtype=np.float32),
              "write": np.array([float(w) for w, _, _ in calls]),
              "samples_per_call": np.array([float(wav.numel()) if w and wav is not None else 0.0 for w, wav, _ in calls])}
    for key in ("asr_tokens", "st_tokens", "mt_tokens", "units", "dur"):
        seen = [tr[key] for _, _, tr in calls if key in tr]
        arrays[key] = np.array(seen[-1] if seen else [], dtype=np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
    return sum(a.nbytes for a in arrays.values())


def run_reference(args):
    """CPU arm: the reference agent's semantics (full-prefix recompute every chunk) in PyTorch fp32 on the host cores."""
    import torch

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle.agent_oracle import OracleS2STAgent
    from oracle.streamspeech_oracle import StreamSpeechOracle
    from streamspeech_b200 import synth
    from streamspeech_b200.config import ModelConfig

    torch.set_grad_enabled(False)
    # torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm runs on rank 0 alone (the other ranks have exited), so it
    # takes every host core explicitly -- the thread count actually used is reported as `cores`
    torch.set_num_threads(host_threads())
    cores = torch.get_num_threads()
    cfg = ModelConfig()
    o = StreamSpeechOracle(cfg, synth.make_model_state_dict(cfg, 0), synth.make_vocoder_state_dict(cfg.vocoder, 1), synth.make_gcmvn(cfg))
    wav = synth.make_audio(UTT_SECONDS, seed=1234)
    n = SAMPLE_RATE * CHUNK_MS // 1000

    def one():
        ag = OracleS2STAgent(o, CHUNK_MS)
        out = 0
        for i in range(0, len(wav), n):
            ag.push(wav[i:i + n].tolist(), finished=i + n >= len(wav))
            a = ag.policy()
            out += len(a.wav) if a.wav else 0
        return out

    for _ in range(args.warmup):
        one()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        one()
    dt = time.perf_counter() - t0
    value = args.steps * UTT_SECONDS / dt
    sample = f"{args.steps} x one {UTT_SECONDS:.0f} s utterance streamed in {CHUNK_MS} ms chunks (full workload per step)"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "audio-s/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": {"workload": WORKLOAD},
            "cpu_baseline": {"value": value, "unit": "audio-s/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def encoder_roofline(engine, peaks, run_utterance):
    """Dominant kernel of the step = the encoder-stack kernel (one launch per 320 ms chunk runs all 12 Conformer layers over the
    <= 16 not-yet-final rows): encoder_layers_cluster_kernel (4 clusters x 16 CTAs, activations in distributed shared memory,
    weights streamed by TMA from repacked blobs) when the step has <= 16 rows, else encoder_layers_persistent_kernel (148 CTAs);
    16.4 % of the summed kernel time in profiles/r2_launches_bench_window_cluster.md, 17.7 % of the utterance's device time measured here.
    It streams every GEMM weight of the stack once per launch -> HBM roofline.  Measured live: the engine brackets each
    launch with CUDA events on the launching stream while one more resident utterance is streamed (32 launches).
    algorithmic bytes per launch = 12 x (4*D*FFN + 7*D*D) x 4 B of weights (122.7 MB) + the K / V cache and
    relative-position rows the attention reads (12 x (3T + nA) x D x 4 B)."""
    import torch

    engine.set_option("persistent_time", 1)
    engine.persistent_time()  # drop stale records
    engine.mt_time()
    c0 = engine.cluster_steps()
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    run_utterance()
    t1.record()
    torch.cuda.synchronize()
    utt_ms = t0.elapsed_time(t1)
    ms, n, nbytes = engine.persistent_time()
    mt_ms, mt_n, mt_steps = engine.mt_time()
    cl = engine.cluster_steps() - c0
    engine.set_option("persistent_time", 0)
    peak = peaks.get("hbm_gbs", 6650.0)
    traffic = None
    cluster = n > 0 and cl * 2 > n  # which kernel took most of the timed launches
    tp = os.path.join(ROOT, "profiles", "r2_cluster_kernel_traffic.json" if cluster else "r2_dominant_kernel_traffic.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get("dram_bytes_per_launch")
    if n == 0:
        return {"bound": "hbm", "achieved": None, "peak": peak, "unit": "GB/s", "frac": None, "traffic": traffic,
                "kernel": "encoder_layers_persistent_kernel", "note": "no persistent launches were recorded"}
    ach = nbytes / (ms * 1e-3) / 1e9
    if cluster:
        kernel = ("encoder_layers_cluster_kernel (fp32, all 12 Conformer layers of one streaming step; 4 clusters x 16 CTAs, DSMEM "
                  "activation exchange, TMA weight ring)")
        note_ = ("batch-1 streaming: 16 rows per launch; per layer 9 distributed-shared-memory exchanges (st.async + mbarrier) and 2 split "
                 "grid barriers; bound by ~25 dependent latencies per layer (mbarrier waits, shuffle trees, L2 round trips), not by bandwidth")
    else:
        kernel = "encoder_layers_persistent_kernel<2048> (fp32, all 12 Conformer layers of one streaming step, 148 CTAs cooperative)"
        note_ = ("batch-1 streaming: 16 rows per launch, 108 grid barriers; the kernel is bound by dependent-phase latency "
                 "(barrier + one L2/HBM round trip per phase), not by bandwidth")
    # second-largest kernel, measured the same way: the single-token MT kernel (one greedy step streams every decoder weight and the
    # tied output projection once)
    cfg = engine.cfg
    mt_bytes_step = (cfg.mt_layers * (6 * cfg.mt_dim * cfg.mt_dim + 2 * cfg.mt_dim * cfg.mt_ffn) + cfg.tgt_vocab * cfg.mt_dim) * 4.0
    mt = None
    if mt_n > 0 and mt_ms > 0:
        mt_ach = mt_bytes_step * mt_steps / (mt_ms * 1e-3) / 1e9
        mt = {"kernel": "mt_decode_persistent_kernel_v2 (fp32, one launch per burst of greedy steps)", "bound": "hbm", "achieved": mt_ach,
              "peak": peak, "unit": "GB/s", "frac": mt_ach / peak, "algorithmic_bytes_per_step": mt_bytes_step, "steps_timed": mt_steps,
              "launches_timed": mt_n, "us_per_step": mt_ms / max(mt_steps, 1.0) * 1e3, "share_of_utterance_time": mt_ms / utt_ms}
    return {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
            "kernel": kernel, "cluster_kernel_launches": cl, "share_of_utterance_time": ms / utt_ms, "second_kernel": mt,
            "algorithmic_bytes_per_launch": nbytes / n, "launches_timed": n, "us_per_launch": ms / n * 1e3,
            "peak_source": "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6.65 TB/s",
            "note": note_}


def gemm_rooflines(engine, peaks):
    """Secondary: the GEMM / conv kernels at the vocoder's heaviest conv shape (L = 5*500 rows, 256 -> 256 channels, k = 11):
    fp32 CUDA cores and the tap-shift tcgen05 kernel with pre-packed weights.
    FLOPs are fp32-equivalent (2*L*C*C*k); the tcgen05 kernels spend 3 bf16 MMAs per product (bf16x3 split)."""
    import torch

    L, C, k = 5 * 500, 256, 11
    x = torch.randn(L, C, device=engine.device)
    w = torch.randn(C, C * k, device=engine.device) / (C * k) ** 0.5
    b = torch.zeros(C, device=engine.device)
    out = {}
    for name, mode, mmas in (("gemm_kernel<128,64> fp32 CUDA cores", 0, 0),
                             ("umma2_kernel tcgen05 bf16x3, tap-shift + cp.async.bulk weights (default path)", 12, 3)):
        fn = lambda: engine.op_conv1d(x, w, b, k, 1, k // 2, 0.1, mode)
        for _ in range(3):
            fn()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        s.record()
        for _ in range(20):
            fn()
        e.record()
        torch.cuda.synchronize()
        ms = s.elapsed_time(e) / 20
        ach = 2.0 * L * C * C * k / (ms * 1e-3) / 1e12
        peak = peaks.get("bf16_tflops", 1590.0)
        out[name] = {"bound": "tensor", "achieved_fp32_equivalent": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                     "us_per_launch": ms * 1e3, "shape": {"L": L, "C_in": C, "C_out": C, "k": k}}
        if mmas:  # every fp32-grade product is `mmas` bf16 MMAs: the tensor pipe itself runs at mmas x the fp32-equivalent rate
            out[name]["bf16_mmas_per_product"] = mmas
            out[name]["tensor_pipe_frac"] = mmas * ach / peak
    return out


def asr_streams_leg(eng, n_streams=32, seconds=10.0, chunk_ms=160, rank=0):
    """BASELINE configs[3]: streaming ASR at chunk = 160 ms, 256 concurrent utterances sharded over 8 GPUs = 32 streams per GPU.
    All streams of a GPU advance together through the stream pool (ss_pool_step: batched fbank -> encoder -> ASR CTC head); the timed
    region includes the host->device copy of every chunk and the device->host read of every stream's tokens (e2e style)."""
    import torch

    from streamspeech_b200 import synth
    from streamspeech_b200.scheduler import StreamPool

    eng.set_chunk(chunk_ms // 40, min(chunk_ms // 40, 16))  # speech_to_text.asr agent :361-375
    pool = StreamPool(eng, n_slots=n_streams, max_seconds=int(seconds) + 1, ctc_heads=1)
    n = SAMPLE_RATE * chunk_ms // 1000
    wavs = [synth.make_audio(seconds, seed=5000 + 97 * rank + j).contiguous() for j in range(n_streams)]
    slots = [pool.acquire() for _ in range(n_streams)]

    def run():
        for sl in slots:
            pool.reset(sl)
        ntok = 0
        for i in range(0, wavs[0].numel(), n):
            for j, sl in enumerate(slots):
                pool.push(sl, wavs[j][i:i + n])
            pool.flush()
            ntok = sum(len(pool.results[sl]["ctc"][0][0]) for sl in slots)
        return ntok

    run()  # warm-up (workspace growth, packed weight caches)
    torch.cuda.synchronize()
    l0 = eng.launch_count()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    ntok = run()
    e.record()
    torch.cuda.synchronize()
    ms = s.elapsed_time(e)
    eng.set_chunk(CHUNK_MS // 40)  # back to the S2ST setting
    return {"workload": f"streaming ASR, chunk {chunk_ms} ms, {n_streams} concurrent {seconds:.0f} s utterances per GPU (BASELINE.json configs[3])",
            "value": n_streams * seconds / (ms * 1e-3), "unit": "audio-s/s", "ms": ms, "streams": n_streams, "steps": pool.steps // 2,
            "rows_per_step": n_streams * 2 * (chunk_ms // 40), "gpu_launches": eng.launch_count() - l0, "tokens_final": ntok,
            "h2d_bytes": int(n_streams * seconds * SAMPLE_RATE * 4)}


def offline_leg(agent, peaks, B=32, seconds=15.0):
    """BASELINE configs[2]: offline S2ST, batch of 32 padded 15 s utterances on one GPU: batched encoder over B x T = 12,000 rows
    (tcgen05 GEMMs), CTC prints, greedy MT, T2U + unit decoder and the vocoder per utterance (the reference's vocoder script is
    batch 1 too: generate_waveform_from_code.py:40-78).  Also times the two kernels the config is quoted for: the FFN GEMM at
    M = 12,000 and the vocoder generator on 750 frames."""
    import torch

    from streamspeech_b200 import synth
    from streamspeech_b200.offline import OfflineS2STGenerator

    eng = agent.engine
    gen = OfflineS2STGenerator(eng, max_len_b_mt=100)
    feats = []
    for b in range(B):
        w = synth.make_audio(seconds, seed=7000 + b).cuda()
        feats.append(eng.fbank(w))
    F = max(f.shape[0] for f in feats)
    src = torch.zeros(B, F, eng.cfg.feat_dim, device="cuda")
    for b, f in enumerate(feats):
        src[b, : f.shape[0]] = f
    lens = [f.shape[0] for f in feats]

    def timed(fn, reps=1):
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(reps):
            r = fn()
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e) / reps, r

    eng.encoder(src, lens)  # warm-up
    ms_enc, _ = timed(lambda: eng.encoder(src, lens), 3)
    ms_gen, res = timed(lambda: gen.generate(src, lens))
    codes = [gen.units_to_codes(r["units"]) for r in res]
    ms_voc, wavs = timed(lambda: [gen.synthesize(c) for c in codes if len(c)])
    out_s = sum(w.numel() for w in wavs) / SAMPLE_RATE
    T = eng.encoder_out_frames(F)
    rows = B * T
    enc_flops = 2.0 * rows * (37_606_400 - 3_072_000 + 12_288 * T)  # SURVEY.md §8(d): MAC per encoder frame without the CTC heads
    line = {"workload": f"offline S2ST, batch {B} x {seconds:.0f} s padded (BASELINE.json configs[2])", "unit": "audio-s/s",
            "value": B * seconds / ((ms_gen + ms_voc) * 1e-3), "ms_encoder_batched": ms_enc, "ms_generate": ms_gen, "ms_vocoder": ms_voc,
            "encoder_rows": rows, "encoder_tflops_fp32_equivalent": enc_flops / (ms_enc * 1e-3) / 1e12, "output_audio_s": out_s}
    # the FFN GEMMs of the batched encoder on the tcgen05 kernel (bf16 x 6 split = fp32-grade), M = B x T rows
    peak = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0))
    g = {}
    x = torch.randn(rows, 256, device="cuda")
    hbuf = torch.randn(rows, 2048, device="cuda")
    w1 = torch.randn(2048, 256, device="cuda") / 16
    w2 = torch.randn(256, 2048, device="cuda") / 45
    b1, b2 = torch.zeros(2048, device="cuda"), torch.zeros(256, device="cuda")
    for name, a, w, b, K, N in (("ffn_w1 M x 256 -> 2048", x, w1, b1, 256, 2048), ("ffn_w2 M x 2048 -> 256", hbuf, w2, b2, 2048, 256)):
        for pieces in (2, 3):
            eng.op_linear_umma(a, w, b, 0, pieces)
            ms, _ = timed(lambda: eng.op_linear_umma(a, w, b, 0, pieces), 10)
            fl = 2.0 * rows * K * N
            mm = 3 if pieces == 2 else 6
            g[f"{name}, bf16x{mm}"] = {"us": ms * 1e3, "tflops_fp32_equivalent": fl / (ms * 1e-3) / 1e12,
                                      "tensor_pipe_frac": mm * fl / (ms * 1e-3) / 1e12 / peak}
    line["ffn_gemm_umma2"] = {"M": rows, "peak_tflops": peak, "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained", "kernels": g}
    # vocoder generator on 750 frames (15 s of output audio)
    codes750 = torch.randint(0, 1000, (750,), device="cuda")
    eng.vocoder_durations(codes750, False)
    eng.vocoder_generate(750, 0, 750, 0)
    ms750, _ = timed(lambda: eng.vocoder_generate(750, 0, 750, 0), 5)
    fl = 750 * 320.8e6  # SURVEY.md §8(d): 320.8 MFLOP per unit frame
    line["vocoder_750_frames"] = {"ms": ms750, "tflops_fp32_equivalent": fl / (ms750 * 1e-3) / 1e12, "tensor_pipe_frac": 3 * fl / (ms750 * 1e-3) / 1e12 / peak,
                                  "audio_s_per_s": 15.0 / (ms750 * 1e-3)}
    eng.set_chunk(CHUNK_MS // 40)
    return line


def mixed_pairs_leg(device_index=0, chunk_ms=640, seconds=10.0, lags=(0, 1, 2, 4)):
    """BASELINE configs[4]: Es-En + De-En simultaneous S2ST in one process at chunk = 640 ms (whole-word policy), latency sweep over
    lagging_k1.  Two language pairs = two weight sets = two engine handles on the same GPU (same shapes, different seeds stand in for
    the two checkpoints); utterances of the two pairs alternate.  Handles share no device state, so this is the single-stream path twice."""
    import torch

    from streamspeech_b200 import synth
    from streamspeech_b200.agent import StreamSpeechS2STAgent

    agents = {}
    for pair, seed in (("es-en", 0), ("de-en", 0)):  # the calibrated synthetic checkpoint, loaded twice: two independent device copies
        a = agent_args(device_index)
        a.model_path, a.vocoder = f"synthetic:{seed}", "synthetic:1"
        a.source_segment_size = chunk_ms
        agents[pair] = StreamSpeechS2STAgent(a)
    n = SAMPLE_RATE * chunk_ms // 1000
    utts = {pair: synth.make_audio(seconds, seed=900 + i).cuda() for i, pair in enumerate(agents)}
    out = {}
    for lag in lags:
        for ag in agents.values():
            ag.lagging_k1 = lag

        def run():
            total = 0
            for pair, ag in agents.items():  # the two pairs alternate utterance by utterance
                u = utts[pair]
                ag.reset()
                for i in range(0, u.numel(), n):
                    end = min(i + n, u.numel())
                    w, wav = ag.step_resident(u, end, end >= u.numel())
                    if w and wav is not None:
                        total += wav.numel()
            return total

        run()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        samples = run()
        e.record()
        torch.cuda.synchronize()
        out[f"lagging_k1={lag}"] = {"audio_s_per_s": 2 * seconds / (s.elapsed_time(e) * 1e-3), "ms": s.elapsed_time(e), "output_audio_s": samples / SAMPLE_RATE}
    for ag in agents.values():
        ag.engine.close()
    return {"workload": f"Es-En + De-En simultaneous S2ST, chunk {chunk_ms} ms, two weight sets on one GPU, alternating {seconds:.0f} s utterances, "
                        "latency sweep over lagging_k1 (BASELINE.json configs[4])", "unit": "audio-s/s", "sweep": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--encoder-mode", type=str, default="cached", choices=["cached", "recompute"])
    ap.add_argument("--no-extras", action="store_true", help="skip the configs[2] / configs[3] legs (extra keys of the JSON line)")
    ap.add_argument("--ncu-window", action="store_true",
                    help="after the timed runs, stream one more resident utterance between cudaProfilerStart/Stop (for `ncu --profile-from-start off`)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (waveform, actions, tokens) as DIR/<name>.npy, to compare two builds")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import torch

    from streamspeech_b200 import synth
    from streamspeech_b200.agent import StreamSpeechS2STAgent
    from streamspeech_b200.simuleval_compat import SpeechSegment

    torch.set_grad_enabled(False)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    a_args = agent_args(local, args.encoder_mode)
    if world > 1:
        # The one collective of the path: the initial weight broadcast over NVLink (SURVEY.md §8e).  Rank 0 owns the
        # checkpoint (model + vocoder, packed into one fp32 blob); the other ranks allocate the blob, receive it with NCCL and
        # build their engine FROM THE RECEIVED BYTES (their own tensors are zero-filled before the broadcast).
        from streamspeech_b200.config import ModelConfig

        cfg0 = ModelConfig()
        if rank == 0:
            sd = synth.make_model_state_dict(cfg0, 0)
            vsd = synth.make_vocoder_state_dict(cfg0.vocoder, 1)
            meta = [[(k, tuple(v.shape)) for k, v in d.items() if v.is_floating_point()] for d in (sd, vsd)]
        else:
            sd, vsd, meta = None, None, None
        box = [meta]
        dist.broadcast_object_list(box, src=0)
        meta = box[0]
        total = sum(int(torch.Size(shp).numel()) for part in meta for _, shp in part)
        flat = torch.zeros(total, dtype=torch.float32, device="cuda")
        if rank == 0:
            flat.copy_(torch.cat([d[k].float().flatten() for d, part in ((sd, meta[0]), (vsd, meta[1])) for k, _ in part]))
        dist.broadcast(flat, src=0)
        torch.cuda.synchronize()
        host = flat.cpu()
        parts, off = [], 0
        for part in meta:
            d = {}
            for k, shp in part:
                nel = int(torch.Size(shp).numel())
                d[k] = host[off:off + nel].view(shp).clone()
                off += nel
            parts.append(d)
        a_args.checkpoint_override = (cfg0, parts[0], parts[1], synth.make_gcmvn(cfg0))
        del flat, host
    agent = StreamSpeechS2STAgent(a_args)
    eng = agent.engine

    n = SAMPLE_RATE * CHUNK_MS // 1000
    utts = [synth.make_audio(UTT_SECONDS, seed=1234 + 7 * rank + i) for i in range(2)]  # rank-specific utterances
    utts_dev = [u.cuda() for u in utts]
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")  # > 126 MB L2

    def stream_resident(u, calls=None):
        agent.reset()
        out = 0
        for i in range(0, u.numel(), n):
            end = min(i + n, u.numel())
            w, wav = agent.step_resident(u, end, end >= u.numel())
            if w and wav is not None:
                out += wav.numel()
            if calls is not None:  # every call returns a fresh wav tensor and trace dict: keeping them costs no device work
                calls.append((w, wav, agent.trace))
        return out

    def stream_e2e(u_host):
        agent.reset()
        out = 0
        for i in range(0, len(u_host), n):
            seg = agent.pushpop(SpeechSegment(content=u_host[i:i + n], sample_rate=SAMPLE_RATE, finished=i + n >= len(u_host)))
            if not seg.is_empty:
                out += len(seg.content)
        return out

    def timed(fn, inputs, steps, warmup, last_calls=None):
        for i in range(warmup):
            fn(inputs[i % len(inputs)])
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        total_ms, out = 0.0, 0
        l0 = eng.launch_count()
        for i in range(steps):
            record = (last_calls,) if last_calls is not None and i == steps - 1 else ()
            flush.fill_(float(i))  # L2 flush between timed iterations (outside the events)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            out += fn(inputs[i % len(inputs)], *record)
            e.record()
            torch.cuda.synchronize()
            total_ms += s.elapsed_time(e)
        launches = eng.launch_count() - l0
        t = torch.tensor([total_ms], device="cuda")
        if dist is not None:
            dist.barrier()
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), out, launches

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    note("timed: resident")
    last_calls = [] if args.dump_outputs and rank == 0 else None
    ms_res, out_res, launches = timed(stream_resident, utts_dev, args.steps, args.warmup, last_calls)
    if last_calls is not None:
        nbytes = dump_outputs(args.dump_outputs, last_calls)
        note(f"outputs of the last timed step: {len(last_calls)} calls, {nbytes} bytes -> {args.dump_outputs}")
        del last_calls
    note("timed: e2e")
    utts_host = [u.tolist() for u in utts]
    ms_e2e, out_e2e, _ = timed(stream_e2e, utts_host, args.steps, max(1, args.warmup // 2))
    extra_asr = None
    if not args.no_extras:
        note("extra: ASR streams leg")
        try:
            extra_asr = asr_streams_leg(eng, rank=rank)
            t = torch.tensor([extra_asr["ms"]], device="cuda")
            if dist is not None:
                dist.barrier()
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            extra_asr["ms"] = float(t.item())
            extra_asr["value"] = extra_asr["streams"] * world * UTT_SECONDS / (extra_asr["ms"] * 1e-3)
            extra_asr["streams_total"] = extra_asr["streams"] * world
        except Exception as ex:  # noqa: BLE001 -- an extra leg must never take the headline down
            extra_asr = {"error": repr(ex)}
            if dist is not None:
                t = torch.tensor([0.0], device="cuda")
                dist.barrier()
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
    clocks = sampler.stop() if rank == 0 else None
    if args.ncu_window and rank == 0:
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        stream_resident(utts_dev[0])
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    peaks = {}
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        peaks = json.load(open(pk))
    audio_s = args.steps * UTT_SECONDS * world
    value = audio_s / (ms_res * 1e-3)
    e2e = audio_s / (ms_e2e * 1e-3)
    line = {"metric": METRIC, "value": value, "unit": "audio-s/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic 16 kHz audio + seeded random-init weights of the StreamSpeech architecture (calibrated token rates, see DESIGN.md)",
            "config": {"workload": WORKLOAD, "utterance_s": UTT_SECONDS, "chunk_ms": CHUNK_MS, "policy_calls_per_step": int(UTT_SECONDS * 1000 // CHUNK_MS) + 1,
                       "l2": "256 MiB flush between timed steps", "encoder_mode": args.encoder_mode, "parallelism": f"utterance-sharded x{world}",
                       "output_audio_s_per_step": out_res / args.steps / SAMPLE_RATE},
            "e2e": {"value": e2e, "unit": "audio-s/s", "h2d_bytes_per_step": int(UTT_SECONDS * SAMPLE_RATE * 4),
                    "d2h_bytes_per_step": int(out_e2e / args.steps * 4), "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches), "clocks": clocks,
            "engine_options": {k: os.environ.get(k) for k in sorted(os.environ) if k.startswith("SS_")}}
    def one_more():
        flush.fill_(0.0)
        stream_resident(utts_dev[0])

    note("roofline legs")
    line["roofline"] = encoder_roofline(eng, peaks, one_more)
    line["roofline_large_gemm"] = gemm_rooflines(eng, peaks)
    if extra_asr is not None:
        line["extra_asr_streams"] = extra_asr
    if world == 1 and not args.no_extras:
        note("extra: offline batch leg")
        try:
            line["extra_offline_batch32"] = offline_leg(agent, peaks)
        except Exception as ex:  # noqa: BLE001
            line["extra_offline_batch32"] = {"error": repr(ex)}
        note("extra: mixed language pairs leg")
        try:
            line["extra_mixed_pairs_640ms"] = mixed_pairs_leg(local)
        except Exception as ex:  # noqa: BLE001
            line["extra_mixed_pairs_640ms"] = {"error": repr(ex)}
    if world == 1 and not args.no_cpu_baseline:
        # bounded CPU sample: the first 4 s of the same utterance through the oracle agent (reference semantics)
        from oracle.agent_oracle import OracleS2STAgent
        from oracle.streamspeech_oracle import StreamSpeechOracle
        from streamspeech_b200.config import ModelConfig

        cfg = ModelConfig()
        o = StreamSpeechOracle(cfg, synth.make_model_state_dict(cfg, 0), synth.make_vocoder_state_dict(cfg.vocoder, 1), synth.make_gcmvn(cfg))
        ag = OracleS2STAgent(o, CHUNK_MS)
        torch.set_num_threads(host_threads())
        note(f"cpu_baseline: oracle agent, {torch.get_num_threads()} threads")
        # bounded sample: the workload utterance chunk by chunk, stopped after ~25 s of CPU time (the reference recomputes the
        # whole prefix every chunk, so a truncated utterance flatters the CPU: later chunks cost more than earlier ones)
        w = utts[0]
        t0 = time.perf_counter()
        done = 0
        for i in range(0, len(w), n):
            ag.push(w[i:i + n].tolist(), finished=i + n >= len(w))
            ag.policy()
            done = min(i + n, len(w))
            if time.perf_counter() - t0 > 25.0:
                break
        dt = time.perf_counter() - t0
        secs = done / SAMPLE_RATE
        line["cpu_baseline"] = {"value": secs / dt, "unit": "audio-s/s", "cores": torch.get_num_threads(), "kind": "port",
                                "sample": f"the first {secs:.2f} s of the workload utterance (25 s CPU-time bound), {CHUNK_MS} ms chunks, oracle agent (reference semantics: full-prefix recompute), {torch.get_num_threads()} threads"}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
