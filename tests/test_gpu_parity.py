"""GPU parity tests: the CUDA path (through the C-ABI) against the golden fixtures dumped from the real
reference modules and against the CPU oracle on the same seeded inputs.

Tolerances (BASELINE.json north_star): integer outputs (CTC / MT / unit tokens, durations) bit-exact;
floating-point intermediates 2e-4 max-abs (fp32 kernels, different summation order than ATen);
vocoder waveform 1e-3 max-abs.
"""
import argparse
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from streamspeech_b200 import synth  # noqa: E402
from streamspeech_b200.config import ModelConfig, VocoderConfig  # noqa: E402

torch.set_grad_enabled(False)
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
FP_TOL = 2e-4
WAV_TOL = 1e-3


def report(name, **kw):
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, "parity_report.jsonl"), "a") as f:
        f.write(json.dumps({"test": name, **{k: (float(v) if isinstance(v, (float, np.floating)) else v) for k, v in kw.items()}}) + "\n")


def maxdiff(a, b):
    a = a.detach().float().cpu() if torch.is_tensor(a) else torch.as_tensor(a)
    b = b.detach().float().cpu() if torch.is_tensor(b) else torch.as_tensor(b)
    assert a.shape == b.shape, (a.shape, b.shape)
    return float((a - b).abs().max())


def golden_cfg():
    cfg = ModelConfig()
    cfg.enc_layers = 3
    return cfg


@pytest.fixture(scope="module")
def eng3():
    from streamspeech_b200.engine import Engine

    cfg = golden_cfg()
    e = Engine(cfg, synth.make_model_state_dict(cfg, 0), synth.make_vocoder_state_dict(cfg.vocoder, 1, weight_norm=True), None)
    yield e
    e.close()


@pytest.fixture(scope="module")
def full():
    """12-layer engine + oracle on the same synthetic checkpoint."""
    from oracle.streamspeech_oracle import StreamSpeechOracle
    from streamspeech_b200.engine import Engine

    cfg = ModelConfig()
    sd = synth.make_model_state_dict(cfg, 0)
    vsd = synth.make_vocoder_state_dict(cfg.vocoder, 1)
    gc = synth.make_gcmvn(cfg)
    e = Engine(cfg, sd, vsd, gc)
    o = StreamSpeechOracle(cfg, sd, vsd, gc, chunk_size=8)
    yield cfg, e, o
    e.close()


def cuda(x):
    return torch.as_tensor(x).cuda().contiguous()


# --------------------------------------------------------------------------------------------- single ops
def test_linear_and_layernorm_ops(eng3):
    g = torch.Generator().manual_seed(0)
    worst = 0.0
    for (M, K, N, act) in [(1, 256, 2048, 2), (7, 2048, 256, 0), (250, 256, 768, 0), (33, 512, 6000, 0), (1000, 128, 1, 0), (129, 512, 1005, 1)]:
        x = torch.randn(M, K, generator=g)
        w = torch.randn(N, K, generator=g) / K ** 0.5
        b = torch.randn(N, generator=g)
        ref = torch.nn.functional.linear(x, w, b)
        ref = {0: ref, 1: torch.relu(ref), 2: torch.nn.functional.silu(ref)}[act]
        got = eng3.op_linear(cuda(x), cuda(w), cuda(b), act)
        d = maxdiff(got, ref)
        worst = max(worst, d)
        assert d < 1e-4, (M, K, N, act, d)
    for C in (128, 256, 512):
        x = torch.randn(37, C, generator=g) * 3 + 1
        gam, bet = torch.randn(C, generator=g), torch.randn(C, generator=g)
        ref = torch.nn.functional.layer_norm(x, (C,), gam, bet, 1e-5)
        d = maxdiff(eng3.op_layer_norm(cuda(x), cuda(gam), cuda(bet)), ref)
        worst = max(worst, d)
        assert d < 2e-5, (C, d)
    report("ops", worst=worst)


# --------------------------------------------------------------------------------------------- fbank
def test_fbank_matches_torchaudio_fixture(eng3, gold):
    g = gold["fbank"]
    wav = cuda(g["wav"])
    got = eng3.fbank(wav)  # engine built without gcmvn -> raw log-mel
    assert got.shape == g["fbank"].shape
    d = maxdiff(got, g["fbank"])
    report("fbank", maxdiff=d)
    assert d < 2e-3, d  # log-mel of a 2^15-scaled signal (values ~10-20); fp32 FFT ordering differs from pocketfft
    # frame caching: any sub-range equals the same rows
    part = eng3.fbank(wav, 10, 25)
    assert torch.equal(part, got[10:35])
    # ragged / empty inputs
    assert eng3.fbank(wav[:239]).shape[0] == 0 and eng3.fbank(wav[:400]).shape[0] == 1


def test_fbank_cmvn_vs_oracle(full):
    from oracle.streamspeech_oracle import online_features

    cfg, e, o = full
    wav = synth.make_audio(3.1, seed=5)
    ref = online_features(wav, o.gcmvn)
    got = e.fbank(cuda(wav))
    d = maxdiff(got, ref)
    report("fbank_cmvn", maxdiff=d)
    assert d < 2e-3, d


# --------------------------------------------------------------------------------------------- encoder
@pytest.mark.parametrize("chunk,conv", [(4, 8), (8, 8), (16, 16), (None, None)])
def test_encoder_golden(eng3, gold, chunk, conv):
    g = gold["encoder"]
    eng3.set_chunk(chunk, conv)
    feats = cuda(g["feats"]).unsqueeze(0)
    out = eng3.encoder(feats)[0]
    d = maxdiff(out, g[f"out_c{chunk}"])
    report(f"encoder_c{chunk}", maxdiff=d)
    assert d < FP_TOL, d


def test_encoder_batched_padded(eng3, gold):
    g = gold["encoder"]
    eng3.set_chunk(8, 8)
    feats = torch.zeros(2, g["feats"].shape[0], 80)
    feats[0] = torch.from_numpy(g["feats"])
    feats[1, :150] = torch.from_numpy(g["feats"][:150])
    out = eng3.encoder(cuda(feats), lengths=g["batched_lens"].tolist())
    ref = torch.from_numpy(g["batched_out"]).transpose(0, 1)  # T x B x C -> B x T x C
    d = maxdiff(out, ref)
    report("encoder_batched", maxdiff=d)
    assert d < FP_TOL, d


def test_encoder_streaming_prefix_invariance(full):
    """Size-independent property (SURVEY §7.2): every frame of a *completed* chunk is final, i.e. the encoder output
    on a longer prefix agrees with the shorter prefix on all chunks but the last one."""
    cfg, e, o = full
    e.set_chunk(8, 8)
    feats = e.fbank(cuda(synth.make_audio(10.0, seed=21)))
    F = feats.shape[0]
    a = e.encoder(feats[: F - 64].unsqueeze(0).contiguous())[0]
    b = e.encoder(feats.unsqueeze(0).contiguous())[0]
    Ta = a.shape[0]
    stable = (Ta // 8 - 1) * 8
    d = maxdiff(a[:stable], b[:stable])
    report("encoder_prefix_invariance", maxdiff=d, frames=stable)
    assert d < 1e-4, d


@pytest.mark.parametrize("seg_ms,attn,conv", [(160, 4, 8), (320, 8, 8), (640, 16, 16), (160, 4, 4), (480, 12, 8), (960, 24, 16), (1600, 40, 16)])
def test_encoder_streaming_cache_equals_recompute(full, seg_ms, attn, conv):
    """ss_encoder_stream_step (K/V + conv-input caches, only the open chunk group recomputed) must reproduce the
    full-prefix recompute that the reference performs on every policy() call, at every call.  (12, 8), (24, 16), (40, 16):
    chunk sizes that do not nest (--source-segment-size 480 / 960 / 1600): rows are final only at common multiples of the
    attention chunk and the conv chunk."""
    cfg, e, o = full
    e.set_chunk(attn, conv)
    feats = e.fbank(cuda(synth.make_audio(5.0, seed=31)))
    buf = torch.zeros(1024, cfg.enc_dim, device="cuda")
    e.encoder_stream_reset()
    step = seg_ms // 10
    worst, calls = 0.0, 0
    ends = list(range(step - 2, feats.shape[0], step)) + [feats.shape[0]]  # fbank lags the audio by 1.5 frames
    for F in ends:
        T, Tf = e.encoder_stream_step(feats[:F].contiguous(), buf)
        ref = e.encoder(feats[:F].unsqueeze(0).contiguous())[0]
        assert T == ref.shape[0] and Tf <= T
        worst = max(worst, maxdiff(buf[:T], ref))
        calls += 1
    report(f"encoder_stream_cache_c{attn}_cc{conv}", maxdiff=worst, calls=calls)
    assert worst < 2e-5, worst
    e.set_chunk(8, 8)


def test_encoder_full_size_vs_oracle(full):
    cfg, e, o = full
    from oracle.streamspeech_oracle import online_features

    o.set_chunk(8)
    e.set_chunk(8)
    wav = synth.make_audio(10.0, seed=1234)
    ref_f = online_features(wav, o.gcmvn)
    ref = o.encoder(ref_f.unsqueeze(0), torch.tensor([ref_f.size(0)]))["encoder_out"][0][:, 0]
    got = e.encoder(cuda(ref_f).unsqueeze(0))[0]
    d = maxdiff(got, ref)
    report("encoder_12L_10s", maxdiff=d)
    assert d < 5e-4, d
    for head, name in ((0, "source_unigram"), (1, "ctc_target_unigram")):
        r = e.ctc_greedy(head, got)
        h = o.ctc_greedy(name, ref.unsqueeze(1))[0]
        n = int(r["count"].item())
        assert r["argmax"].tolist() == h["org_tokens"], name
        assert r["tokens"][:n].tolist() == h["tokens"] and r["index"][:n].tolist() == h["index"], name


# --------------------------------------------------------------------------------------------- decoders
def test_ctc_heads_golden(eng3, gold):
    g = gold["decoders"]
    enc = cuda(g["enc_out"])
    for head, name in ((0, "source_unigram"), (1, "ctc_target_unigram")):
        r = eng3.ctc_greedy(head, enc)
        n = int(r["count"].item())
        assert r["argmax"].cpu().numpy().tolist() == g[f"ctc_{name}_argmax"].tolist()
        assert r["tokens"][:n].tolist() == g[f"ctc_{name}_tokens"].tolist()
        assert r["index"][:n].tolist() == g[f"ctc_{name}_index"].tolist()


def test_mt_decoder_golden(eng3, gold):
    g = gold["decoders"]
    enc = cuda(g["enc_out"])
    feats, logits = eng3.mt_features(enc, g["mt_tokens"][0].tolist(), want_logits=True)
    d1, d2 = maxdiff(feats, g["mt_feats"]), maxdiff(logits, g["mt_logits_last"])
    fp = eng3.mt_features(enc, g["mt_tokens_pad"][0].tolist())
    d3 = maxdiff(fp, g["mt_feats_pad"])
    report("mt_decoder", feats=d1, logits=d2, feats_pad=d3)
    assert d1 < FP_TOL and d2 < FP_TOL and d3 < FP_TOL, (d1, d2, d3)


def test_t2u_unit_decoder_golden(eng3, gold):
    g = gold["decoders"]
    r = eng3.t2u_unit_decode(cuda(g["mt_feats"]), debug=True)
    d1 = maxdiff(r["t2u_out"], g["t2u_out"])
    d2 = maxdiff(r["logits"][:4], g["unit_logits_first"])
    report("t2u_unit", t2u=d1, logits=d2)
    assert d1 < FP_TOL and d2 < 5e-4, (d1, d2)
    assert r["argmax"].tolist() == g["unit_argmax"].tolist()
    n = int(r["count"].item())
    assert r["units"][:n].tolist() == g["unit_tokens"].tolist()
    rp = eng3.t2u_unit_decode(cuda(g["mt_feats_pad"]), n_pad_tail=1)
    assert rp["argmax"].tolist() == g["unit_argmax_pad"].tolist()


def test_mt_greedy_vs_oracle(full):
    cfg, e, o = full
    from oracle.streamspeech_oracle import online_features

    o.set_chunk(8)
    e.set_chunk(8)
    f = online_features(synth.make_audio(4.0, seed=9), o.gcmvn)
    eo = o.encoder(f.unsqueeze(0), torch.tensor([f.size(0)]))["encoder_out"][0]
    enc = cuda(eo[:, 0])
    for prefix, new in ((None, 3), ([17, 256, 4099], 2), ([17, 256, 4099], 0), (None, -1)):
        ref = o.mt_greedy(eo, prefix, new)
        toks, feats = e.mt_greedy(enc, prefix, new)
        assert toks == ref[:-1], (prefix, new, toks, ref)
        rf = o.mt_features(torch.tensor([[cfg.eos] + toks]), eo)[0]
        d = maxdiff(feats, rf)
        assert d < FP_TOL, d


# --------------------------------------------------------------------------------------------- vocoder
def test_vocoder_golden(eng3, gold):
    g = gold["vocoder"]
    codes = cuda(g["code"][0].astype(np.int64))
    dur, cum = eng3.vocoder_durations(codes, True)
    assert dur.tolist() == g["dur"][0].tolist()
    total = int(cum[-1].item())
    wav = eng3.vocoder_generate(total, 0, total, 0)
    d = maxdiff(wav, g["wav"])
    report("vocoder", maxdiff=d, samples=wav.numel())
    assert wav.numel() == g["wav"].shape[0] and d < WAV_TOL, d
    # tail generation with the receptive field as left context == the same samples of the full pass
    tail = 17
    part = eng3.vocoder_generate(total, total - tail, tail, -1)
    d2 = maxdiff(part, wav[-tail * eng3.hop:])
    report("vocoder_incremental", maxdiff=d2, receptive_field=eng3.vocoder_receptive_field)
    assert d2 < 1e-5, d2
    # no duration prediction: one frame per code
    dur1, cum1 = eng3.vocoder_durations(codes, False)
    assert dur1.tolist() == [1] * codes.numel() and int(cum1[-1].item()) == codes.numel()


def test_vocoder_graph_replay_is_identical(eng3, gold):
    """The generator runs eagerly the first time a frame count is seen and as a CUDA-graph replay afterwards: same kernels,
    same split decisions, so the samples must be bit-identical; and identical to the eager path with the option off."""
    g = gold["vocoder"]
    codes = cuda(g["code"][0].astype(np.int64))
    dur, cum = eng3.vocoder_durations(codes, True)
    total = int(cum[-1].item())
    eng3.set_option("vocoder_graph", 1)
    first = eng3.vocoder_generate(total, total - 21, 21, -1).clone()   # eager + capture
    l0 = eng3.launch_count()
    second = eng3.vocoder_generate(total, total - 21, 21, -1).clone()  # replay
    replay_launches = eng3.launch_count() - l0
    third = eng3.vocoder_generate(total, total - 21, 21, -1).clone()
    eng3.set_option("vocoder_graph", 0)
    l0 = eng3.launch_count()
    eager = eng3.vocoder_generate(total, total - 21, 21, -1).clone()
    eager_launches = eng3.launch_count() - l0
    eng3.set_option("vocoder_graph", 1)
    report("vocoder_graph", replay_vs_first=maxdiff(second, first), eager_vs_replay=maxdiff(eager, second), replay_launches=replay_launches,
           eager_launches=eager_launches)
    assert torch.equal(first, second) and torch.equal(second, third) and torch.equal(eager, second)
    assert replay_launches == eager_launches  # the replay accounts for every kernel node it runs


# --------------------------------------------------------------------------------------------- tcgen05 kernels
@pytest.mark.parametrize("shape", [(128, 32, 16, 1, 1, 0, 1.0), (100, 64, 128, 3, 1, 1, 0.1), (260, 256, 256, 11, 5, 25, 0.1),
                                   (1040, 128, 128, 7, 3, 9, 0.1), (16640, 16, 16, 7, 5, 15, 0.1), (300, 128, 512, 7, 1, 3, 1.0),
                                   (775, 512, 2048, 1, 1, 0, 1.0), (200, 512, 1005, 1, 1, 0, 1.0), (130, 48, 48, 5, 2, 4, 0.1)])
def test_tcgen05_conv_vs_fp64_reference(eng3, shape):
    """kernels_umma2.cu (tap-shift implicit GEMM, bf16x3 / bf16x6 operand splitting) against torch conv1d in fp64 and against
    the fp32 CUDA-core kernel: 2 pieces within 2e-3 (vocoder path, waveform bar 1e-3 after 40 layers is checked by the
    vocoder tests), 3 pieces within 2e-4 (same bar as the fp32 kernels)."""
    import torch.nn.functional as F

    L, C, N, k, dil, pad, slope = shape
    g = torch.Generator().manual_seed(L + C + N + k)
    x = torch.randn(L, C, generator=g)
    w = torch.randn(N, k * C, generator=g) / (k * C) ** 0.5
    b = torch.randn(N, generator=g)
    xx = x.double()
    if slope != 1.0:
        xx = torch.where(xx > 0, xx, xx * slope)
    wt = w.double().view(N, k, C).permute(0, 2, 1).contiguous()
    ref = F.conv1d(F.pad(xx.t().unsqueeze(0), (pad, (k - 1) * dil - pad)), wt, b.double(), dilation=dil)[0].t().float()
    xd, wd, bd = cuda(x), cuda(w), cuda(b)
    d0 = maxdiff(eng3.op_conv1d(xd, wd, bd, k, dil, pad, slope, 0), ref)
    eng3.set_option("umma2_cache_clear", 1)  # weights of an earlier case may have lived at the same address
    d2 = maxdiff(eng3.op_conv1d(xd, wd, bd, k, dil, pad, slope, 12), ref)
    eng3.set_option("umma2_cache_clear", 1)
    d3 = maxdiff(eng3.op_conv1d(xd, wd, bd, k, dil, pad, slope, 13), ref)
    eng3.set_option("umma2_cache_clear", 1)
    report("tcgen05_conv", shape=list(shape), fp32=d0, bf16x3=d2, bf16x6=d3)
    assert d0 < FP_TOL and d2 < 2e-3 and d3 < FP_TOL, (d0, d2, d3)


def test_mt_cross_kv_reuse_of_final_rows(full):
    """ss_mt_stable_rows: cross-attention K / V of encoder rows declared final are projected once.  Two calls on a growing
    encoder buffer (the non-final tail changes between them) must give the tokens / features of hint-free calls."""
    cfg, e, o = full
    g = torch.Generator().manual_seed(3)
    buf = torch.randn(64, cfg.enc_dim, generator=g).cuda()
    e.encoder_stream_reset()
    t1, f1 = e.mt_greedy(buf[:24], None, 2, stable_rows=16)
    buf[16:40] = torch.randn(24, cfg.enc_dim, generator=g).cuda()  # rows >= 16 were provisional; 16 more arrive
    t2, f2 = e.mt_greedy(buf[:40], t1, 2, stable_rows=32)
    f2 = f2.clone()
    e.encoder_stream_reset()
    r2, g2 = e.mt_greedy(buf[:40].clone(), t1, 2)  # different buffer, no hint: every row projected
    d = maxdiff(f2, g2)
    report("mt_cross_reuse", feats=d)
    assert t2 == r2 and d < FP_TOL, (t2, r2, d)


# --------------------------------------------------------------------------------------------- end to end
def agent_args(**kw):
    d = dict(model_path="synthetic", data_bin=".", config_yaml=None, multitask_config_yaml=None, global_stats=None,
             tgt_splitter_type="SentencePiece", tgt_splitter_path=None, user_dir="", agent_dir="", max_len=200, force_finish=False,
             shift_size=10, window_size=25, sample_rate=16000, feature_dim=80, vocoder="synthetic", vocoder_cfg=None,
             dur_prediction=True, lagging_k1=0, lagging_k2=0, segment_size=320, stride_n=1, stride_n2=1, unit_per_subword=15,
             extra_output_dir=None, output_asr_translation=False, source_segment_size=320, vocoder_context="receptive-field",
             device_index=0, device="gpu")
    d.update(kw)
    return argparse.Namespace(**d)


@pytest.mark.parametrize("seconds,seed,mode,seg_ms", [(4.0, 1234, "cached", 320), (6.4, 77, "cached", 320), (3.0, 1234, "recompute", 320),
                                                     (10.0, 1234, "cached", 320),   # the utterance bench.py times (configs[1])
                                                     (5.12, 1234, "cached", 640),   # whole-word path (agent:540-574), configs[4] chunk
                                                     (4.8, 7, "cached", 480)])      # attention chunk 12 / conv chunk 8 (not nested); seed without a 1e-6 arg-max tie
def test_streaming_s2st_agent_vs_oracle(seconds, seed, mode, seg_ms):
    """Config 2 shape (chunk 320 ms, batch 1) and the 640 / 480 ms variants: every policy() call must reproduce the oracle
    agent's action, token sequences bit-exactly and the emitted waveform within 1e-3."""
    from oracle.agent_oracle import OracleS2STAgent
    from oracle.streamspeech_oracle import StreamSpeechOracle
    from streamspeech_b200.agent import StreamSpeechS2STAgent
    from streamspeech_b200.dictionary import Dictionary
    from streamspeech_b200.simuleval_compat import SpeechSegment

    cfg = ModelConfig()
    o = StreamSpeechOracle(cfg, synth.make_model_state_dict(cfg, 0), synth.make_vocoder_state_dict(cfg.vocoder, 1), synth.make_gcmvn(cfg))
    d = Dictionary.synthetic(cfg.tgt_vocab)
    ref = OracleS2STAgent(o, seg_ms, is_word_start=lambda t: d[t].startswith("\u2581"))
    agent = StreamSpeechS2STAgent(agent_args(encoder_mode=mode, vocoder_context="full" if mode == "recompute" else "receptive-field",
                                             source_segment_size=seg_ms))
    wav = synth.make_audio(seconds, seed=seed)
    n = 16 * seg_ms
    worst, writes = 0.0, 0
    for i in range(0, len(wav), n):
        fin = i + n >= len(wav)
        chunk = wav[i:i + n].tolist()
        ref.push(chunk, finished=fin)
        a_ref = ref.policy()
        seg = agent.pushpop(SpeechSegment(content=chunk, sample_rate=16000, finished=fin))
        for k in ("asr_tokens", "st_tokens", "new_subword_tokens", "mt_tokens", "units", "dur"):
            assert agent.trace.get(k) == a_ref.trace.get(k), (i // n, k, agent.trace.get(k), a_ref.trace.get(k))
        if a_ref.kind == "read":
            assert seg.is_empty, i // n
        else:
            assert not seg.is_empty and len(seg.content) == len(a_ref.wav), (i // n, len(seg.content), len(a_ref.wav))
            assert seg.finished == a_ref.seg_finished
            if len(a_ref.wav):
                worst = max(worst, float(np.abs(np.array(seg.content) - np.array(a_ref.wav)).max()))
                writes += 1
    report(f"s2st_streaming_{mode}_{seg_ms}ms", seconds=seconds, wav_maxdiff=worst, writes=writes)
    assert writes >= 1 and worst < WAV_TOL, (writes, worst)
    agent.engine.close()


def test_streaming_asr_agent_vs_oracle():
    from oracle.agent_oracle import OracleASRAgent
    from oracle.streamspeech_oracle import StreamSpeechOracle
    from streamspeech_b200.agent import StreamSpeechASRAgent
    from streamspeech_b200.simuleval_compat import SpeechSegment

    cfg = ModelConfig()
    o = StreamSpeechOracle(cfg, synth.make_model_state_dict(cfg, 0), None, synth.make_gcmvn(cfg))
    ref = OracleASRAgent(o, 160)
    agent = StreamSpeechASRAgent(agent_args(source_segment_size=160))
    wav = synth.make_audio(3.0, seed=3)
    n = 2560
    for i in range(0, len(wav), n):
        fin = i + n >= len(wav)
        chunk = wav[i:i + n].tolist()
        ref.push(chunk, finished=fin)
        a_ref = ref.policy()
        agent.pushpop(SpeechSegment(content=chunk, sample_rate=16000, finished=fin))
        if a_ref.kind == "write":
            assert agent.trace["asr_tokens"] == a_ref.trace["asr_tokens"], i // n
    agent.engine.close()


def test_missing_weight_fails_loudly():
    from streamspeech_b200.engine import Engine, EngineError

    cfg = golden_cfg()
    sd = synth.make_model_state_dict(cfg, 0)
    del sd["encoder.conformer_layers.1.ffn2.w_2.weight"]
    with pytest.raises(EngineError, match="ffn2.w_2.weight"):
        Engine(cfg, sd, None, None)


def test_unit_decoder_grouped_first_layer(eng3, gold):
    """Option unit_grouped: layer 1 of the unit decoder attends over the S distinct T2U rows with multiplicities instead of the
    25*S identical copies (reference quirk N1 makes the copies identical).  Must reproduce the full computation: fixture
    logits / arg-max, a long sequence, and the padded-tail variant."""
    g = gold["decoders"]
    feats = cuda(g["mt_feats"])
    big = feats.repeat(7, 1).contiguous() * torch.linspace(0.8, 1.2, 7 * feats.shape[0], device="cuda").unsqueeze(1)  # 49 tokens -> 1225 positions
    eng3.set_option("unit_grouped", 0)  # the reference of this test is the FULL 25*S-row first layer
    ref_small = eng3.t2u_unit_decode(feats, debug=True)
    ref_big = eng3.t2u_unit_decode(big, debug=True)
    ref_pad = eng3.t2u_unit_decode(cuda(g["mt_feats_pad"]), n_pad_tail=1, debug=True)
    ref_small = {k: v.clone() for k, v in ref_small.items() if v is not None}
    ref_big = {k: v.clone() for k, v in ref_big.items() if v is not None}
    ref_pad = {k: v.clone() for k, v in ref_pad.items() if v is not None}
    eng3.set_option("unit_grouped", 1)
    try:
        r = eng3.t2u_unit_decode(feats, debug=True)
        d1 = maxdiff(r["logits"], ref_small["logits"])
        d0 = maxdiff(r["logits"][:4], g["unit_logits_first"])
        assert r["argmax"].tolist() == g["unit_argmax"].tolist()
        rb = eng3.t2u_unit_decode(big, debug=True)
        d2 = maxdiff(rb["logits"], ref_big["logits"])
        assert rb["argmax"].tolist() == ref_big["argmax"].tolist()
        rp = eng3.t2u_unit_decode(cuda(g["mt_feats_pad"]), n_pad_tail=1, debug=True)
        d3 = maxdiff(rp["logits"], ref_pad["logits"])
        assert rp["argmax"].tolist() == g["unit_argmax_pad"].tolist()
    finally:
        eng3.set_option("unit_grouped", 1)  # the engine default
    report("unit_grouped", vs_full=d1, vs_fixture=d0, long_vs_full=d2, pad_vs_full=d3)
    assert d1 > 0.0, "the full-attention reference was not computed with unit_grouped = 0"
    assert d1 < 5e-5 and d0 < 5e-4 and d2 < 1e-4 and d3 < 5e-5, (d1, d0, d2, d3)


# --------------------------------------------------------------------------------------------- fixtures from the reference's own generator / policy
def test_mt_greedy_reference_generate_decoder_fixture(full, gold):
    """M1 against the REAL reference: tests/golden/mt_greedy.npz holds the tokens `SequenceGenerator.generate_decoder`
    (agent/sequence_generator.py:165-582, imported unchanged) finalized on the reference MT decoder."""
    cfg, e, o = full
    g = gold["mt_greedy"]
    e.set_chunk(8)
    enc = cuda(g["enc_out"])
    for i in range(int(g["n_cases"])):
        prefix = g[f"case{i}_prefix"].tolist() if bool(g[f"case{i}_has_prefix"]) else None
        toks, _ = e.mt_greedy(enc, prefix, int(g[f"case{i}_max_new"]), max_len_b=100)
        ref = g[f"case{i}_tokens"].tolist()
        assert ref[-1] == cfg.eos and toks == ref[:-1], (i, toks, ref)


@pytest.mark.parametrize("tag", ["c320", "c640"])
def test_s2st_agent_vs_reference_policy_fixture(gold, tag):
    """A1 / P1 against the REAL reference: tests/golden/agent_policy_<tag>.npz is the action sequence of the reference's own policy()
    (agent:422-770, executed from its source on reference generator / module objects, oracle/gen_golden_agent.py).  The engine
    agent must take the same READ / WRITE decisions, emit the same units and the same waveform (1e-3)."""
    from streamspeech_b200.agent import StreamSpeechS2STAgent
    from streamspeech_b200.simuleval_compat import SpeechSegment

    g = gold[f"agent_policy_{tag}"]
    seg_ms, seconds, seed = int(g[f"{tag}_segment_ms"]), float(g[f"{tag}_seconds"]), int(g[f"{tag}_seed"])
    agent = StreamSpeechS2STAgent(agent_args(source_segment_size=seg_ms))
    wav = synth.make_audio(seconds, seed=seed)
    n = 16 * seg_ms
    kinds = g[f"{tag}_kinds"].tolist()
    worst, writes = 0.0, 0
    for ci, i in enumerate(range(0, len(wav), n)):
        fin = i + n >= len(wav)
        seg = agent.pushpop(SpeechSegment(content=wav[i:i + n].tolist(), sample_rate=16000, finished=fin))
        assert (not seg.is_empty) == bool(kinds[ci]), (tag, ci)
        if kinds[ci]:
            ref = g[f"{tag}_call{ci}_wav"]
            assert len(seg.content) == len(ref), (tag, ci, len(seg.content), len(ref))
            assert bool(seg.finished) == bool(g[f"{tag}_call{ci}_flags"][1]), (tag, ci)
            if len(ref):
                assert agent.trace.get("units") == g[f"{tag}_call{ci}_units"].tolist(), (tag, ci)
                assert agent.trace.get("dur") == g[f"{tag}_call{ci}_dur"].tolist(), (tag, ci)
                worst = max(worst, float(np.abs(np.array(seg.content, dtype=np.float32) - ref).max()))
                writes += 1
    report("s2st_reference_policy_" + tag, wav_maxdiff=worst, writes=writes)
    assert writes >= 1 and worst < WAV_TOL, (writes, worst)
    agent.engine.close()


def test_s2tt_agent_vs_reference_policy_fixture_and_oracle(gold):
    """Row f1: StreamSpeechS2TTAgent (incremental MT decoder states across policy() calls, SURVEY.md N12) against (a) the action
    sequence of the reference's own S2TT policy() (tests/golden/agent_policy_s2tt320.npz, oracle/gen_golden_agent.py) and (b) the
    oracle agent on a second utterance: every text delta and every hypothesis bit-exact."""
    from oracle.agent_oracle import OracleS2TTAgent
    from oracle.streamspeech_oracle import StreamSpeechOracle
    from streamspeech_b200.agent import StreamSpeechS2TTAgent
    from streamspeech_b200.dictionary import Dictionary
    from streamspeech_b200.simuleval_compat import SpeechSegment

    g = gold["agent_policy_s2tt320"]
    tag = "s2tt320"
    seg_ms, seconds, seed = int(g[f"{tag}_segment_ms"]), float(g[f"{tag}_seconds"]), int(g[f"{tag}_seed"])
    agent = StreamSpeechS2TTAgent(agent_args(source_segment_size=seg_ms))
    wav = synth.make_audio(seconds, seed=seed)
    n = 16 * seg_ms
    kinds, texts = g[f"{tag}_kinds"].tolist(), g[f"{tag}_texts"].tolist()
    for ci, i in enumerate(range(0, len(wav), n)):
        fin = i + n >= len(wav)
        seg = agent.pushpop(SpeechSegment(content=wav[i:i + n].tolist(), sample_rate=16000, finished=fin))
        assert (not seg.is_empty) == bool(kinds[ci]), ci
        if kinds[ci]:
            assert seg.content == texts[ci], (ci, seg.content, texts[ci])
            assert agent.trace["mt_tokens"] == g[f"{tag}_call{ci}_mt_tokens"].tolist(), ci
    # (b) a second utterance through the same agent object (reset() must clear the incremental state), vs the oracle
    cfg = ModelConfig()
    o = StreamSpeechOracle(cfg, synth.make_model_state_dict(cfg, 0), None, synth.make_gcmvn(cfg))
    d = Dictionary.synthetic(cfg.tgt_vocab)
    ref = OracleS2TTAgent(o, seg_ms, symbols=lambda t: d[t])
    wav = synth.make_audio(3.2, seed=99)
    writes = 0
    for ci, i in enumerate(range(0, len(wav), n)):
        fin = i + n >= len(wav)
        chunk = wav[i:i + n].tolist()
        ref.push(chunk, finished=fin)
        a = ref.policy()
        seg = agent.pushpop(SpeechSegment(content=chunk, sample_rate=16000, finished=fin))
        assert seg.is_empty == (a.kind == "read"), ci
        if a.kind == "write":
            assert seg.content == a.wav and agent.trace["mt_tokens"] == a.trace["mt_tokens"], ci
            writes += 1
    report("s2tt_agent", writes=writes)
    assert writes >= 2
    agent.engine.close()


def test_grid_barrier_error_flag_is_clear_after_the_suite(full):
    """ss_async_error: no persistent-kernel grid barrier timed out during the tests above on this handle."""
    cfg, e, o = full
    e.check_async_error()


def test_ctc_pair_equals_single_heads(eng3, gold):
    """ss_ctc_greedy_pair (one [rows][2V] projection + fused arg-max / collapse with the last-block ticket) against the
    single-head entry point and the reference fixture, full sequence and incremental (row0 > 0) forms."""
    g = gold["decoders"]
    enc = cuda(g["enc_out"])
    T = enc.shape[0]
    am = [torch.zeros(T, dtype=torch.int64, device="cuda") for _ in range(2)]
    for row0 in (0, T - 9, T):
        if row0 > 0:  # rows below row0 must already hold their arg-max
            for hd in (0, 1):
                am[hd][:row0] = eng3.ctc_greedy(hd, enc)["argmax"][:row0]
                am[hd][row0:] = -7
        a, b = eng3.ctc_greedy_rows_pair(enc, [row0, row0], am)
        for hd, name, (toks, idx) in ((0, "source_unigram", a), (1, "ctc_target_unigram", b)):
            assert am[hd].tolist() == g[f"ctc_{name}_argmax"].tolist(), (row0, name)
            assert toks == g[f"ctc_{name}_tokens"].tolist() and idx == g[f"ctc_{name}_index"].tolist(), (row0, name)


@pytest.mark.parametrize("option", ["persistent_ffn_fused", "persistent_mt_prefix", "persistent_mt_v2"])
def test_persistent_kernel_variants_agree(full, option):
    """A / B of the round-2 persistent-kernel restructurings against the paths they replace: fused FFN phases (hidden-split
    rank-16 updates + deterministic reduce) vs separate W1 / W2 phases in the encoder step; cooperative MT prefix pass vs the
    per-kernel prefix pass; single-token MT kernel with 6 barriers per layer (head-group partial projections) vs 8.  Same function,
    different summation order."""
    cfg, e, o = full
    e.set_chunk(8, 8)
    feats = e.fbank(cuda(synth.make_audio(3.0, seed=5)))
    outs = {}
    for v in (0, 1):
        e.set_option(option, v)
        buf = torch.zeros(1024, cfg.enc_dim, device="cuda")
        e.encoder_stream_reset()
        T = 0
        for F in list(range(30, feats.shape[0], 32)) + [feats.shape[0]]:
            T, _ = e.encoder_stream_step(feats[:F].contiguous(), buf)
        toks, mt_feats = e.mt_greedy(buf[:T].contiguous(), [17, 256, 4099, 31, 5, 977, 1203, 44], 3)
        outs[v] = (buf[:T].clone(), toks, mt_feats.clone())
    e.set_option(option, 1)
    d_enc, d_mt = maxdiff(outs[0][0], outs[1][0]), maxdiff(outs[0][2], outs[1][2])
    report("persistent_variant_" + option, enc=d_enc, mt_feats=d_mt)
    assert outs[0][1] == outs[1][1] and d_enc < 2e-5 and d_mt < 1e-4, (d_enc, d_mt)
    e.encoder_stream_reset()


@pytest.mark.parametrize("attn_chunk,conv_chunk,step_frames", [(8, 8, 32), (16, 16, 64), (16, 8, 64), (8, 8, 17), (32, 16, 128), (4, 8, 16), (2, 8, 8)])
def test_cluster_encoder_kernel_agrees(full, attn_chunk, conv_chunk, step_frames):
    """A / B of the cluster encoder kernel (kernels_persist_cl.cu: 4 clusters x 16 CTAs, activations in distributed shared memory,
    weights streamed from repacked blobs) against the 148-CTA kernel on the same stream of calls, including ragged step sizes and a
    chunk size whose steps exceed 16 active rows (those steps must fall back to the 148-CTA kernel, not fail).  Same function, different
    summation order; the streaming caches written by one kernel are read by the other in the mixed case."""
    cfg, e, o = full
    e.set_chunk(attn_chunk, conv_chunk)
    feats = e.fbank(cuda(synth.make_audio(4.0, seed=9)))
    outs = {}
    steps = {}
    for v in (0, 1):
        e.set_option("persistent_encoder_cluster", v)
        buf = torch.zeros(1024, cfg.enc_dim, device="cuda")
        e.encoder_stream_reset()
        n0 = e.cluster_steps()
        T = 0
        snaps = []
        for F in list(range(step_frames - 2, feats.shape[0], step_frames)) + [feats.shape[0]]:
            T, Tf = e.encoder_stream_step(feats[:F].contiguous(), buf)
            snaps.append(buf[:T].clone())
        steps[v] = e.cluster_steps() - n0
        toks = [e.ctc_greedy(h, buf[:T].contiguous())["argmax"].tolist() for h in (0, 1)]
        outs[v] = (snaps, toks)
    e.set_option("persistent_encoder_cluster", 1)
    e.check_async_error()
    assert steps[0] == 0
    assert steps[1] > 0 or attn_chunk > 16, steps
    d = max(maxdiff(a, b) for a, b in zip(outs[0][0], outs[1][0]))
    report(f"cluster_encoder_{attn_chunk}_{conv_chunk}_{step_frames}", enc=d, cluster_steps=steps[1], calls=len(outs[0][0]))
    assert d < 5e-5 and outs[0][1] == outs[1][1], d
    e.encoder_stream_reset()


def test_cluster_encoder_kernel_long_utterance(full):
    """The cluster kernel on a 38 s stream (T up to ~950 rows: several batches of key slots per CTA in the attention, long L2 prefetch
    lists) against the 148-CTA kernel; only every 8th call is compared in full."""
    cfg, e, o = full
    e.set_chunk(8, 8)
    feats = e.fbank(cuda(synth.make_audio(38.0, seed=11)))
    outs = {}
    for v in (0, 1):
        e.set_option("persistent_encoder_cluster", v)
        buf = torch.zeros(1024, cfg.enc_dim, device="cuda")
        e.encoder_stream_reset()
        n0 = e.cluster_steps()
        snaps = []
        T = 0
        for k, F in enumerate(list(range(30, feats.shape[0], 32)) + [feats.shape[0]]):
            T, _ = e.encoder_stream_step(feats[:F].contiguous(), buf)
            if k % 8 == 7:
                snaps.append(buf[:T].clone())
        snaps.append(buf[:T].clone())
        outs[v] = (snaps, e.cluster_steps() - n0, T)
    e.set_option("persistent_encoder_cluster", 1)
    e.check_async_error()
    assert outs[1][1] > 100 and outs[0][1] == 0 and outs[1][2] > 900, (outs[0][1:], outs[1][1:])
    d = max(maxdiff(a, b) for a, b in zip(outs[0][0], outs[1][0]))
    report("cluster_encoder_38s", enc=d, cluster_steps=outs[1][1], T=outs[1][2])
    assert d < 5e-5, d
    e.encoder_stream_reset()


def test_resample_48k_to_16k_vs_torchaudio(eng3):
    """f3 wire format: ss_resample_48k_to_16k against torchaudio.functional.resample (the CPU oracle of this front end; the
    reference's sox `rate` is not available in this image, DESIGN.md) on whole signals of awkward lengths, and the streaming rule
    (only samples with complete filter support while the source is open) reproducing the whole-signal result incrementally."""
    import torchaudio

    g = torch.Generator().manual_seed(5)
    for n in (1, 21, 22, 23, 480, 15360, 48000 + 1, 160001):
        x = torch.rand(n, generator=g) * 2 - 1
        ref = torchaudio.functional.resample(x, 48000, 16000)
        xd = cuda(x)
        out = torch.zeros(ref.numel(), device="cuda")
        assert eng3.resample_out_len(n, True) == ref.numel()
        # incrementally: chunks of 7001 input samples, final flush at the end
        done = 0
        for end in list(range(7001, n, 7001)) + [n]:
            fin = end == n
            avail = eng3.resample_out_len(end, fin)
            if avail > done:
                eng3.resample_48k_to_16k(xd[:end].contiguous(), out, done, avail - done)
                done = avail
        assert done == ref.numel()
        d = maxdiff(out, ref)
        assert d < 2e-6, (n, d)


def test_s2st_agent_48k_source_equals_16k_agent_on_resampled_audio():
    """The reference's default: states.source at 48 kHz (agent:32-35,66).  The agent with --sample-rate 48000 must behave like the
    16 kHz agent fed the resampled signal, call by call."""
    import torchaudio

    from streamspeech_b200.agent import StreamSpeechS2STAgent
    from streamspeech_b200.simuleval_compat import SpeechSegment

    x48 = synth.make_audio(9.6, seed=8)[: 3 * 51200]  # any 48 kHz signal: 3.2 s
    x16 = torchaudio.functional.resample(x48, 48000, 16000)
    a48 = StreamSpeechS2STAgent(agent_args(sample_rate=48000))
    a16 = StreamSpeechS2STAgent(agent_args(sample_rate=16000))
    n = 5120
    writes = 0
    for i in range(0, x16.numel(), n):
        fin = i + n >= x16.numel()
        s48 = a48.pushpop(SpeechSegment(content=x48[3 * i:3 * (i + n)].tolist(), sample_rate=48000, finished=fin))
        s16 = a16.pushpop(SpeechSegment(content=x16[i:i + n].tolist(), sample_rate=16000, finished=fin))
        assert s48.is_empty == s16.is_empty, i // n
        for k in ("asr_tokens", "st_tokens", "mt_tokens", "units", "dur"):
            assert a48.trace.get(k) == a16.trace.get(k), (i // n, k)
        if not s16.is_empty and len(s16.content):
            assert len(s48.content) == len(s16.content)
            assert float(np.abs(np.array(s48.content) - np.array(s16.content)).max()) < WAV_TOL
            writes += 1
    assert writes >= 1
    a48.engine.close()
    a16.engine.close()


def test_fairseq_surface_model_on_the_engine(gold):
    """§8b(ii): the nn.Module shims of fairseq_surface.py driven the way the reference agent drives its model object: chunk-size
    pokes (agent:404-413), encoder.forward -> fairseq-shaped dict (s2t_conformer.py:154-163), CTC decoder modules, MT features."""
    from streamspeech_b200.fairseq_surface import StreamSpeechB200Model

    cfg = golden_cfg()
    sd = synth.make_model_state_dict(cfg, 0)
    model = StreamSpeechB200Model.from_checkpoint(sd, None, None)
    assert model.cfg.enc_layers == 3 and model.mt_task_name == "target_unigram"
    g = gold["encoder"]
    model.encoder.chunk_size = 8
    for conv in model.encoder.subsample.conv_layers:
        conv.chunk_size = 8
    for layer in model.encoder.conformer_layers:
        layer.conv_module.depthwise_conv.chunk_size = 8
    src = torch.from_numpy(g["feats"])
    F = src.shape[0]
    fb = torch.zeros(2, F, 80)
    fb[0] = src
    fb[1, :150] = src[:150]
    out = model.encoder(fb, torch.tensor([F, 150]))
    eo = out["encoder_out"][0]
    assert eo.shape[1] == 2 and len(out["encoder_padding_mask"]) == 1 and out["encoder_padding_mask"][0].shape == (2, eo.shape[0])
    assert g["batched_lens"].tolist() == [F, 150]
    d = maxdiff(eo, g["batched_out"])
    report("fairseq_surface_encoder", maxdiff=d)
    assert d < FP_TOL, d
    dg = gold["decoders"]
    enc = cuda(dg["enc_out"]).unsqueeze(1)
    for name in ("source_unigram", "ctc_target_unigram"):
        logits = getattr(model, f"{name}_decoder")(enc)["encoder_out"]
        lp = model.get_normalized_probs([logits], log_probs=True)
        lp[:, :, cfg.pad] = float("-inf")
        lp[:, :, cfg.unk] = float("-inf")
        assert lp.argmax(-1)[:, 0].tolist() == dg[f"ctc_{name}_argmax"].tolist(), name
    x, extra = model.target_unigram_decoder(torch.from_numpy(dg["mt_tokens"]), encoder_out={"encoder_out": [enc]}, features_only=True)
    assert maxdiff(x[0], dg["mt_feats"]) < FP_TOL
    model.engine.close()


def test_generate_waveform_from_code_front_door(tmp_path, gold):
    """§8 f4: the reference's vocoder script interface (generate_waveform_from_code.py:40-111) on the engine: code file in,
    <i>_pred.wav out, waveform = the fixture of the reference CodeGenerator within the 16-bit quantisation of the file."""
    import json
    import wave

    from streamspeech_b200.generate_waveform_from_code import cli_main

    g = gold["vocoder"]
    (tmp_path / "unit.txt").write_text(" ".join(str(int(c)) for c in g["code"][0]) + "\n" + "5 5 17 900\n")
    json.dump(VocoderConfig().to_json_dict(), open(tmp_path / "config.json", "w"))
    n = cli_main(["--in-code-file", str(tmp_path / "unit.txt"), "--vocoder", "synthetic", "--vocoder-cfg", str(tmp_path / "config.json"),
                  "--results-path", str(tmp_path / "out"), "--dur-prediction"])
    assert n == 2
    with wave.open(str(tmp_path / "out" / "0_pred.wav")) as w:
        assert w.getframerate() == 16000 and w.getnchannels() == 1
        pcm = np.frombuffer(w.readframes(w.getnframes()), dtype="<i2").astype(np.float32) / 32768.0
    assert pcm.shape[0] == g["wav"].shape[0]
    assert float(np.abs(pcm - np.clip(g["wav"], -1, 32767 / 32768)).max()) < 1e-3 + 1.0 / 32768


def test_umma2_in_kernel_split_reduction_is_bit_identical(eng3, gold):
    """The last-ticket CTA of an output tile reduces the split partial sums inside umma2_kernel (no splitk_epilogue launch): same
    slice order and arithmetic as the separate reduce kernel, so the vocoder waveform and the unit-decoder logits must be
    bit-identical with the option on and off."""
    g = gold["vocoder"]
    code = torch.from_numpy(g["code"][0]).cuda()
    feats = cuda(gold["decoders"]["mt_feats"])
    res = {}
    for v in (0, 1):
        eng3.set_option("umma2_fused_reduce", v)
        l0 = eng3.launch_count()
        dur, cum = eng3.vocoder_durations(code, True)
        total = int(cum[-1].item())
        wav = eng3.vocoder_generate(total, 0, total, 0).clone()
        r = eng3.t2u_unit_decode(feats.repeat(5, 1).contiguous(), debug=True)
        res[v] = (wav, r["logits"].clone(), eng3.launch_count() - l0)
    eng3.set_option("umma2_fused_reduce", 0)  # the engine default (the in-kernel reduction measured slower, kernels_umma2.cu)
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])
    report("umma2_fused_reduce", launches_separate=res[0][2], launches_fused=res[1][2])
    assert res[1][2] < res[0][2]


def test_capacity_and_misuse_fail_loudly(eng3):
    """Error behaviour of the C-ABI (SURVEY.md §5: status codes, never a silent wrong answer): sequences beyond the configured
    maximum, a chunk-less model on the streaming entry point, a prefix the incremental MT state did not produce."""
    from streamspeech_b200.engine import Engine, EngineError

    cfg = golden_cfg()
    e = Engine(cfg, synth.make_model_state_dict(cfg, 0), None, None, max_enc_frames=64)
    try:
        e.set_chunk(8, 8)
        feats = torch.zeros(64 * 4 + 40, cfg.feat_dim, device="cuda")
        buf = torch.zeros(128, cfg.enc_dim, device="cuda")
        with pytest.raises(EngineError, match="max_enc_frames"):
            e.encoder_stream_step(feats, buf)
        with pytest.raises(EngineError, match="max_enc_frames"):
            e.encoder(feats.unsqueeze(0))
        e.set_chunk(None)
        with pytest.raises(EngineError, match="chunked model"):
            e.encoder_stream_step(feats[:40].contiguous(), buf)
        e.set_chunk(8, 8)
        enc = torch.randn(20, cfg.enc_dim, device="cuda")
        e.mt_incremental_reset()
        with pytest.raises(EngineError, match="incremental MT state is shorter"):
            e.mt_greedy_incremental(enc, [17, 18, 19], 2, 100)
        with pytest.raises(EngineError, match="no vocoder"):
            e.vocoder_durations(torch.zeros(4, dtype=torch.int64, device="cuda"))
    finally:
        e.close()
