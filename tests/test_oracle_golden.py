"""CPU: the oracle restatement reproduces the fixtures dumped from the REAL reference modules
(oracle/gen_golden.py) and the reference's own known-answer tests for this path."""
import numpy as np
import pytest
import torch

from oracle.streamspeech_oracle import (StreamSpeechOracle, kaldi_fbank, online_features, rel_positional_encoding,
                                        rel_shift, ctc_collapse, num_fbank_frames)
from streamspeech_b200 import synth
from streamspeech_b200.config import ModelConfig, VocoderConfig

torch.set_grad_enabled(False)


def golden_cfg():
    cfg = ModelConfig()
    cfg.enc_layers = 3  # what oracle/gen_golden.py used
    return cfg


def test_kat_rel_shift_and_positional_encoding(gold):
    # fairseq/tests/test_espnet_multihead_attention.py:99-115 and test_positional_encoding.py:17-59
    g = gold["kat_relpos"]
    assert np.array_equal(rel_shift(torch.from_numpy(g["shift_in"])).numpy(), g["shift_out"])
    assert np.array_equal(rel_positional_encoding(3, 4).numpy(), g["pe_T3_d4"])
    # the values the reference test hard-codes for rel_shift on arange(30).view(1,2,3,5)
    exp = torch.tensor([[[[2.0, 3, 4], [6, 7, 8], [10, 11, 12]], [[17, 18, 19], [21, 22, 23], [25, 26, 27]]]])
    assert torch.equal(rel_shift(torch.arange(0, 30, dtype=torch.float32).view(1, 2, 3, 5)), exp)


def test_fbank_matches_torchaudio_fixture(gold):
    g = gold["fbank"]
    mine = kaldi_fbank(torch.from_numpy(g["wav"]) * 2 ** 15)
    assert mine.shape == g["fbank"].shape
    assert np.abs(mine.numpy() - g["fbank"]).max() < 1e-4


def test_num_frames_rule():
    # agent:70-81: F = floor((n - 240) / 160)
    assert num_fbank_frames(160000) == 998 and num_fbank_frames(5120) == 30 and num_fbank_frames(239) == 0
    assert num_fbank_frames(400) == 1 and num_fbank_frames(399) == 0


def test_encoder_fixtures(gold):
    g = gold["encoder"]
    cfg = golden_cfg()
    sd = synth.make_model_state_dict(cfg, seed=0)
    feats = torch.from_numpy(g["feats"])
    for chunk, conv in ((4, 8), (8, 8), (16, 16), (None, None)):
        o = StreamSpeechOracle(cfg, sd, None, None, chunk_size=chunk, conv_chunk_size=conv)
        out = o.encoder(feats.unsqueeze(0), torch.tensor([feats.size(0)]), return_layers=True)
        assert np.abs(out["encoder_out"][0][:, 0].numpy() - g[f"out_c{chunk}"]).max() < 2e-5
        assert np.abs(out["encoder_states"][0][:, 0].numpy() - g[f"layer0_c{chunk}"]).max() < 2e-5
        sub, _ = o.subsample(feats.unsqueeze(0), torch.tensor([feats.size(0)]))
        assert np.abs(sub[:, 0].numpy() - g[f"sub_c{chunk}"]).max() < 2e-5
    o = StreamSpeechOracle(cfg, sd, None, None, chunk_size=8, conv_chunk_size=8)
    fb = torch.zeros(2, feats.size(0), 80)
    fb[0] = feats
    fb[1, :150] = feats[:150]
    out = o.encoder(fb, torch.from_numpy(g["batched_lens"]))
    assert np.abs(out["encoder_out"][0].numpy() - g["batched_out"]).max() < 2e-5


def test_decoder_fixtures(gold):
    g = gold["decoders"]
    cfg = golden_cfg()
    sd = synth.make_model_state_dict(cfg, seed=0)
    o = StreamSpeechOracle(cfg, sd, None, None, chunk_size=8)
    eo = torch.from_numpy(g["enc_out"]).unsqueeze(1)
    for name in ("source_unigram", "ctc_target_unigram"):
        h = o.ctc_greedy(name, eo)[0]
        assert h["org_tokens"] == g[f"ctc_{name}_argmax"].tolist()
        assert h["tokens"] == g[f"ctc_{name}_tokens"].tolist()
        assert h["index"] == g[f"ctc_{name}_index"].tolist()
    toks = torch.from_numpy(g["mt_tokens"])
    assert np.abs(o.mt_features(toks, eo)[0].numpy() - g["mt_feats"]).max() < 2e-5
    assert np.abs(o.mt_logits(toks, eo)[0, -1].numpy() - g["mt_logits_last"]).max() < 5e-5
    tp = torch.from_numpy(g["mt_tokens_pad"])
    fp = o.mt_features(tp, eo)
    assert np.abs(fp[0].numpy() - g["mt_feats_pad"]).max() < 2e-5
    x = torch.from_numpy(g["mt_feats"]).unsqueeze(1)
    t2u = o.t2u_encoder(x, None)
    assert np.abs(t2u[:, 0].numpy() - g["t2u_out"]).max() < 2e-5
    lg = o.unit_decoder_logits(t2u, None)
    assert np.abs(lg[0, :4].numpy() - g["unit_logits_first"]).max() < 1e-4
    h = o.unit_ctc_greedy(lg)[0]
    assert h["org_tokens"] == g["unit_argmax"].tolist()
    assert h["tokens"] == g["unit_tokens"].tolist()
    pm = tp.eq(1)
    lgp = o.unit_decoder_logits(o.t2u_encoder(fp.transpose(0, 1), pm), pm)
    assert lgp[0].argmax(-1).tolist() == g["unit_argmax_pad"].tolist()


def test_vocoder_fixture(gold):
    g = gold["vocoder"]
    cfg = golden_cfg()
    for wn in (True, False):
        vsd = synth.make_vocoder_state_dict(VocoderConfig(), seed=1, weight_norm=wn)
        o = StreamSpeechOracle(cfg, synth.make_model_state_dict(cfg.tiny(), 0, None), vsd, None)
        wav, dur = o.vocoder(g["code"][0].tolist(), True)
        assert np.array_equal(dur.numpy(), g["dur"])
        assert np.abs(wav.numpy() - g["wav"]).max() < 1e-5


def test_ctc_collapse_edge_cases():
    assert ctc_collapse([], 0, 1) == ([], [])
    assert ctc_collapse([0, 0, 0], 0, 1) == ([], [])
    assert ctc_collapse([5, 5, 0, 5, 1, 7, 7], 0, 1) == ([5, 5, 7], [0, 3, 5])


def test_mt_greedy_semantics():
    """Forced EOS at max_len, min_len ban of EOS at step 0, prefix forcing (agent/sequence_generator.py:205-215,362-379)."""
    cfg = ModelConfig().tiny()
    sd = synth.make_model_state_dict(cfg, seed=0)
    o = StreamSpeechOracle(cfg, sd, None, None, chunk_size=8)
    eo = torch.randn(12, 1, cfg.enc_dim, generator=torch.Generator().manual_seed(0))
    h = o.mt_greedy(eo, None, 3)
    assert h[-1] == cfg.eos and 2 <= len(h) <= 4 and cfg.eos not in h[:-1]
    h2 = o.mt_greedy(eo, h[:-1], 2)
    assert h2[: len(h) - 1] == h[:-1] and h2[-1] == cfg.eos and len(h2) <= len(h) - 1 + 3
    h0 = o.mt_greedy(eo, h[:-1], 0)  # no new tokens allowed: eos is forced immediately
    assert h0 == h[:-1] + [cfg.eos]


def test_unit_decoder_first_layer_grouped_attention_identity(gold):
    """What the engine's grouped first layer (kernels_attn.cu: grouped_causal_attn_kernel) relies on, checked on the oracle:
    (1) quirk N1 gives every one of the 25 upsampled copies of a T2U state the same positional row, so the copies enter
    layer 1 identical; (2) causal self-attention over such a sequence equals attention over the S distinct keys with
    multiplicities 25 (earlier groups) and r + 1 (own group) -- including the padded-tail variant."""
    import torch.nn.functional as F

    from oracle.streamspeech_oracle import StreamSpeechOracle, _lin, _ln, make_positions, mha, sinusoidal_table
    from streamspeech_b200 import synth as synth_
    from streamspeech_b200.config import ModelConfig as MC

    cfg = MC()
    cfg.enc_layers = 3
    sd = synth_.make_model_state_dict(cfg, 0)
    o = StreamSpeechOracle(cfg, sd, None, synth_.make_gcmvn(cfg), chunk_size=8)
    t2u = torch.from_numpy(gold["decoders"]["t2u_out"]).unsqueeze(1)  # [S, 1, 512]
    S, R, H, E = t2u.shape[0], cfg.ctc_upsample_rate, cfg.unit_heads, cfg.unit_dim
    x = t2u.unsqueeze(1).repeat(1, R, 1, 1).contiguous().view(S * R, 1, E)
    table = sinusoidal_table(cfg.pad + 4, E, cfg.pad)
    x = x + table.index_select(0, make_positions(x[:, :, 0], cfg.pad).view(-1)).view(S * R, 1, -1)
    assert torch.equal(x.view(S, R, E), x.view(S, R, E)[:, :1].expand(S, R, E))  # (1)
    p = "decoder.layers.0"
    y = _ln(x, o.sd, p + ".self_attn_layer_norm")
    L = S * R
    causal = torch.triu(torch.ones(L, L, dtype=torch.bool), 1)
    for n_valid in (S, S - 1):
        pad = None
        if n_valid < S:
            pad = (torch.arange(S) >= n_valid).unsqueeze(0).unsqueeze(2).repeat(1, 1, R).view(1, L)
        full = mha(o.sd, p + ".self_attn", y, y, H, causal, pad)
        # grouped: S distinct rows, multiplicities
        yg = y.view(S, R, E)[:, 0]
        hd = E // H
        q = (_lin(yg, o.sd, p + ".self_attn.q_proj") * hd ** -0.5).view(S, H, hd)
        k = _lin(yg, o.sd, p + ".self_attn.k_proj").view(S, H, hd)
        v = _lin(yg, o.sd, p + ".self_attn.v_proj").view(S, H, hd)
        out = torch.zeros(S, R, H, hd)
        for g in range(S):
            n_prev, own = min(g, n_valid), g < n_valid
            keys = list(range(n_prev)) + ([g] if own else [])
            for h in range(H):
                s = torch.stack([q[g, h] @ k[j, h] for j in keys])
                e = torch.exp(s - s.max())
                a = e[:n_prev].sum()
                A = (e[:n_prev, None] * v[:n_prev, h]).sum(0) if n_prev else torch.zeros(hd)
                for r in range(R):
                    c = float(r + 1) if own else 0.0
                    e_own = e[n_prev] if own else torch.tensor(0.0)
                    out[g, r, h] = (R * A + c * e_own * (v[g, h] if own else 0)) / (R * a + c * e_own)
        grouped = _lin(out.view(L, 1, E), o.sd, p + ".self_attn.out_proj")
        assert float((grouped - full).abs().max()) < 2e-5, n_valid


def test_mt_greedy_matches_reference_generate_decoder(gold):
    """M1 pin: tests/golden/mt_greedy.npz holds the finalized tokens of the reference's own
    `agent/sequence_generator.py:SequenceGenerator.generate_decoder` (beam 1, the agent's constructor arguments) on the
    reference MT decoder (oracle/gen_golden_agent.py); the restatement must return the same tokens for every
    (prefix, max_new_tokens) case, including the forced-eos and max_new_tokens = -1 cases."""
    g = gold["mt_greedy"]
    cfg = ModelConfig()
    o = StreamSpeechOracle(cfg, synth.make_model_state_dict(cfg, 0), None, synth.make_gcmvn(cfg), chunk_size=8)
    eo = torch.from_numpy(g["enc_out"]).unsqueeze(1)
    for i in range(int(g["n_cases"])):
        prefix = g[f"case{i}_prefix"].tolist() if bool(g[f"case{i}_has_prefix"]) else None
        k = int(g[f"case{i}_max_new"])
        if k == -1 and i not in (2,):  # the 99-step cases cost ~10 s each on the CPU: one of them is enough here
            continue
        assert o.mt_greedy(eo, prefix, k, max_len_b=100, max_decoder_positions=1200) == g[f"case{i}_tokens"].tolist(), i


@pytest.mark.parametrize("tag", ["c320", "c640"])
def test_agent_oracle_matches_reference_policy_fixture(gold, tag):
    """A1 / P1 pin: tests/golden/agent_policy_<tag>.npz is the action sequence of the reference's own `policy()` (executed from its
    source on reference generator / module objects, oracle/gen_golden_agent.py) for a 320 ms utterance and a 640 ms
    (whole-word, agent:540-574) utterance.  OracleS2STAgent must reproduce every READ / WRITE, the flags, and the waveform."""
    from oracle.agent_oracle import OracleS2STAgent
    from streamspeech_b200.dictionary import Dictionary

    g = gold[f"agent_policy_{tag}"]
    cfg = ModelConfig()
    o = StreamSpeechOracle(cfg, synth.make_model_state_dict(cfg, 0), synth.make_vocoder_state_dict(cfg.vocoder, 1, weight_norm=True),
                           synth.make_gcmvn(cfg))
    d = Dictionary.synthetic(cfg.tgt_vocab)
    seg_ms, seconds, seed = int(g[f"{tag}_segment_ms"]), float(g[f"{tag}_seconds"]), int(g[f"{tag}_seed"])
    ag = OracleS2STAgent(o, seg_ms, is_word_start=lambda t: d[t].startswith("▁"))
    wav = synth.make_audio(seconds, seed=seed)
    n = 16 * seg_ms
    kinds = g[f"{tag}_kinds"].tolist()
    for ci, i in enumerate(range(0, len(wav), n)):
        fin = i + n >= len(wav)
        ag.push(wav[i:i + n].tolist(), finished=fin)
        a = ag.policy()
        assert (a.kind == "write") == bool(kinds[ci]), (tag, ci)
        if a.kind == "write":
            ref = g[f"{tag}_call{ci}_wav"]
            assert len(a.wav) == len(ref), (tag, ci)
            assert [a.finished, a.seg_finished] == g[f"{tag}_call{ci}_flags"].tolist()
            if len(ref):
                assert float(np.abs(np.array(a.wav, dtype=np.float32) - ref).max()) < 1e-5, (tag, ci)
            assert a.trace.get("units", []) == g[f"{tag}_call{ci}_units"].tolist()


def test_s2tt_oracle_matches_reference_policy_fixture(gold):
    """f1 pin: the S2TT agent's policy() (agent/speech_to_text.s2tt.streamspeech.agent.py:381-545) executed from its own source
    with the reference SequenceGenerator in incremental-state mode (N12: duplicate self-attention entry per call, stale
    cross-attention K / V).  OracleS2TTAgent must emit the same text deltas."""
    from oracle.agent_oracle import OracleS2TTAgent
    from streamspeech_b200.dictionary import Dictionary

    g = gold["agent_policy_s2tt320"]
    cfg = ModelConfig()
    o = StreamSpeechOracle(cfg, synth.make_model_state_dict(cfg, 0), None, synth.make_gcmvn(cfg))
    d = Dictionary.synthetic(cfg.tgt_vocab)
    tag = "s2tt320"
    seg_ms, seconds, seed = int(g[f"{tag}_segment_ms"]), float(g[f"{tag}_seconds"]), int(g[f"{tag}_seed"])
    ag = OracleS2TTAgent(o, seg_ms, symbols=lambda t: d[t])
    wav = synth.make_audio(seconds, seed=seed)
    n = 16 * seg_ms
    kinds, texts = g[f"{tag}_kinds"].tolist(), g[f"{tag}_texts"].tolist()
    for ci, i in enumerate(range(0, len(wav), n)):
        fin = i + n >= len(wav)
        ag.push(wav[i:i + n].tolist(), finished=fin)
        a = ag.policy()
        assert (a.kind == "write") == bool(kinds[ci]), ci
        if a.kind == "write":
            assert a.wav == texts[ci], (ci, a.wav, texts[ci])
            assert a.trace["mt_tokens"] == g[f"{tag}_call{ci}_mt_tokens"].tolist()
