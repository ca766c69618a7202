"""Pin M1 (greedy generate_decoder) and A1 / P1 (the agent's policy()) to the REAL reference code (build container only).

Run:  python -m oracle.gen_golden_agent        (needs /root/reference; CPU only, ~2 min)

M1.  The reference's own `agent/sequence_generator.py:SequenceGenerator` (imported unchanged, on top of the unchanged
     `fairseq/sequence_generator.py` and `fairseq/search.py`; the only stub added to oracle/ref_loader is a bare
     `fairseq.data` package) is constructed with the agent's arguments (agent:163-181) and `generate_decoder` (:165-582) is run
     on the reference `TransformerDecoderBase` for (prefix, max_new_tokens) cases incl. -1.  `StreamSpeechOracle.mt_greedy` must
     return the same finalized tokens.
A1.  `StreamSpeechS2STAgent.policy` and `.reset` (agent:328-347,422-770) and `OnlineFeatureExtractor.__call__/transform`
     (agent:66-98) are executed FROM THEIR OWN SOURCE (ast) against a `self` whose members are the reference's own generator /
     module objects (SequenceGenerator, CTCDecoder, CTCSequenceGenerator, CodeGenerator behind CodeHiFiGANVocoderWithDur.forward,
     the reference encoder and decoders), the SimulEval action / segment / states classes loaded from their own files.  The only
     substitutions: `convert_waveform` is the identity (16 kHz mono input; torchaudio.sox_effects does not exist in this image) and
     the checkpoint is the seeded synthetic one.  Utterances at 320 ms (plain path) and 640 ms (whole-word path, agent:540-574)
     are streamed; `OracleS2STAgent` must reproduce every action: READ / WRITE, the flags, token sequences, units, durations and
     the waveform.

Both write fixtures to tests/golden/ (mt_greedy.npz, agent_policy_<tag>.npz) that the CPU tests replay against the oracle and the
GPU tests against the engine.
"""
from __future__ import annotations

import ast
import importlib.util
import math
import os
import sys
import types
from copy import deepcopy

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_loader  # noqa: E402
from oracle.gen_golden import (FakeDict, build_reference_ctc_generators, build_reference_decoders, build_reference_encoder,  # noqa: E402
                               extract_functions, maxdiff)
from oracle.agent_oracle import OracleS2STAgent  # noqa: E402
from oracle.streamspeech_oracle import StreamSpeechOracle  # noqa: E402
from streamspeech_b200 import synth  # noqa: E402
from streamspeech_b200.config import ModelConfig, VocoderConfig  # noqa: E402
from streamspeech_b200.dictionary import Dictionary  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
REF = ref_loader.REF


def load_reference_generators():
    """fairseq.search / fairseq.sequence_generator / agent.sequence_generator, unchanged."""
    ref_loader.load_full()
    if "fairseq.data" not in sys.modules:
        fd = types.ModuleType("fairseq.data")
        fd.__path__ = [REF + "/fairseq/fairseq/data"]
        sys.modules["fairseq.data"] = fd
        du = types.ModuleType("fairseq.data.data_utils")  # only imported, never called on this path
        sys.modules["fairseq.data.data_utils"] = du
        fd.data_utils = du
    import fairseq.search as search

    sys.modules["fairseq"].search = search
    from agent.sequence_generator import SequenceGenerator

    return search, SequenceGenerator


def load_file_module(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


class RefEncoderShim(nn.Module):
    """The reference encoder (real Conv1dSubsampler / ChunkConformerEncoderLayer modules + the reference's own `_forward`)
    behind the two methods the generators call (fairseq S2T encoders: forward_torchscript, reorder_encoder_out)."""

    def __init__(self, enc):
        super().__init__()
        self.enc = enc

    def forward_torchscript(self, net_input):
        return self.enc._forward(net_input["src_tokens"], net_input["src_lengths"])

    def reorder_encoder_out(self, encoder_out, new_order):  # fairseq/models/speech_to_text/s2t_transformer.py reorder_encoder_out
        return {
            "encoder_out": [x.index_select(1, new_order) for x in encoder_out["encoder_out"]],
            "encoder_padding_mask": [x.index_select(0, new_order) for x in encoder_out["encoder_padding_mask"]],
            "encoder_embedding": [x.index_select(0, new_order) for x in encoder_out["encoder_embedding"]],
            "encoder_states": [x.index_select(1, new_order) for x in encoder_out["encoder_states"]],
            "src_tokens": [],
            "src_lengths": [],
        }


class FakeStreamSpeechModel(nn.Module):
    """The attribute surface of StreamSpeechModel the agent touches (streamspeech_model.py:182-258), made of reference modules."""

    mt_task_name = "target_unigram"

    def __init__(self, enc, mods):
        super().__init__()
        self.encoder = RefEncoderShim(enc)
        self.source_unigram_decoder = mods["source_unigram"]
        self.ctc_target_unigram_decoder = mods["ctc_target_unigram"]
        self.target_unigram_decoder = mods["mt"]
        self.synthesizer_encoder = mods["t2u"]
        self.decoder = mods["unit"]

    def max_decoder_positions(self):  # FairseqEncoderDecoderModel: self.decoder.max_positions() = max_target_positions
        return 1200

    def get_normalized_probs(self, net_output, log_probs, sample=None):
        logits = net_output[0].float()
        return F.log_softmax(logits, dim=-1) if log_probs else F.softmax(logits, dim=-1)


def build_reference_agent(cfg, sd, vsd_wn, gcmvn, segment_ms, kind="s2st"):
    """A `self` for the reference policy(): reference objects everywhere, construction as in agent:111-211,355-420
    (kind "s2tt": agent/speech_to_text.s2tt.streamspeech.agent.py:107-195,355-372)."""
    search, SequenceGenerator = load_reference_generators()
    RefCTC, RefUnitCTC = build_reference_ctc_generators()
    from agent.tts.codehifigan import CodeGenerator

    seg = load_file_module("_ref_simuleval_segments", REF + "/SimulEval/simuleval/data/segments.py")
    # agents/actions.py and states.py import `simuleval.data.segments`: register the loaded module under that name first
    for name in ("simuleval", "simuleval.data", "simuleval.agents"):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.__path__ = []
            sys.modules[name] = m
    sys.modules["simuleval.data.segments"] = seg
    act = load_file_module("simuleval.agents.actions", REF + "/SimulEval/simuleval/agents/actions.py")
    sys.modules["simuleval.agents.actions"] = act
    sts = load_file_module("simuleval.agents.states", REF + "/SimulEval/simuleval/agents/states.py")

    chunk = segment_ms // 40
    conv_chunk = (16 if chunk >= 16 else 8) if kind == "s2st" else min(chunk, 16)  # agent:404-413 / s2tt agent :359-366
    enc = build_reference_encoder(cfg, sd, chunk, conv_chunk)
    mods = build_reference_decoders(cfg, sd)
    model = FakeStreamSpeechModel(enc, mods).eval()
    tgt_dict_mt = Dictionary.synthetic(cfg.tgt_vocab)
    tgt_dict = Dictionary.units(cfg.unit_vocab - 5)
    dicts = {"tgt": tgt_dict, "source_unigram": Dictionary.synthetic(cfg.src_vocab), "ctc_target_unigram": Dictionary.synthetic(cfg.tgt_vocab),
             "target_unigram": tgt_dict_mt}

    # CodeHiFiGANVocoderWithDur (agent/tts/vocoder.py:31-60): the constructor reads files, forward is run from its own source
    gen = CodeGenerator(VocoderConfig().to_json_dict())
    gen.load_state_dict(vsd_wn, strict=True)
    gen.eval()
    gen.remove_weight_norm()
    voc_forward = extract_functions(REF + "/agent/tts/vocoder.py", "CodeHiFiGANVocoderWithDur", ["forward"],
                                    {"torch": torch, "Dict": dict})["forward"]

    class Vocoder:
        model = gen

        def __call__(self, x, dur_prediction=False):
            return voc_forward(self, x, dur_prediction)

    glb = {"torch": torch, "np": np, "math": math, "deepcopy": deepcopy, "ReadAction": act.ReadAction, "WriteAction": act.WriteAction,
           "SpeechSegment": seg.SpeechSegment, "SAMPLE_RATE": 16000, "ORG_SAMPLE_RATE": 48000,
           "convert_waveform": lambda w, sr, to_mono=True, to_sample_rate=None: (w, 16000)}
    # extract_fbank_features (fairseq/examples/speech_to_text/data_utils.py:73-98) + _get_torchaudio_fbank (audio_utils.py:236-249)
    tree = ast.parse(open(REF + "/fairseq/fairseq/data/audio/audio_utils.py").read())
    fn = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "_get_torchaudio_fbank"]
    ns = {"torch": torch, "np": np, "Optional": __import__("typing").Optional}
    exec(compile(ast.Module(body=fn, type_ignores=[]), "audio_utils.py", "exec"), ns)
    tree = ast.parse(open(REF + "/fairseq/examples/speech_to_text/data_utils.py").read())
    fn = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "extract_fbank_features"]
    ns2 = {"torch": torch, "np": np, "Optional": __import__("typing").Optional, "Path": __import__("pathlib").Path,
           "convert_waveform": glb["convert_waveform"], "_get_kaldi_fbank": lambda *a: None, "_get_torchaudio_fbank": ns["_get_torchaudio_fbank"]}
    exec(compile(ast.Module(body=fn, type_ignores=[]), "data_utils.py", "exec"), ns2)
    glb["extract_fbank_features"] = ns2["extract_fbank_features"]

    fe = extract_functions(REF + "/agent/speech_to_speech.streamspeech.agent.py", "OnlineFeatureExtractor", ["__call__", "transform"], glb)

    class FeatureExtractor:  # OnlineFeatureExtractor.__init__ (agent:46-61) with args.sample_rate = 16000
        shift_size, window_size, sample_rate, feature_dim = 10, 25, 16000, 80
        num_samples_per_shift = 160
        num_samples_per_window = 400
        len_ms_to_samples = staticmethod(lambda x: x * 16000 / 1000)
        global_cmvn = gcmvn
        device = "cpu"
        __call__ = fe["__call__"]
        transform = fe["transform"]

    if kind == "s2st":
        ag = extract_functions(REF + "/agent/speech_to_speech.streamspeech.agent.py", "StreamSpeechS2STAgent", ["policy", "reset"], glb)
    else:
        ag = extract_functions(REF + "/agent/speech_to_text.s2tt.streamspeech.agent.py", "StreamSpeechS2TTAgent", ["policy", "reset"], glb)

    class RefAgent:
        policy = ag["policy"]
        reset = ag["reset"]

        def __init__(self):
            self.device = "cpu"
            self.eos = 2
            self.states = sts.AgentStates()
            self.feature_extractor = FeatureExtractor()
            self.models = [model]
            self.dict = dicts
            inc = kind == "s2tt"  # s2tt agent :136,178: both generators keep incremental states
            self.ctc_generator = RefUnitCTC(tgt_dict, self.models, use_incremental_states=inc)
            self.asr_ctc_generator = RefCTC(dicts["source_unigram"], self.models)
            self.st_ctc_generator = RefCTC(dicts["ctc_target_unigram"], self.models)
            common = dict(beam_size=1, max_len=0, min_len=1, normalize_scores=True, len_penalty=1.0, unk_penalty=0.0, temperature=1.0,
                          match_source_len=False, no_repeat_ngram_size=0, symbols_to_strip_from_output=None)
            self.generator = SequenceGenerator(self.models, tgt_dict, max_len_a=1, max_len_b=200, search_strategy=search.BeamSearch(tgt_dict),
                                               eos=tgt_dict.eos(), **common)
            self.generator_mt = SequenceGenerator(self.models, tgt_dict_mt, max_len_a=1 if inc else 0, max_len_b=200 if inc else 100,
                                                  search_strategy=search.BeamSearch(tgt_dict_mt), eos=tgt_dict_mt.eos(),
                                                  use_incremental_states=inc, **common)
            self.vocoder = Vocoder()
            self.dur_prediction = True
            self.lagging_k1, self.lagging_k2, self.stride_n, self.stride_n2 = 0, 0, 1, 1
            self.segment_size, self.unit_per_subword = segment_ms, 15
            self.quiet, self.output_asr_translation = True, False
            self.whole_word = segment_ms >= 640
            self.reset()

        def push(self, samples, finished):  # SimulEval agents/agent.py:71-83 -> states.update_source (states.py:33-47)
            self.states.update_source(seg.SpeechSegment(content=samples, sample_rate=16000, finished=finished))

    return RefAgent(), model, seg, act


def pin_mt_greedy(cfg, sd, gcmvn, report):
    """M1: SequenceGenerator.generate_decoder of the reference on the reference MT decoder vs oracle.mt_greedy."""
    search, SequenceGenerator = load_reference_generators()
    enc = build_reference_encoder(cfg, sd, 8, 8)
    mods = build_reference_decoders(cfg, sd)
    model = FakeStreamSpeechModel(enc, mods).eval()
    d = Dictionary.synthetic(cfg.tgt_vocab)
    gen = SequenceGenerator([model], d, beam_size=1, max_len_a=0, max_len_b=100, max_len=0, min_len=1, normalize_scores=True, len_penalty=1.0,
                            unk_penalty=0.0, temperature=1.0, match_source_len=False, no_repeat_ngram_size=0,
                            search_strategy=search.BeamSearch(d), eos=d.eos(), symbols_to_strip_from_output=None, use_incremental_states=False)
    gold = np.load(os.path.join(GOLD, "decoders.npz"))
    eo = torch.from_numpy(gold["enc_out"]).unsqueeze(1)  # [T,1,256], produced by the reference encoder in gen_golden.py
    T = eo.size(0)
    enc_outs = [{"encoder_out": [eo], "encoder_padding_mask": [], "encoder_embedding": [], "encoder_states": [], "src_tokens": [], "src_lengths": []}]
    src = torch.zeros(1, 4 * T, 80)
    lens = torch.tensor([4 * T])
    orc = StreamSpeechOracle(cfg, sd, None, gcmvn, chunk_size=8)
    out = {"enc_out": gold["enc_out"]}
    cases = [(None, 3), (None, 1), (None, -1)]
    # prefixes taken from the model's own greedy output so that forced-prefix decoding continues a plausible hypothesis
    full = gen.generate_decoder(enc_outs, src, lens, {"id": 1, "net_input": {"src_tokens": src, "src_lengths": lens}}, None, None, None,
                                aux_task_name="target_unigram", max_new_tokens=-1)[0][0]["tokens"].tolist()
    body = [t for t in full if t != cfg.eos]
    cases += [(body[:2], 2), (body[:5], 1), (body[:3], -1), ([17, 256, 4099], 4), ([17, 256, 4099], -1)]
    for i, (prefix, k) in enumerate(cases):
        pt = torch.tensor([prefix], dtype=torch.long) if prefix is not None else None
        fin = gen.generate_decoder(enc_outs, src, lens, {"id": 1, "net_input": {"src_tokens": src, "src_lengths": lens}}, pt, None, None,
                                   aux_task_name="target_unigram", max_new_tokens=k)
        ref_tokens = fin[0][0]["tokens"].tolist()
        mine = orc.mt_greedy(eo, prefix, k, max_len_b=100, max_decoder_positions=1200)
        assert ref_tokens == mine, (i, prefix, k, ref_tokens, mine)
        out[f"case{i}_prefix"] = np.array(prefix if prefix is not None else [], dtype=np.int64)
        out[f"case{i}_has_prefix"] = np.array(prefix is not None)
        out[f"case{i}_max_new"] = np.array(k)
        out[f"case{i}_tokens"] = np.array(ref_tokens, dtype=np.int64)
        report[f"mt_greedy_case{i}"] = f"prefix={prefix} max_new={k} -> {len(ref_tokens)} tokens (incl. eos), oracle identical"
    out["n_cases"] = np.array(len(cases))
    np.savez_compressed(os.path.join(GOLD, "mt_greedy.npz"), **out)


def run_policy_pair(cfg, sd, vsd_wn, gcmvn, segment_ms, seconds, seed, report, tag):
    ref, model, seg, act = build_reference_agent(cfg, sd, vsd_wn, gcmvn, segment_ms)
    orc = StreamSpeechOracle(cfg, sd, vsd_wn, gcmvn)
    d = Dictionary.synthetic(cfg.tgt_vocab)
    mine = OracleS2STAgent(orc, segment_ms, is_word_start=lambda t: d[t].startswith("▁"))
    wav = synth.make_audio(seconds, seed=seed)
    n = 16 * segment_ms
    out = {"segment_ms": np.array(segment_ms), "seconds": np.array(seconds), "seed": np.array(seed)}
    kinds, worst, n_write, n_calls = [], 0.0, 0, 0
    for ci, i in enumerate(range(0, len(wav), n)):
        fin = i + n >= len(wav)
        chunk = wav[i:i + n].tolist()
        ref.push(chunk, fin)
        mine.push(chunk, finished=fin)
        a_ref = ref.policy()
        a = mine.policy()
        n_calls += 1
        if a_ref.is_read():
            assert a.kind == "read", (tag, ci)
            kinds.append(0)
            continue
        assert a.kind == "write", (tag, ci)
        kinds.append(1)
        content = a_ref.content.content
        assert a_ref.finished == a.finished and a_ref.content.finished == a.seg_finished, (tag, ci)
        assert len(content) == len(a.wav), (tag, ci, len(content), len(a.wav))
        if len(content):
            worst = max(worst, float(np.abs(np.array(content) - np.array(a.wav)).max()))
            n_write += 1
        out[f"call{ci}_wav"] = np.array(content, dtype=np.float32)
        out[f"call{ci}_flags"] = np.array([a_ref.finished, a_ref.content.finished])
        for k in ("asr_tokens", "st_tokens", "mt_tokens", "units", "dur"):
            out[f"call{ci}_{k}"] = np.array(a.trace.get(k, []), dtype=np.int64)
        # the reference keeps its state on `self`; after a finishing WRITE it has been reset
        if not fin:
            assert ref.tgt_subwords_indices.view(-1).tolist() == mine.tgt_subwords_indices, (tag, ci)
            assert ref.unit == mine.unit, (tag, ci)
            assert ref.prev_output_tokens_mt.view(-1).tolist() == mine.prev_output_tokens_mt, (tag, ci)
    assert worst < 1e-5, (tag, worst)
    assert n_write >= 1, (tag, "no WRITE action in the fixture utterance")
    out["kinds"] = np.array(kinds)
    report[f"policy_{tag}"] = f"{n_calls} calls, {n_write} non-empty WRITEs, wav max-abs {worst:.2e}, kinds {''.join(map(str, kinds))}"
    return out


def run_s2tt_pair(cfg, sd, gcmvn, segment_ms, seconds, seed, report, tag):
    """S2TT agent (incremental decoder states across policy() calls, N12): reference policy() vs OracleS2TTAgent."""
    from oracle.agent_oracle import OracleS2TTAgent

    vsd_wn = synth.make_vocoder_state_dict(cfg.vocoder, 1, weight_norm=True)
    ref, model, seg, act = build_reference_agent(cfg, sd, vsd_wn, gcmvn, segment_ms, kind="s2tt")
    orc = StreamSpeechOracle(cfg, sd, None, gcmvn)
    d = Dictionary.synthetic(cfg.tgt_vocab)
    mine = OracleS2TTAgent(orc, segment_ms, symbols=lambda t: d[t])
    wav = synth.make_audio(seconds, seed=seed)
    n = 16 * segment_ms
    out = {"segment_ms": np.array(segment_ms), "seconds": np.array(seconds), "seed": np.array(seed)}
    kinds, texts = [], []
    for ci, i in enumerate(range(0, len(wav), n)):
        fin = i + n >= len(wav)
        chunk = wav[i:i + n].tolist()
        ref.push(chunk, fin)
        mine.push(chunk, finished=fin)
        a_ref = ref.policy()
        a = mine.policy()
        if a_ref.is_read():
            assert a.kind == "read", (tag, ci)
            kinds.append(0)
            texts.append("")
            continue
        assert a.kind == "write", (tag, ci)
        assert a_ref.content == a.wav and a_ref.finished == a.finished, (tag, ci, a_ref.content, a.wav)
        kinds.append(1)
        texts.append(a_ref.content)
        out[f"call{ci}_mt_tokens"] = np.array(a.trace.get("mt_tokens", []), dtype=np.int64)
        out[f"call{ci}_finished"] = np.array(a_ref.finished)
    assert sum(kinds) >= 3, (tag, kinds)
    out["kinds"] = np.array(kinds)
    out["texts"] = np.array(texts)
    report[f"policy_{tag}"] = f"{len(kinds)} calls, kinds {''.join(map(str, kinds))}, final hypothesis {len(out[f'call{len(kinds) - 1}_mt_tokens'])} tokens"
    return out


def main():
    torch.set_grad_enabled(False)
    cfg = ModelConfig()
    sd = synth.make_model_state_dict(cfg, 0)
    vsd_wn = synth.make_vocoder_state_dict(cfg.vocoder, 1, weight_norm=True)
    gcmvn = synth.make_gcmvn(cfg)
    report = {}
    pin_mt_greedy(cfg, sd, gcmvn, report)
    # one file per utterance keeps every fixture file under 1 MB
    for tag, seg_ms, seconds, seed in (("c320", 320, 3.2, 1234), ("c640", 640, 3.84, 1234)):
        r = run_policy_pair(cfg, sd, vsd_wn, gcmvn, seg_ms, seconds, seed, report, tag)
        np.savez_compressed(os.path.join(GOLD, f"agent_policy_{tag}.npz"), **{f"{tag}_{k}": v for k, v in r.items()})
    r = run_s2tt_pair(cfg, sd, gcmvn, 320, 2.56, 1234, report, "s2tt320")
    np.savez_compressed(os.path.join(GOLD, "agent_policy_s2tt320.npz"), **{f"s2tt320_{k}": v for k, v in r.items()})
    for k, v in report.items():
        print(f"{k:28s} {v}")


if __name__ == "__main__":
    main()
