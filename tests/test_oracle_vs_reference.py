"""CPU: the oracle restatement against what the REFERENCE's own modules (imported unmodified by oracle/ref_import.py)
returned on inputs OTHER than tests/golden/{vocoder,conditioning}_*.npz — ragged lengths, a one-frame chunk, several
speakers, reference audio that is cut into more than one conditioning chunk.  The reference's values are stored in
tests/golden/oracle_vs_reference.npz (tests/reference_records.py: XTTS_RECORD_REFERENCE=1 re-runs the reference)."""
import importlib.util
import os

import numpy as np
import pytest
import torch

from auralis_b200.config import XTTSDims
from oracle import ref_import
from oracle import xtts_oracle as O
from reference_records import Records, sample

rec = Records("oracle_vs_reference")


def _golden_tools():
    spec = importlib.util.spec_from_file_location(
        "make_golden", os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "make_golden.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _ref():
    return ref_import.load()


@pytest.mark.parametrize("T", [1, 2, 7, 33])
def test_vocoder_live(dims_small, state_small, T):
    def reference(lat, gv):
        ref = _ref()
        hd = _golden_tools().ref_vocoder(ref, dims_small, state_small[1])
        with torch.no_grad():
            return ref.HifiDecoder.forward(hd, lat[None], g=gv.reshape(1, -1, 1)).reshape(-1)
    g = torch.Generator().manual_seed(1000 + T)
    for spk in range(2):
        lat = torch.randn(T, dims_small.voc.in_dim, generator=g)
        gv = torch.nn.functional.normalize(torch.randn(dims_small.voc.d_vector, generator=g), dim=0)
        shape, want = rec(f"vocoder[T={T},spk={spk}]", lambda: sample(reference(lat, gv)))
        got = O.vocoder(lat, gv, state_small[1], dims_small)
        assert got.shape == shape == (dims_small.voc.n_samples(T),)
        np.testing.assert_allclose(sample(got)[1], want, atol=2e-6, rtol=0)


@pytest.mark.parametrize("seconds,f0", [(0.4, 95.0), (1.3, 180.0)])
def test_conditioning_live(dims_small, state_small, seconds, f0):
    cs, dims = state_small[1], dims_small
    wav22 = O.synthetic_reference_wav(seconds, 22050, f0, 21)
    mel, h, want = rec(f"conditioning[{seconds},{f0}]", lambda: [sample(x[0]) for x in _reference_conditioning(wav22, cs, dims)])
    got_mel = O.mel_cloning(wav22, cs["mel_stats"], dims.cond.n_mels)
    got_h = O.cond_encoder(got_mel, cs, dims)
    got = O.perceiver(got_h.t(), cs, dims)
    for x, (shape, s), atol in ((got_mel, mel, 2e-5), (got_h, h, 2e-5), (got, want, 5e-5)):
        assert tuple(x.shape) == shape
        np.testing.assert_allclose(sample(x)[1], s, atol=atol, rtol=0)


def _reference_conditioning(wav22, cs, dims):
    ref = _ref()
    mel = ref.wav_to_mel_cloning(wav22[None], mel_norms=cs["mel_stats"], n_fft=2048, hop_length=256, win_length=1024, power=2,
                                 normalized=False, sample_rate=22050, f_min=0, f_max=8000, n_mels=80)
    ce = ref.ConditioningEncoder(dims.cond.n_mels, dims.gpt.hidden, attn_blocks=dims.cond.cond_blocks, num_attn_heads=dims.gpt.heads)
    ce.load_state_dict({k[len("conditioning_encoder."):]: t for k, t in cs.items() if k.startswith("conditioning_encoder.")})
    pr = ref.PerceiverResampler(dim=dims.gpt.hidden, depth=dims.cond.perceiver_depth, dim_context=dims.gpt.hidden,
                                num_latents=dims.gpt.n_cond_latents, dim_head=dims.cond.perceiver_dim_head,
                                heads=dims.cond.perceiver_heads, ff_mult=dims.cond.perceiver_ff_mult, use_flash_attn=False)
    pr.load_state_dict({k[len("conditioning_perceiver."):]: t for k, t in cs.items() if k.startswith("conditioning_perceiver.")})
    with torch.no_grad():
        h = ce(mel)
        return mel, h, pr(h.permute(0, 2, 1))


def test_speaker_encoder_live(dims_small, state_small):
    cs, dims = state_small[1], dims_small
    for seconds, f0 in ((0.35, 110.0), (0.9, 210.0)):
        wav16 = O.synthetic_reference_wav(seconds, 16000, f0, 5)
        want = rec(f"speaker_encoder[{seconds},{f0}]", lambda: _reference_speaker_encoder(cs, dims)(wav16[None].clone(), l2_norm=True)[0])
        np.testing.assert_allclose(O.speaker_embedding(wav16, cs, dims).numpy(), want, atol=2e-6, rtol=0)


def _reference_speaker_encoder(cs, dims):
    se = _ref().ResNetSpeakerEncoder(input_dim=dims.cond.spk_mels, proj_dim=dims.cond.spk_proj, layers=list(dims.cond.spk_layers),
                                  num_filters=list(dims.cond.spk_filters), log_input=True, use_torch_spec=True,
                                  audio_config={"fft_size": 512, "win_length": 400, "hop_length": 160, "sample_rate": 16000,
                                                "preemphasis": 0.97, "num_mels": 64})
    pre = "hifigan_decoder.speaker_encoder."
    se.load_state_dict({k[len(pre):]: t for k, t in cs.items() if k.startswith(pre)})
    se.eval()
    return torch.no_grad()(se.forward)


def _lift_methods(path, cls_name, names):
    """Methods of a reference class lifted by source into plain functions (the module itself imports vLLM 0.6.4)."""
    import ast
    tree = ast.parse(open(path).read())
    cls = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == cls_name)
    fns = [n for n in cls.body if isinstance(n, (ast.FunctionDef, ast.AsyncFunctionDef)) and n.name in names]
    assert len(fns) == len(names)
    return fns


COND_LATENT_CASES = ((2.6, 30, 1), (2.6, 2, 1), (1.2, 30, 4), (2.2, 30, 1))     # 2.2 s / 1 s: last piece 0.2 s is dropped


def test_gpt_cond_latents_chunking_live(dims_small, state_small):
    """XTTSv2Engine.get_gpt_cond_latents (XTTSv2.py:349-407) run AS WRITTEN — truncation to `length` seconds, `chunk_length`
    pieces, pieces under 0.33 s dropped, mean over pieces — on the reference's own encoder modules, against the oracle."""
    cs, dims = state_small[1], dims_small
    wants = rec("gpt_cond_latents", lambda: [sample(w) for w in _reference_gpt_cond_latents(cs, dims)])
    for (seconds, length, chunk), (shape, want) in zip(COND_LATENT_CASES, wants, strict=True):
        wav = O.synthetic_reference_wav(seconds, 22050, 140.0, 31)
        got = O.gpt_cond_latents(wav, cs, dims, length=length, chunk_length=chunk)
        assert got.shape == shape == (dims.gpt.n_cond_latents, dims.gpt.hidden)
        np.testing.assert_allclose(sample(got)[1], want, atol=5e-5, rtol=0)


def _reference_gpt_cond_latents(cs, dims):
    import ast
    import types
    from typing import Optional
    import torchaudio
    ref = _ref()
    path = os.path.join(ref_import.REF_SRC, "auralis", "models", "xttsv2", "XTTSv2.py")
    fns = _lift_methods(path, "XTTSv2Engine", ("get_gpt_cond_latents", "get_style_emb"))
    ns = {"torch": torch, "torchaudio": torchaudio, "wav_to_mel_cloning": ref.wav_to_mel_cloning, "Optional": Optional}
    exec(compile(ast.Module(body=fns, type_ignores=[]), path, "exec"), ns)
    ce = ref.ConditioningEncoder(dims.cond.n_mels, dims.gpt.hidden, attn_blocks=dims.cond.cond_blocks, num_attn_heads=dims.gpt.heads)
    ce.load_state_dict({k[len("conditioning_encoder."):]: t for k, t in cs.items() if k.startswith("conditioning_encoder.")})
    pr = ref.PerceiverResampler(dim=dims.gpt.hidden, depth=dims.cond.perceiver_depth, dim_context=dims.gpt.hidden,
                                num_latents=dims.gpt.n_cond_latents, dim_head=dims.cond.perceiver_dim_head,
                                heads=dims.cond.perceiver_heads, ff_mult=dims.cond.perceiver_ff_mult, use_flash_attn=False)
    pr.load_state_dict({k[len("conditioning_perceiver."):]: t for k, t in cs.items() if k.startswith("conditioning_perceiver.")})
    me = types.SimpleNamespace(gpt_config=types.SimpleNamespace(use_perceiver_resampler=True), mel_stats=cs["mel_stats"],
                               device=torch.device("cpu"), conditioning_encoder=ce, conditioning_perceiver=pr)
    me.get_style_emb = lambda mel, rl=False: ns["get_style_emb"](me, mel, rl)
    wants = []
    for seconds, length, chunk in COND_LATENT_CASES:
        wav = O.synthetic_reference_wav(seconds, 22050, 140.0, 31)
        with torch.no_grad():
            wants.append(ns["get_gpt_cond_latents"](me, wav[None], 22050, length=length, chunk_length=chunk)[0])      # [32, H]
    return wants


def test_prompt_construction_live(dims_small, state_small, speakers_small):
    """Rows a1-a2 of the hot path: XTTSv2Engine.prepare_text_tokens_async + _merge_conditioning (XTTSv2.py:506-543,330-347)
    and LearnedPositionEmbeddings (vllm_mm_gpt.py:165-214), lifted by source and executed as written with the synthetic
    embedding tables, against the oracle's prompt rows ([cond latents ; text_emb + text_pos] — the audio-bos row is added by
    the GPT wrapper, vllm_mm_gpt.py:806-813)."""
    gs, cs = state_small
    g = dims_small.gpt
    orc = O.GPTOracle(gs, cs, dims_small)
    cond = speakers_small[0][0]                                        # [32, H]
    for n_chunks, seed in ((1, 0), (3, 1)):
        rng = np.random.RandomState(seed)
        chunks = [rng.randint(2, g.n_text_tokens, size=int(rng.randint(1, g.max_text_tokens - 1))).tolist() for _ in range(n_chunks)]
        fake_lens, merged = rec(f"prompts[{n_chunks},{seed}]",
                                lambda: (lambda f, m: (f, [sample(x) for x in m]))(*_reference_prompts(cs, g, chunks, cond)))
        assert fake_lens == [len(c) + 2 for c in chunks]                  # placeholder ids [1]*(L+2) (App. A.2)
        for c, m in zip(chunks, merged, strict=True):
            ids = [0] + c + [1]
            rows = orc.prompt_rows(cond, ids)
            assert rows.shape[0] == g.n_cond_latents + len(ids) + 1
            assert tuple(rows[:-1].shape) == m[0]
            np.testing.assert_allclose(sample(rows[:-1])[1], m[1], atol=1e-6, rtol=0)


def _reference_prompts(cs, g, chunks, cond):
    """-> (lengths of the placeholder id lists, merged prompt embeddings) of the lifted reference methods"""
    import ast
    import asyncio
    import logging
    import random
    import types
    from typing import List, Tuple, Union
    base = os.path.join(ref_import.REF_SRC, "auralis", "models", "xttsv2")
    fns = _lift_methods(os.path.join(base, "XTTSv2.py"), "XTTSv2Engine", ("prepare_text_tokens_async", "_merge_conditioning"))
    tree = ast.parse(open(os.path.join(base, "components", "vllm_mm_gpt.py")).read())
    lpe = [n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "LearnedPositionEmbeddings"]
    ns = {"torch": torch, "nn": torch.nn, "random": random, "List": List, "Tuple": Tuple, "Union": Union}
    exec(compile(ast.Module(body=lpe + fns, type_ignores=[]), "lifted", "exec"), ns)
    text_emb = torch.nn.Embedding(g.n_text_tokens, g.hidden)
    text_emb.weight.data.copy_(cs["text_embedding.weight"])
    text_pos = ns["LearnedPositionEmbeddings"](g.max_text_tokens + 2, g.hidden)
    text_pos.emb.weight.data.copy_(cs["text_pos_embedding.emb.weight"])
    tok = types.SimpleNamespace(bos_token_id=0, eos_token_id=1, batch_encode_with_split=lambda text, lang: [list(c) for c in chunks])
    me = types.SimpleNamespace(tokenizer=tok, text_embedding=text_emb, text_pos_embedding=text_pos, logger=logging.getLogger("x"),
                               llm_engine=types.SimpleNamespace(engine=types.SimpleNamespace(model_config=types.SimpleNamespace(dtype=torch.float32))))

    async def go():
        fake, embeds = await ns["prepare_text_tokens_async"](me, "ignored", "en", split_text=True)
        merged = await ns["_merge_conditioning"](me, embeds, cond[None])
        return fake, merged
    with torch.no_grad():
        fake, merged = asyncio.new_event_loop().run_until_complete(go())
    return [len(f) for f in fake], list(merged)


def test_gpt_wrapper_embedding_and_splice_live(dims_small, state_small, speakers_small):
    """Row a5: the embedding / conditioning-splice part of the reference's GPT2Model.forward (vllm_mm_gpt.py:768-833) lifted by
    source and executed as written with zero transformer layers: prefill rows = [prefix ; wte[start] + wpe[0]], decode row k =
    wte[t_k] + wpe[k], and a mixed prefill + decode batch — against the oracle's prompt_rows / audio_row."""
    gs, cs = state_small
    g = dims_small.gpt
    orc = O.GPTOracle(gs, cs, dims_small)
    cond = speakers_small[1][0]
    ids = [0, 17, 5, 44, 9, 1]
    rows = orc.prompt_rows(cond, ids)
    prefix = rows[:-1]                                                         # what _merge_conditioning hands to vLLM
    decodes = ((3, 1), (g.start_audio_token - 1, 7), (60, g.max_audio_tokens))
    got = rec("gpt2_forward", lambda: _reference_gpt2_forward(gs, g, prefix, decodes))
    assert got["prefill"][0] == tuple(rows.shape)
    np.testing.assert_allclose(got["prefill"][1], sample(rows)[1], atol=1e-6, rtol=0)
    for (tok, k), row in zip(decodes, got["decode"], strict=True):
        np.testing.assert_allclose(row[0], orc.audio_row(tok, k).numpy(), atol=1e-6, rtol=0)
    # one sequence decoding (row first), another one starting in the same step (spliced after it)
    want = torch.cat([orc.audio_row(9, 4)[None], rows], dim=0)
    assert got["mixed"][0] == tuple(want.shape)
    np.testing.assert_allclose(got["mixed"][1], sample(want)[1], atol=1e-6, rtol=0)


def _reference_gpt2_forward(gs, g, prefix, decodes):
    import __future__
    import ast
    import random
    import types
    path = os.path.join(ref_import.REF_SRC, "auralis", "models", "xttsv2", "components", "vllm_mm_gpt.py")
    tree = ast.parse(open(path).read())
    lpe = [n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "LearnedPositionEmbeddings"]
    fns = _lift_methods(path, "GPT2Model", ("forward", "_insert_conditioning_into_hidden_states"))
    for f in fns:
        f.decorator_list = []
    ns = {"torch": torch, "nn": torch.nn, "random": random,
          "get_pp_group": lambda: types.SimpleNamespace(is_first_rank=True, is_last_rank=True)}
    exec(compile(ast.Module(body=lpe + fns, type_ignores=[]), "lifted", "exec", flags=__future__.annotations.compiler_flag), ns)
    wte = torch.nn.Embedding(g.n_audio_tokens, g.hidden)
    wte.weight.data.copy_(gs["gpt.wte.weight"])
    wpe = ns["LearnedPositionEmbeddings"](g.max_audio_tokens + 3, g.hidden)
    wpe.emb.weight.data.copy_(gs["gpt.wpe.emb.weight"])
    me = types.SimpleNamespace(wte=wte, wpe=wpe, audio_start_generation_token=g.start_audio_token, embed_dim=g.hidden,
                               start_layer=0, end_layer=0, h=[], ln_f=lambda x: x,
                               _insert_conditioning_into_hidden_states=ns["_insert_conditioning_into_hidden_states"])
    empty = torch.empty(0, dtype=torch.long)
    with torch.no_grad():
        return {"prefill": sample(ns["forward"](me, empty, empty, [], None, None, input_embeds=[prefix[None]],
                                                starting_sequence_start_ids=[0], is_logit_only=torch.tensor([False]))),
                "decode": [ns["forward"](me, torch.tensor([tok]), torch.tensor([k]), [], None, None) for tok, k in decodes],
                "mixed": sample(ns["forward"](me, torch.tensor([9]), torch.tensor([4]), [], None, None, input_embeds=[prefix[None]],
                                              starting_sequence_start_ids=[1], is_logit_only=torch.tensor([False])))}


def test_placeholder_prompt_and_penalty_seed_live(dims_small):
    """Row a3: input_processor_for_xtts2_gpt (vllm_mm_gpt.py:296-334) executed as written — the prompt vLLM sees is
    [1]*(32+Lt) + [start_audio_token], so the repetition penaliser's prompt set is {1, start} (App. B.7), which is what the
    oracle and the CUDA sampler seed their 'seen' set with."""
    g = dims_small.gpt
    for n_text in (3, 17):
        ids = rec(f"placeholder_prompt[{n_text}]", lambda: _reference_placeholder_prompt(g, n_text))
        assert ids == [1] * (g.n_cond_latents + n_text) + [g.start_audio_token]
        assert set(ids) == O.prompt_seen_set(g)


def _reference_placeholder_prompt(g, n_text):
    import __future__
    import ast
    import types
    path = os.path.join(ref_import.REF_SRC, "auralis", "models", "xttsv2", "components", "vllm_mm_gpt.py")
    tree = ast.parse(open(path).read())
    fn = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "input_processor_for_xtts2_gpt"]
    ns = {"token_inputs": lambda **kw: kw, "PlaceholderRange": lambda **kw: kw}
    exec(compile(ast.Module(body=fn, type_ignores=[]), "lifted", "exec", flags=__future__.annotations.compiler_flag), ns)
    ctx = types.SimpleNamespace(model_config=types.SimpleNamespace(hf_config=types.SimpleNamespace(start_audio_token=g.start_audio_token)))
    embeds = torch.zeros(g.n_cond_latents + n_text, g.hidden)
    out = ns["input_processor_for_xtts2_gpt"](ctx, {"multi_modal_data": {"audio": {"embeds": embeds}}, "prompt_token_ids": [1] * n_text})
    return list(out["prompt_token_ids"])
