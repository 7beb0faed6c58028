"""CPU: the GPT restatement against HF transformers.GPT2Model (the arithmetic-equivalent stand-in for the
un-vendored vLLM GPT2Block, SURVEY.md §8c), plus the loop semantics of SURVEY App. A.2-A.4."""
import os

import numpy as np
import pytest
import torch

from oracle import xtts_oracle as O
from conftest import text_ids


@pytest.fixture(scope="module")
def orc(dims_small, state_small):
    return O.GPTOracle(state_small[0], state_small[1], dims_small)


def test_blocks_match_hf_gpt2(orc, dims_small, state_small, speakers_small):
    from transformers import GPT2Config, GPT2Model
    g = dims_small.gpt
    cfg = GPT2Config(vocab_size=8, n_positions=512, n_embd=g.hidden, n_layer=g.layers, n_head=g.heads, n_inner=g.ff,
                     activation_function="gelu_new", layer_norm_epsilon=g.ln_eps, resid_pdrop=0.0, embd_pdrop=0.0,
                     attn_pdrop=0.0)
    m = GPT2Model(cfg).eval()
    sd = m.state_dict()
    for k in list(sd):
        if k.startswith("h.") or k.startswith("ln_f"):
            sd[k] = state_small[0]["gpt." + k]
    sd["wpe.weight"] = torch.zeros_like(sd["wpe.weight"])
    m.load_state_dict(sd)
    rows = orc.prompt_rows(speakers_small[0][0], text_ids(dims_small, 12, 1))
    with torch.no_grad():
        ref = m(inputs_embeds=rows[None]).last_hidden_state[0]
        mine, _ = orc.forward_rows(rows)
    np.testing.assert_allclose(mine.numpy(), ref.numpy(), atol=2e-5, rtol=0)


def test_incremental_equals_second_pass(orc, dims_small, speakers_small):
    """decode-time hidden states == the reference's 2nd prefill pass (XTTSv2.py:617-687), SURVEY A.4."""
    g = dims_small.gpt
    sp = O.SamplingParams(temperature=0.0, max_tokens=16, stop_token=g.stop_audio_token)
    ids = text_ids(dims_small, 9, 2)
    toks, lats, lg = orc.generate(speakers_small[1][0], ids, sp, return_logits=True)
    assert len(toks) == 16 and lats.shape == (16, g.hidden)
    lg2, lats2 = orc.teacher_forced(speakers_small[1][0], ids, toks)
    np.testing.assert_allclose(lg.numpy(), lg2.numpy(), atol=2e-5, rtol=0)
    np.testing.assert_allclose(lats.numpy(), lats2.numpy(), atol=2e-5, rtol=0)


def test_stop_token_is_kept_and_ends_generation(orc, dims_small, speakers_small):
    g = dims_small.gpt
    sp = O.SamplingParams(temperature=0.0, max_tokens=12, stop_token=g.stop_audio_token)
    ids = text_ids(dims_small, 5, 3)
    toks, _ = orc.generate(speakers_small[0][0], ids, sp)
    sp2 = O.SamplingParams(temperature=0.0, max_tokens=12, stop_token=toks[4])
    toks2, lats2 = orc.generate(speakers_small[0][0], ids, sp2)
    assert toks2 == toks[:5] and lats2.shape[0] == 5           # ids include the stop token; T = len(ids)


def test_repetition_penalty_semantics():
    z = torch.tensor([2.0, -1.0, 0.5, 3.0, -4.0])
    out = O.apply_repetition_penalty(z.clone(), {0, 1, 4}, 5.0)
    np.testing.assert_allclose(out.numpy(), [0.4, -5.0, 0.5, 3.0, -20.0])
    assert torch.equal(O.apply_repetition_penalty(z.clone(), {0}, 1.0), z)


def test_topk_topp_mask():
    z = torch.log(torch.tensor([0.5, 0.2, 0.15, 0.1, 0.05]))
    m = O.topk_topp_mask(z.clone(), top_k=4, top_p=0.85)
    # top-k drops 0.05; top-p on {0.1,0.15,0.2,0.5}/0.95: ascending cum = .105,.263,.474,1 -> drop <= .15
    assert torch.isinf(m[4]) and torch.isinf(m[3]) and not torch.isinf(m[:3]).any()
    m = O.topk_topp_mask(z.clone(), top_k=0, top_p=1.0)
    assert not torch.isinf(m).any()


def test_philox_known_answer():
    """Random123 KAT for philox4x32-10: counter=key=0 and the all-ones vector."""
    r = O.philox4x32((0, 0, 0, 0), (0, 0))
    assert [hex(int(x)) for x in r] == ["0x6627e8d5", "0xe169c58d", "0xbc57ac4c", "0x9b00dbd8"]
    r = O.philox4x32((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2)
    assert [hex(int(x)) for x in r] == ["0x408f276d", "0x41c83b0e", "0xa20bc7c6", "0x6d5451fd"]


def test_exp_noise_is_exp1():
    e = np.concatenate([O.exp_noise(5, s, 0, 1024) for s in range(40)])
    assert (e > 0).all() and np.isfinite(e).all()
    assert abs(e.mean() - 1.0) < 0.03 and abs(e.var() - 1.0) < 0.08


def test_sampling_distribution_matches_softmax():
    """argmax(p / Exp(1)) samples from p (what vLLM's q.exponential_() trick does)."""
    z = torch.log(torch.tensor([0.6, 0.3, 0.1]))
    sp = O.SamplingParams(temperature=1.0, top_p=1.0, top_k=0, repetition_penalty=1.0, seed=11)
    n = 3000
    c = np.bincount([O.sample_token(z.clone(), set(), sp, s, 0) for s in range(n)], minlength=3) / n
    assert np.abs(c - [0.6, 0.3, 0.1]).max() < 0.03


def _installed_vllm_topk_topp():
    """`apply_top_k_top_p_pytorch` lifted out of the INSTALLED vLLM (0.22, v1 sampler) by source — importing the package
    needs libcuda.  It is a stand-in for the pinned, un-vendored vLLM 0.6.4.post1 sampler (SURVEY.md §8c): same published
    algorithm (ascending sort, k-th value threshold, cumulative-softmax <= 1-p with the maximum always kept)."""
    import ast
    import importlib.util
    spec = importlib.util.find_spec("vllm")
    if spec is None or not spec.submodule_search_locations:
        return None
    path = os.path.join(list(spec.submodule_search_locations)[0], "v1", "sample", "ops", "topk_topp_sampler.py")
    if not os.path.exists(path):
        return None
    tree = ast.parse(open(path).read())
    fns = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in ("apply_top_k_top_p_pytorch", "apply_top_k_only")]
    if len(fns) != 2:
        return None
    ns = {"torch": torch}
    exec(compile(ast.Module(body=fns, type_ignores=[]), path, "exec"), ns)
    return ns["apply_top_k_top_p_pytorch"]


def test_topk_topp_mask_matches_installed_vllm_sampler():
    fn = _installed_vllm_topk_topp()
    if fn is None:
        pytest.skip("no installed vLLM sampler source to compare with")
    g = torch.Generator().manual_seed(3)
    for trial in range(40):
        V = [130, 1026, 7][trial % 3]
        z = torch.randn(V, generator=g) * (1.0 + trial % 5)
        if trial % 4 == 0:
            z[torch.randint(0, V, (V // 3,), generator=g)] = float(z[0])            # ties at and around the thresholds
        k = [1, 5, 50, V - 1, V][trial % 5]
        p = [0.05, 0.5, 0.85, 0.999][trial % 4]
        want = fn(z.clone()[None], torch.tensor([min(k, V)]), torch.tensor([p], dtype=torch.float32))[0]
        got = O.topk_topp_mask(z.clone(), k, p)
        assert torch.equal(torch.isinf(got), torch.isinf(want)), (trial, V, k, p)
        assert torch.equal(got[~torch.isinf(got)], want[~torch.isinf(want)])


def _reference_penalizer():
    """`LogitsRepetitionPenalizer` lifted by source out of the reference's hijack.py (the module itself imports vLLM 0.6.4)."""
    import ast
    from oracle import ref_import
    path = os.path.join(ref_import.REF_SRC, "auralis", "models", "xttsv2", "components", "vllm", "hijack.py")
    if not os.path.exists(path):
        return None
    tree = ast.parse(open(path).read())
    cls = [n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "LogitsRepetitionPenalizer"]
    from typing import List
    ns = {"torch": torch, "List": List}
    exec(compile(ast.Module(body=cls, type_ignores=[]), path, "exec"), ns)
    return ns["LogitsRepetitionPenalizer"]


def test_repetition_penalty_matches_the_reference_class(dims_small):
    """hijack.py:49-88 — the reference's OWN penaliser, run as-is on the prompt the reference builds
    (`[1]*(32+Lt)+[start]`, vllm_mm_gpt.py:325) plus a generated history with repeats.  What it changed is stored in
    tests/golden/oracle_gpt_reference.npz (tests/reference_records.py)."""
    from reference_records import Records
    rec = Records("oracle_gpt_reference")

    def reference(prompt, gen, z, p):
        want = _reference_penalizer()(p)(prompt, gen, z.clone())
        changed = torch.nonzero(want != z).reshape(-1)
        return changed, want[changed]
    g = dims_small.gpt
    rng = np.random.RandomState(4)
    for trial in range(20):
        V = g.n_audio_tokens
        z = torch.from_numpy(rng.randn(V).astype(np.float32) * 3)
        n_text = int(rng.randint(3, 20))
        prompt = [1] * (g.n_cond_latents + n_text) + [g.start_audio_token]
        gen = rng.randint(0, V, size=int(rng.randint(0, 30))).tolist()
        gen = gen + gen[:3]                                              # repeats must be penalised once
        p = [5.0, 1.0, 2.5, 0.5][trial % 4]
        changed, values = rec(f"repetition_penalty[{trial}]", lambda: reference(prompt, gen, z, p))
        want = z.clone()
        want[torch.from_numpy(changed)] = torch.from_numpy(values)
        seen = O.prompt_seen_set(g) | set(gen)
        got = O.apply_repetition_penalty(z.clone(), seen, p)
        assert torch.equal(got, want), (trial, p)


def test_batched_decode_equals_per_sequence_decode():
    """oracle.generate_batched (the CPU arm of bench.py decodes B chunks per step, like a batched deployment of the reference
    would) against the per-sequence `generate`: same greedy tokens, latents and logits to fp32 rounding, for prompts of
    different lengths and chunks that stop at different steps."""
    import numpy as np
    import torch
    from auralis_b200.config import XTTSDims
    from auralis_b200.weights import synth_state
    from oracle import xtts_oracle as O
    dims = XTTSDims.small()
    gs, cs = synth_state(dims, 1234)
    orc = O.GPTOracle(gs, cs, dims)
    g = torch.Generator().manual_seed(3)
    conds = [torch.randn(dims.gpt.n_cond_latents, dims.gpt.hidden, generator=g) for _ in range(4)]
    ids = [[0] + list(range(5, 5 + n)) + [1] for n in (6, 19, 11, 3)]
    sp = O.SamplingParams(temperature=0.0, repetition_penalty=5.0, max_tokens=14, stop_token=dims.gpt.stop_audio_token)
    toks, lats, lgs = orc.generate_batched(conds, ids, sp, return_logits=True)
    for b in range(4):
        et, el, elg = orc.generate(conds[b], ids[b], sp, return_logits=True)
        assert toks[b] == et
        np.testing.assert_allclose(lats[b].numpy(), el.numpy(), atol=2e-4)
        np.testing.assert_allclose(lgs[b].numpy(), elg.numpy(), atol=2e-4)
    # seeded sampling through the shared Philox stream: token-for-token (seq_seed = row index)
    sp2 = O.SamplingParams(temperature=0.75, top_p=0.85, top_k=50, repetition_penalty=5.0, max_tokens=10,
                           stop_token=dims.gpt.stop_audio_token, seed=5)
    toks2, _ = orc.generate_batched(conds, ids, sp2)
    for b in range(4):
        assert toks2[b] == orc.generate(conds[b], ids[b], sp2, seq_seed=b)[0]
