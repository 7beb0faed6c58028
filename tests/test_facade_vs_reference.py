"""CPU: the public façade (`auralis_b200.TTS` / `TTSRequest` / `TTSOutput`) against what the REFERENCE's own classes
(`auralis.core.tts.TTS` etc., imported unmodified by oracle/ref_facade.py) returned, stored in
tests/golden/facade_vs_reference.npz (tests/reference_records.py).  Both are driven by the same fake engine
— per chunk one waveform whose values encode (request text length, chunk index), earlier chunks finishing LATER — and must
return the same audio in the same order for: one-shot generation, streaming, several chunks, the 100 000-character request
split (`split_requests`), a prepared speaker (`prepare_for_streaming_generation`), the async API, and a failing chunk."""
import asyncio
import os

import numpy as np
import pytest

import auralis_b200 as ours
from oracle import ref_import
from reference_records import Records, sample

pytestmark = pytest.mark.timeout(120)
rec = Records("facade_vs_reference")


def make_engine(ns_output, cond_config, fail_at=None):
    """A fake engine speaking the plugin API (`models/base.py:57-224`); `ns_output` is the TTSOutput class of the side under
    test, so each façade receives its own output type."""

    class Engine:
        def __init__(self):
            self.cond_calls = 0

        @property
        def conditioning_config(self):
            return cond_config

        async def get_audio_conditioning(self, speaker_files, *a, **k):
            self.cond_calls += 1
            return np.full((1, 32, 8), 0.5, np.float32), np.full((1, 4, 1), 0.25, np.float32)

        async def get_generation_context(self, request, gpt_cond_latent=None, speaker_embeddings=None):
            if gpt_cond_latent is None:
                gpt_cond_latent, speaker_embeddings = await self.get_audio_conditioning(request.speaker_files)
            n = max(1, len(request.text) // 10)

            async def gen(i):
                await asyncio.sleep(0.003 * (n - i))
                if fail_at == i:
                    raise RuntimeError(f"chunk {i} exploded")
                yield (len(request.text), i)
            return [gen(i) for i in range(n)], [f"{request.request_id}_{i}" for i in range(n)], speaker_embeddings, [gpt_cond_latent] * n

        async def process_tokens_to_speech(self, generator, speaker_embeddings, multimodal_data=None, request=None):
            assert speaker_embeddings is not None and multimodal_data is not None
            async for (L, i) in generator:
                yield ns_output(array=np.full(3 + i, float(1000 * L + i), np.float32), token_length=i + 1,
                                start_time=getattr(request, "start_time", None))

        async def shutdown(self):
            pass
    return Engine()


def _ref():
    from oracle import ref_facade
    return ref_facade.load()


def _side(which, conc=4, **kw):
    """(TTS driving the fake engine, TTSRequest class) of the reference's façade ("ref") or ours"""
    if which == "ref":
        import importlib
        ref = _ref()
        RefCC = importlib.import_module("auralis.models.base").ConditioningConfig
        r = ref.TTS(scheduler_max_concurrency=conc)
        r._ensure_event_loop()
        r.tts_engine = make_engine(ref.TTSOutput, RefCC(speaker_embeddings=True, gpt_like_decoder_conditioning=True), **kw)
        return r, ref.TTSRequest
    from auralis_b200.base import ConditioningConfig as OursCC
    return ours.TTS(scheduler_max_concurrency=conc).from_engine(make_engine(ours.TTSOutput, OursCC(True, True), **kw)), ours.TTSRequest


def _both(key, body, **kw):
    """-> (what body(tts, Req) returned on the reference's façade, as recorded; what it returns on ours)"""
    return rec(key, lambda: body(*_side("ref", **kw))), body(*_side("ours", **kw))


@pytest.mark.parametrize("n_chars", [5, 55, 200])
def test_generate_speech_same_audio(n_chars):
    def body(tts, Req):
        out = tts.generate_speech(Req(text="x" * n_chars, speaker_files=["s.wav"], language="en"))
        return np.asarray(out.array), out.sample_rate
    res = _both(f"generate_speech[{n_chars}]", body)
    np.testing.assert_array_equal(res[0][0], res[1][0])
    assert res[0][1] == res[1][1] == 24000


def test_streaming_same_chunks_in_same_order():
    def body(tts, Req):
        chunks = list(tts.generate_speech(Req(text="y" * 64, speaker_files=["s.wav"], language="en", stream=True)))
        return [(np.asarray(c.array).tolist(), c.token_length) for c in chunks]
    res = _both("streaming", body)
    assert res[0] == res[1] and len(res[0]) == 6


def test_long_request_is_split_like_the_reference():
    def split(tts, Req):
        req = Req(text="z" * 250_035, speaker_files=["s.wav"], language="en")
        parts = tts.split_requests(req, max_length=100_000)
        assert len({p.request_id for p in parts}) == len(parts)
        return [len(p.text) for p in parts]
    res = _both("split_requests", split)
    assert res[0] == res[1] == [100_000, 100_000, 50_035]

    # and the audio of a (smaller) split request is the concatenation of its parts, in order
    def audio(tts, Req):
        tts.split_requests = lambda request, max_length=100000, _f=type(tts).split_requests: _f(request, 30)
        out = tts.generate_speech(Req(text="w" * 75, speaker_files=["s.wav"], language="en"))
        return np.asarray(out.array)
    res = _both("split_request_audio", audio)
    np.testing.assert_array_equal(res[0], res[1])


def test_prepared_speaker_and_async_api():
    def body(tts, Req):
        base = Req(text="q" * 40, speaker_files=["s.wav"], language="en")
        fn = tts.loop.run_until_complete(tts.prepare_for_streaming_generation(base))
        calls = tts.tts_engine.cond_calls

        async def go():
            a = await tts.generate_speech_async(Req(text="q" * 40, speaker_files=["s.wav"], language="en", context_partial_function=fn))
            gen = await tts.generate_speech_async(Req(text="q" * 30, speaker_files=["s.wav"], language="en", stream=True,
                                                      context_partial_function=fn))
            b = [np.asarray(c.array).tolist() async for c in gen]
            return np.asarray(a.array).tolist(), b
        out = tts.loop.run_until_complete(go())
        assert tts.tts_engine.cond_calls == calls                  # the prepared conditioning is reused, not recomputed
        return out
    res = _both("prepared_speaker", body)
    assert res[0] == res[1]


def test_failing_chunk_raises_the_same_error():
    def body(tts, Req):
        with pytest.raises(Exception) as ei:
            tts.generate_speech(Req(text="x" * 30, speaker_files=["s.wav"], language="en"))
        return type(ei.value).__name__, str(ei.value)
    errs = _both("failing_chunk", body, fail_at=1)
    assert errs[0] == errs[1] == ("RuntimeError", "chunk 1 exploded")


def test_request_defaults_and_validation_match():
    def body(cls):
        r = cls(text="hi", speaker_files=["a.wav"])
        with pytest.raises(ValueError):
            cls(text="hi", speaker_files=["a.wav"], language="klingon")
        return {f: getattr(r, f) for f in ("temperature", "top_p", "top_k", "repetition_penalty", "length_penalty", "do_sample",
                                           "max_ref_length", "gpt_cond_len", "gpt_cond_chunk_len", "stream", "enhance_speech",
                                           "load_sample_rate", "sound_norm_refs", "language")}
    want = rec("request_defaults", lambda: body(_ref().TTSRequest))
    got = body(ours.TTSRequest)
    for f in want:
        assert got[f] == want[f], f


def test_output_helpers_match():
    """TTSOutput: bytes constructor (int16 + fade-in), combine_outputs, pcm encodings, resample, get_info, from_tensor."""
    import torch
    rng = np.random.RandomState(1)
    x = (rng.rand(4800).astype(np.float32) * 1.9 - 0.95)
    pcm = (rng.randint(-30000, 30000, size=600)).astype(np.int16).tobytes()

    def body(Out):
        a, b, c = Out(array=x.copy()), Out(array=x[::-1].copy()), Out(array=pcm)
        comb = Out.combine_outputs([a, b, c])
        rs = a.resample(16000)
        side = dict(
            from_bytes=np.asarray(c.array), comb=np.asarray(comb.array), comb_sr=comb.sample_rate,
            pcm2=a.to_bytes("pcm", 2), pcm4=a.to_bytes("pcm", 4), pcm1=a.to_bytes("pcm", 1),
            rs=np.asarray(rs.array), rs_sr=rs.sample_rate, info=a.get_info(),
            ft=np.asarray(Out.from_tensor(torch.from_numpy(x)[None], 22050).array), tensor=a.to_tensor().numpy())
        with pytest.raises(ValueError):
            a.to_bytes("ogg")
        return {k: sample(np.frombuffer(v, np.uint8) if isinstance(v, bytes) else v) if isinstance(v, (bytes, np.ndarray)) else v
                for k, v in side.items()}
    r, o = rec("output_helpers", lambda: body(_ref().TTSOutput)), body(ours.TTSOutput)
    for k in r:
        if isinstance(r[k], tuple) and isinstance(r[k][1], np.ndarray):       # sample() of an array or bytes
            assert o[k][0] == r[k][0], k
            np.testing.assert_array_equal(o[k][1], r[k][1], err_msg=k)
        else:
            assert o[k] == r[k], k


def test_load_audio_matches_the_reference_pipeline(tmp_path):
    """common/utilities.py:72-97 lifted by source (mono mix, torchaudio resample, clip) with `torchaudio.load` replaced by a
    stdlib WAV reader (the image has no codec backend): same samples as `auralis_b200.engine.load_audio` for a 48 kHz stereo
    16-bit file, a 22.05 kHz mono one and in-memory bytes."""
    import ast
    import io
    import types
    import wave
    import torch
    import torchaudio
    from auralis_b200.engine import load_audio

    def wav_bytes(sr, nch, seconds=0.25, seed=0):
        rng = np.random.RandomState(seed)
        x = (rng.rand(int(sr * seconds), nch) * 1.6 - 0.8)
        buf = io.BytesIO()
        with wave.open(buf, "wb") as w:
            w.setnchannels(nch); w.setsampwidth(2); w.setframerate(sr)
            w.writeframes((x * 32767).astype(np.int16).tobytes())
        return buf.getvalue()

    def fake_load(src):
        f = io.BytesIO(src) if isinstance(src, (bytes, bytearray)) else str(src)
        with wave.open(f, "rb") as w:
            nch, sr, raw = w.getnchannels(), w.getframerate(), w.readframes(w.getnframes())
        a = torch.from_numpy(np.frombuffer(raw, dtype="<i2").astype(np.float32) / 32768.0).reshape(-1, nch).t().contiguous()
        return a, sr
    def reference_load_audio(b):
        path = os.path.join(ref_import.REF_SRC, "auralis", "common", "utilities.py")
        tree = ast.parse(open(path).read())
        fn = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "load_audio"]
        ns = {"torch": torch, "torchaudio": types.SimpleNamespace(load=fake_load, functional=torchaudio.functional)}
        exec(compile(ast.Module(body=fn, type_ignores=[]), path, "exec"), ns)
        return ns["load_audio"](b, 22050)[0]
    for sr, nch in ((48000, 2), (22050, 1), (16000, 1), (44100, 2)):
        b = wav_bytes(sr, nch, seed=sr)
        shape, want = rec(f"load_audio[{sr},{nch}]", lambda: sample(reference_load_audio(b)))
        got = load_audio(b, 22050)
        assert got.dtype == np.float32 and got.shape == shape
        np.testing.assert_allclose(sample(got)[1], want, atol=1e-6, rtol=0)
        f = tmp_path / f"a{sr}.wav"
        f.write_bytes(b)
        np.testing.assert_allclose(load_audio(str(f), 22050), got, atol=1e-6, rtol=0)
    # IEEE-float WAV (what the reference's own TTSOutput.save writes) is accepted as a speaker reference too
    x = (np.random.RandomState(5).rand(4000).astype(np.float32) * 1.2 - 0.6)
    ours.TTSOutput(array=x, sample_rate=22050).save(tmp_path / "f32.wav")
    np.testing.assert_array_equal(load_audio(str(tmp_path / "f32.wav"), 22050), x)


def test_randomised_requests_same_results():
    """30 random (length, stream, failing chunk, scheduler concurrency) cases: both façades return the same audio in the same
    pieces, or fail with the same error."""
    rng = np.random.RandomState(2024)
    for case in range(30):
        n_chars = int(rng.randint(1, 140))
        stream = bool(rng.randint(2))
        n_chunks = max(1, n_chars // 10)
        fail_at = int(rng.randint(n_chunks)) if rng.rand() < 0.25 else None
        conc = int(rng.choice([1, 2, 5, 16]))

        def body(tts, Req):
            try:
                out = tts.generate_speech(Req(text="r" * n_chars, speaker_files=["s.wav"], language="en", stream=stream))
                if stream:
                    return ("ok", [np.asarray(c.array).tolist() for c in out])
                return ("ok", np.asarray(out.array).tolist())
            except Exception as e:      # noqa: BLE001
                return ("err", type(e).__name__, str(e))
        results = _both(f"randomised[{case}]", body, conc=conc, fail_at=fail_at)
        if results[0][0] == "err" and stream:
            assert results[1][0] == "err" and results[1][1:] == results[0][1:], (case, results)
        else:
            assert results[0] == results[1], (case, n_chars, stream, fail_at, conc)
