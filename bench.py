#!/usr/bin/env python
"""bench.py — the hot path's headline metric on N B200s of one node.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference ...                      (CPU arm: the oracle port on the host cores)

Workload (BASELINE.json configs[1]): per GPU, 32 requests x 1 000 chars of synthetic English, 4 shared
speakers, temperature 0.75 / top_p 0.85 / top_k 50 / repetition penalty 5.0, random-init XTTSv2 weights of
the full geometry (30 x 1024 GPT-2, HiFi-GAN 512->32 ch).  With random weights the stop token never wins, so
every <=250-char chunk runs the full 605 tokens = 28.096 s of 24 kHz audio (SURVEY.md §8d) — a fixed unit of
work.  Weak scaling: the per-GPU request count is fixed as N grows.

One "step" = one pass of the hot path over the batch: text chunks -> GPT prefill + 605 decode steps with
continuous batching -> latents -> vocoder -> waveforms.
  * `value`  : audio-seconds per wall-second with inputs resident on the device (token ids uploaded before the
               timed region, waveforms left in HBM).
  * `e2e`    : the same metric through the public API (`TTS.generate_speech_batch(TTSRequest...)`): host text in,
               host float32 waveforms out, tokenisation, H2D and D2H inside the timed region.
Prints ONE JSON line on rank 0.
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

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SEED = 1234
DUMP_WAV_CHUNKS = 16            # --dump-outputs: a full step's waveforms are ~440 MB, 16 chunks ~40 MB
WORDS = ("the of and to in is that it was for on are as with his they at be this from have or by one had not but what "
         "all were when we there can an your which their said if do will each about how up out them then she many some "
         "so these would other into has more her two like him see time could no make than first been its who now people "
         "my made over did down only way find use may water long little very after words called just where most know "
         "get through back much before go good new write our used me man too any day same right look think also around "
         "another came come work three word must because does part even place well such here take why things help put "
         "years different away again off went old number great tell men say small every found still between name should "
         "home big give air line set own under read last never us left end along while might next sound below saw "
         "something thought both few those always looked show large often together asked house world going want").split()


def make_text(n_chars: int, seed: int) -> str:
    """Synthetic English: sentences of 60-120 chars from a fixed word list (SURVEY.md §8d)."""
    rng = np.random.RandomState(seed)
    out, total = [], 0
    while total < n_chars:
        target = rng.randint(60, 121)
        s = []
        n = 0
        while n < target:
            w = WORDS[rng.randint(len(WORDS))]
            s.append(w)
            n += len(w) + 1
        sent = " ".join(s).capitalize() + "."
        out.append(sent)
        total += len(sent) + 1
    return " ".join(out)[:n_chars]


def synthetic_wav_bytes(seconds: float, f0: float, seed: int, sr: int = 22050) -> bytes:
    """RIFF bytes of the synthetic speaker reference (SURVEY.md §8d)."""
    import io
    import wave
    t = np.arange(int(seconds * sr), dtype=np.float64) / sr
    rng = np.random.RandomState(seed)
    x = 0.3 * np.sin(2 * np.pi * (f0 + 40.0 * np.sin(2 * np.pi * 3.0 * t)) * t) + 0.01 * rng.randn(t.size)
    buf = io.BytesIO()
    with wave.open(buf, "wb") as w:
        w.setnchannels(1); w.setsampwidth(2); w.setframerate(sr)
        w.writeframes((np.clip(x, -1, 1) * 32767).astype(np.int16).tobytes())
    return buf.getvalue()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0: float, t1: float) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 <= t <= t1 and len(r) >= 7] or [r for (_, r) in self.rows if len(r) >= 7]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = [float(r[0]) for r in rows]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": float(rows[0][1]), "reasons": reasons,
                "power_w_max": max(float(r[2]) for r in rows), "samples": len(rows)}


def dump_outputs(out_dir: str, res: dict) -> None:
    """Writes one step's results {seq_id: (result, tokens, wav or None, _)} as float32 .npy files: tokens [chunks, max
    tokens] padded with -1, n_tokens / n_samples [chunks], the fetched waveforms [k, max samples] zero-padded and their
    seq ids [k].  Every value is an integer below 2^24 or a float32 sample, so float32 holds it exactly."""
    os.makedirs(out_dir, exist_ok=True)
    sids = sorted(res)
    n_tok = np.array([res[s][0].n_tokens for s in sids], np.float32)
    toks = np.full((len(sids), max(1, int(n_tok.max(initial=0)))), -1, np.float32)
    for i, s in enumerate(sids):
        toks[i, : len(res[s][1])] = res[s][1]
    wav_ids = [s for s in sids if res[s][2] is not None]
    wavs = np.zeros((len(wav_ids), max([res[s][2].size for s in wav_ids], default=0)), np.float32)
    for i, s in enumerate(wav_ids):
        wavs[i, : res[s][2].size] = res[s][2]
    arrays = {"tokens": toks, "n_tokens": n_tok, "n_samples": np.array([res[s][0].n_samples for s in sids], np.float32),
              "waveforms": wavs, "waveform_seq_ids": np.array(wav_ids, np.float32)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# =====================================================================================================
def cpu_reference_sample(dims, state, n_threads: int, chunks=None, n_chunks: int = 8, max_tokens: int = 48) -> dict:
    """One TIMED pass of the reference's CPU path (the oracle port, fp32 torch ops, all host threads) over a bounded sample
    of the same workload: the first `n_chunks` text chunks of the bench's own requests, every chunk truncated to
    `max_tokens` audio tokens (instead of 605), run COMPLETELY — prompt prefill, batched KV-cached decode of all chunks
    together (`GPTOracle.generate_batched`: a B = 1 loop would stream the 1.5 GB of fp32 weights once per token), sampling
    at the workload's temperature / top-p / top-k / penalty, and the vocoder on every chunk's latents.
    `value` = audio-seconds this pass produced / its wall time: nothing is extrapolated.  (The truncation over-weights the
    prompt prefill — ~12 % of the pass — and under-weights the attention over long contexts, both small next to the
    vocoder, which is ~70 % of the CPU time at any chunk length.)"""
    import torch
    from oracle import xtts_oracle as O
    torch.set_num_threads(n_threads)
    gs, cs = state
    orc = O.GPTOracle(gs, cs, dims)
    g = torch.Generator().manual_seed(500)
    conds = [torch.randn(dims.gpt.n_cond_latents, dims.gpt.hidden, generator=g) for _ in range(4)]
    dvs = [torch.nn.functional.normalize(torch.randn(dims.voc.d_vector, generator=g), dim=0) for _ in range(4)]
    if not chunks:
        rng = np.random.RandomState(0)
        chunks = [[0] + rng.randint(2, dims.gpt.n_text_tokens, size=60 + 5 * i).tolist() + [1] for i in range(n_chunks)]
    chunks = [list(c) for c in chunks[:n_chunks]]
    sp = O.SamplingParams(temperature=0.75, top_p=0.85, top_k=50, repetition_penalty=5.0, max_tokens=max_tokens,
                          stop_token=dims.gpt.stop_audio_token, seed=1)
    with torch.no_grad():
        t0 = time.perf_counter()
        toks, lats = orc.generate_batched([conds[i % 4] for i in range(len(chunks))], chunks, sp, fast_rng=True)
        t_gpt = time.perf_counter() - t0
        n_samples = 0
        for i, lat in enumerate(lats):
            n_samples += int(O.vocoder(lat, dvs[i % 4], cs, dims).numel())
        t_all = time.perf_counter() - t0
    audio_s = n_samples / 24000.0
    n_tok = sum(len(t) for t in toks)
    return {"value": audio_s / t_all, "unit": "audio-s/s", "cores": n_threads, "kind": "port",
            "sample": f"{len(chunks)} chunks of the workload x {max_tokens} tokens max (605 in the GPU arm), run completely: "
                      f"prefill + batched decode {t_gpt:.2f}s ({n_tok} tokens), vocoder {t_all - t_gpt:.2f}s -> {audio_s:.1f} audio-s in {t_all:.2f}s; no extrapolation",
            "seconds": t_all, "audio_s": audio_s, "gpt_tokens_per_s": n_tok / t_gpt,
            "vocoder_audio_s_per_s": audio_s / max(1e-9, t_all - t_gpt)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2, help="timed steps (>= 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="fp16", choices=["bf16", "fp16", "fp32"],
                    help="16-bit tensor-core operand format of the GPT (fp16 and bf16 run the same kernels at the same rate; fp16 is 8x closer to the fp32 parity mode) or fp32")
    ap.add_argument("--requests", type=int, default=32, help="requests per GPU")
    ap.add_argument("--chars", type=int, default=1000)
    ap.add_argument("--max-tokens", type=int, default=605)
    ap.add_argument("--microbatches", type=int, default=2, help="concurrent decode branches per step (engine option; unfused decode only)")
    ap.add_argument("--engine-opt", action="append", default=[], help="extra engine option key=value (repeatable)")
    ap.add_argument("--decode-chain", type=int, default=0, help="1 = fused persistent per-layer chain kernel in the decode step")
    ap.add_argument("--voc-segment", type=int, default=96, help="tokens per vocoder window while a chunk decodes (engine option voc_segment; 0 = whole chunks at the end)")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra arms (ragged lengths, cfg3 time-to-first-audio, fp32 parity mode, strong scaling)")
    ap.add_argument("--sweep", action="store_true", help="option sweeps only: skip the e2e arm and the CPU baseline (the line says so; not a headline run)")
    ap.add_argument("--small", action="store_true", help="tiny geometry (plumbing check only; not a valid bench number)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (B200 arm: rank 0's tokens of every chunk "
                         f"and the waveforms of {DUMP_WAV_CHUNKS} chunks picked with a fixed seed) to compare two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the B200 arm")

    import torch
    from auralis_b200.config import XTTSDims
    from auralis_b200.weights import synth_state
    from auralis_b200 import parallel

    if args.impl == "reference":
        # CPU arm: no process group, no CUDA context — ranks other than 0 leave immediately (nothing to tear down)
        rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), 0
    else:
        rank, world, local = parallel.init_from_env()
    dims = XTTSDims.small() if args.small else XTTSDims.full()
    # torch CPU ops on these shapes stop scaling (and regress) beyond ~32 threads: use the best of what the host has
    n_threads = min(os.cpu_count() or 1, 32)
    workload = f"cfg2: {args.requests} x {args.chars}-char English requests per GPU, 4 speakers, T=0.75 top_p=0.85 top_k=50 rep=5.0"

    # ------------------------------------------------------------------------------- reference (CPU) arm
    if args.impl == "reference":
        if rank != 0:
            return
        torch.set_num_threads(n_threads)
        state = synth_state(dims, SEED)
        from auralis_b200.text import XTTSTokenizer
        tok = XTTSTokenizer(dims.gpt.n_text_tokens, dims.gpt.max_text_tokens)
        chunks = []
        for i in range(args.requests):
            for ids in tok.batch_encode_with_split(make_text(args.chars, i), "en"):
                chunks.append([tok.bos_token_id] + ids + [tok.eos_token_id])
        for i in range(args.warmup):
            cpu_reference_sample(dims, state, n_threads, chunks)
        t0 = time.perf_counter()
        vals = [cpu_reference_sample(dims, state, n_threads, chunks) for _ in range(args.steps)]
        dt = time.perf_counter() - t0
        r = vals[-1]
        v = sum(x["audio_s"] for x in vals) / dt           # units processed in the timed region / its wall time
        r["value"] = v
        line = {"metric": "audio_seconds_per_second", "value": v, "unit": "audio-s/s", "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(1, args.steps), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
                "config": {"workload": workload, "sample": r["sample"], "note": "reference CPU path = oracle port "
                           "(the reference cannot run without CUDA + vLLM 0.6.4, SURVEY.md §8c); each step is one complete "
                           "pass over the bounded sample, timed as a whole"},
                "cpu_baseline": r, "gpu_launches": 0,
                "e2e": {"value": v, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------------------- B200 arm
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 arm has no CPU fallback (use --impl reference)")
    from auralis_b200 import TTS, TTSRequest, native
    from auralis_b200.engine import XTTSv2Engine, tune_host_allocator
    malloc_tuned = tune_host_allocator()      # output buffers stay on the heap (no page-fault storm per step), see engine.py
    torch.cuda.set_device(local)
    state = synth_state(dims, SEED)
    n_chunks_est = args.requests * (args.chars // 200 + 2)
    eng = XTTSv2Engine(dims, state[0], state[1], device=local, precision=args.precision,
                       max_concurrency=min(256, max(8, n_chunks_est)), max_speakers=8)
    ne = eng.native
    tts = TTS(scheduler_max_concurrency=4096).from_engine(eng)

    # speakers: 4 synthetic references, conditioned on the GPU once (cached per speaker, SURVEY §3.4)
    spk_bytes = [synthetic_wav_bytes(6.0, 100.0 + 25.0 * i, 7 + i) for i in range(4)]
    loop = tts.loop
    spk = [loop.run_until_complete(eng.get_audio_conditioning(b, 60, 30, 4)) for b in spk_bytes]
    spk_slots = [c.slot for c, _ in spk]

    texts = [make_text(args.chars, 1000 * rank + i) for i in range(args.requests)]
    reqs_chunks = [eng.prepare_text_tokens(t, "en") for t in texts]
    n_chunks = sum(len(c) for c in reqs_chunks)
    max_tok = min(args.max_tokens, dims.gpt.max_audio_tokens)

    # --dump-outputs: the last timed step copies these chunks' waveforms out of HBM (the others stay there, as in every step)
    dump_wav_ids = set()
    if args.dump_outputs:
        dump_wav_ids = set(np.random.RandomState(SEED).choice(n_chunks, min(DUMP_WAV_CHUNKS, n_chunks), replace=False).tolist())
    dumped = {}

    def device_step(step_idx: int, lengths=None, chunk_lists=None, want_wav=False):
        """lengths: per-chunk max_tokens (the ragged arm); chunk_lists: another request set (the strong-scaling arm);
        want_wav: seq ids whose waveforms are fetched, the results are then kept in `dumped`"""
        jobs, sid = [], 0
        for ri, chunks in enumerate(chunk_lists if chunk_lists is not None else reqs_chunks):
            for ci, ids in enumerate(chunks):
                sp = native.Sampling(temperature=0.75, top_p=0.85, top_k=50, repetition_penalty=5.0,
                                     max_tokens=max_tok if lengths is None else int(lengths[sid]),
                                     stop_token=dims.gpt.stop_audio_token, seed=SEED + step_idx, seq_seed=sid, vocode=True)
                jobs.append((sid, ids, spk_slots[ri % 4], sp))
                sid += 1
        res = eng.run_batch_direct(jobs, timeout_s=900, want_wav=want_wav)
        if want_wav:
            dumped.clear()
            dumped.update(res)
        return sum(r.n_samples for (r, _, _, _) in res.values()), sum(r.n_tokens for (r, _, _, _) in res.values())

    def timed_device_step(step_idx: int):
        return device_step(step_idx, want_wav=dump_wav_ids if step_idx == args.steps - 1 else False)

    def e2e_step(step_idx: int):
        reqs = [TTSRequest(text=t, speaker_files=spk_bytes[i % 4], language="en", temperature=0.75, top_p=0.85, top_k=50,
                           repetition_penalty=5.0, seed=SEED + 100 + step_idx) for i, t in enumerate(texts)]
        if max_tok != dims.gpt.max_audio_tokens:
            eng.dims.gpt.max_audio_tokens = max_tok          # reduced runs only (flagged in config)
        outs = tts.generate_speech_batch(reqs)
        # DP epilogue: every rank's waveforms go to rank 0 (the consumer) over NCCL.  Like the output shipping of a serving
        # system it runs BESIDE the next step: a worker thread issues the gather on its own CUDA stream while this thread
        # already generates step i + 1; the timed region ends only when the last gather has landed (gather_pool.join).
        if world > 1:
            local_w = {rank * len(outs) + i: o.array for i, o in enumerate(outs)}
            gather_jobs.append(gather_pool.submit(_gather, local_w, world * len(outs), step_idx))
        return sum(o.array.shape[0] for o in outs), sum(len(t) for t in texts)

    import concurrent.futures
    gather_pool = concurrent.futures.ThreadPoolExecutor(max_workers=1)
    gather_jobs = []
    gather_stream = torch.cuda.Stream(device=local) if world > 1 else None

    def _gather(local_w, n_items, step_idx):
        torch.cuda.set_device(local)
        with torch.cuda.stream(gather_stream):
            out = parallel.gather_waveforms(local_w, n_items, torch.device("cuda", local), dst=0, tag=f"s{step_idx % 2}")
            gather_stream.synchronize()
        return 0 if out is None else sum(int(w.shape[0]) for w in out)

    def gather_join():
        for f in gather_jobs:
            f.result(timeout=600)
        gather_jobs.clear()

    def log(msg):
        if rank == 0:
            print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def timed(fn, warm, steps):
        """-> (seconds on the device clock, seconds of host wall clock, per-step results, wall span).  The device figure is
        the distance between two CUDA events recorded on the engine's own stream: the first with the device idle (after the
        barrier + synchronize), the second behind the last step's work."""
        for i in range(warm):
            fn(i)
        gather_join()
        barrier()
        t0w = time.time(); t0 = time.perf_counter()
        ne.timer_start()
        acc = [fn(warm + i) for i in range(steps)]
        dt_ev = ne.timer_stop_ms() * 1e-3
        gather_join()                      # (e2e arm, N > 1) the last step's waveform gather is inside the timed region
        barrier()
        dt = time.perf_counter() - t0
        return dt_ev, dt, acc, (t0w, time.time())

    # ---- device-resident arm
    log(f"engine up: {n_chunks} chunks/GPU, {max_tok} tokens/chunk, precision {args.precision}")
    ne.set_option("d2h_wav", 0)
    ne.set_option("microbatches", args.microbatches)
    ne.set_option("decode_chain", args.decode_chain)
    ne.set_option("voc_segment", args.voc_segment)
    for kv in args.engine_opt:
        ne.set_option(kv.split("=")[0], int(kv.split("=")[1]))
    eng.park_poller(True)                 # the device arm drives the native completion queue directly
    sampler = ClockSampler(local) if rank == 0 else None
    for i in range(args.warmup):
        t_w = time.perf_counter()
        device_step(i)
        log(f"warm-up step {i}: {time.perf_counter() - t_w:.2f}s")
    ne.set_option("reset_stats", 0)
    if sampler:
        sampler.start()
    dt_dev, wall_dev, acc_dev, span = timed(timed_device_step, 0, args.steps)
    clocks = sampler.stop(*span) if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dumped)
    st = ne.stats()
    samples_dev = sum(a[0] for a in acc_dev)
    tokens_dev = sum(a[1] for a in acc_dev)
    log(f"device arm: {dt_dev:.2f}s (CUDA events; host wall {wall_dev:.2f}s) for {args.steps} step(s); engine clocks: gpt {st.gpt_ms:.0f} ms, vocoder {st.vocoder_ms:.0f} ms, "
        f"{st.decode_steps} decode steps, {st.kernel_launches} kernels")
    # ---- kernel-family profile: one more identical step with a CUDA event on either side of every launch.  The decode
    # step is replayed from a graph that carries the events as event-record nodes (no host launch gap inside the bracket,
    # full dependencies instead of PDL edges); prefill and vocoder launches are bracketed eagerly (long kernels).
    # The profile step also runs the decode rows as ONE branch: concurrent micro-batch branches overlap kernels of
    # different families, which would smear each family's own duration.
    ne.set_option("microbatches", 1)
    ne.set_option("voc_segment", 0)          # the vocoder after the decode, not beside it: each family's own duration
    ne.set_option("profile", 1)
    device_step(args.warmup + args.steps)
    prof = ne.kernel_profile()
    ne.set_option("profile", 0)
    ne.set_option("microbatches", args.microbatches)
    ne.set_option("voc_segment", args.voc_segment)
    for kv in args.engine_opt:
        ne.set_option(kv.split("=")[0], int(kv.split("=")[1]))

    extras = {}
    do_extras = not (args.sweep or args.no_extras or args.small)
    # ---- extra arm 1: LENGTH-DISTRIBUTED chunks (per-chunk max_tokens ~ U(150, 605)): what real weights produce — the stop
    # token lands at a different step per chunk, so chunks finish (and reach the vocoder) at different times and in ragged
    # batches.  Device-resident like `value`.
    if do_extras:
        rng_len = np.random.RandomState(SEED + 17)
        lens = rng_len.randint(150, max_tok + 1, size=n_chunks)
        device_step(900, lens)
        barrier()
        ne.timer_start()
        acc_r = [device_step(901 + i, lens) for i in range(2)]
        dt_r = ne.timer_stop_ms() * 1e-3
        extras["ragged"] = {"value": sum(a[0] for a in acc_r) / 24000.0 / dt_r, "unit": "audio-s/s", "steps": 2,
                            "ms_per_step": 1e3 * dt_r / 2, "tokens_per_s": sum(a[1] for a in acc_r) / dt_r,
                            "workload": f"same {n_chunks} chunks per GPU, per-chunk max_tokens ~ U(150, {max_tok}) (mean {float(lens.mean()):.0f}); "
                                        "chunks finish at different steps, the vocoder batches ragged windows"}
        log(f"ragged arm: {extras['ragged']['value']:.1f} audio-s/s")
    # ---- extra arm 2 (N > 1): STRONG scaling — the north-star headline shape, 64 x 1k-char requests in TOTAL
    if do_extras and world > 1:
        per_rank = max(1, 64 // world)
        strong_chunks = reqs_chunks[:per_rank]
        device_step(950, None, strong_chunks)
        barrier()
        ne.timer_start()
        acc_s = [device_step(951 + i, None, strong_chunks) for i in range(2)]
        dt_s = ne.timer_stop_ms() * 1e-3
        extras["_strong_local"] = (sum(a[0] for a in acc_s) / 24000.0, dt_s, per_rank)
    eng.park_poller(False)
    log("profile step done")

    # ---- end-to-end arm (public API, host buffers)
    ne.set_option("d2h_wav", 1)
    if args.sweep:
        ev_e2e, dt_e2e, acc_e2e, samples_e2e = 0.0, float("nan"), [], 0
    else:
        # two warm-up steps: the waveform gather alternates two sets of pinned staging buffers, both must exist before the clock
        ev_e2e, dt_e2e, acc_e2e, _ = timed(e2e_step, 2, args.steps)      # e2e = host wall clock: tokenisation and the host copies count
        samples_e2e = sum(a[0] for a in acc_e2e)
        log(f"e2e arm: {dt_e2e:.2f}s for {args.steps} step(s)")
    h2d = sum(len(ids) * 4 for chunks in reqs_chunks for ids in chunks)
    d2h = samples_e2e // max(1, args.steps) * 4 + n_chunks * max_tok * 4

    # ---- extra arm 3 (N = 1): cfg3 time-to-first-audio — 64 mixed-length requests streamed at t = 0 through the public async
    # API, without and with streaming pieces (first piece after 58 tokens = 2.7 s of audio)
    if do_extras and world == 1:
        import asyncio
        rng3 = np.random.RandomState(11)
        lens3 = rng3.randint(128, 4097, size=64)
        texts3 = [make_text(int(n), 5000 + i) for i, n in enumerate(lens3)]

        async def one(i, t0):
            req = TTSRequest(text=texts3[i], speaker_files=spk_bytes[i % 4], language="en", stream=True, seed=SEED + i)
            gen = await tts.generate_speech_async(req)
            first = None
            async for chunk in gen:
                if first is None:
                    first = time.perf_counter() - t0
            return first

        async def run3():
            t0 = time.perf_counter()
            return await asyncio.gather(*[one(i, t0) for i in range(len(texts3))])
        ttfa = {}
        for early in (0, 58):
            eng.early_emit_tokens = early
            tt = np.array(loop.run_until_complete(run3()))
            ttfa[f"early_{early}"] = {"p50_s": float(np.percentile(tt, 50)), "p99_s": float(np.percentile(tt, 99))}
        eng.early_emit_tokens = 0
        extras["cfg3_ttfa"] = {"requests": 64, "chars": "128..4096", "speakers": 4, **ttfa,
                               "note": "early_58: streaming pieces (xtts_sampling.early_tokens = 58): the first 2.7 s of a request's audio "
                                       "leave the engine ~65 decode steps after admission instead of after the whole 605-token chunk"}
        log(f"cfg3 time-to-first-audio: {ttfa}")

    # ---- max over ranks, aggregate over ranks
    if world > 1:
        t = torch.tensor([dt_dev, dt_e2e, wall_dev], dtype=torch.float64, device="cuda")
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        dt_dev, dt_e2e, wall_dev = float(t[0]), float(t[1]), float(t[2])
        s = torch.tensor([samples_dev, tokens_dev, samples_e2e], dtype=torch.float64, device="cuda")
        torch.distributed.all_reduce(s, op=torch.distributed.ReduceOp.SUM)
        samples_dev, tokens_dev, samples_e2e = float(s[0]), float(s[1]), float(s[2])
    if "_strong_local" in extras:
        a_s, dt_s, per_rank = extras.pop("_strong_local")
        t = torch.tensor([dt_s], dtype=torch.float64, device="cuda")
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        a = torch.tensor([a_s], dtype=torch.float64, device="cuda")
        torch.distributed.all_reduce(a, op=torch.distributed.ReduceOp.SUM)
        extras["strong"] = {"value": float(a[0]) / float(t[0]), "unit": "audio-s/s", "requests_total": per_rank * world,
                            "requests_per_gpu": per_rank, "steps": 2, "ms_per_step": 1e3 * float(t[0]) / 2,
                            "workload": "north-star headline shape: 64 x 1k-char requests in total, split over the GPUs (strong scaling)"}
    if rank != 0:
        loop.run_until_complete(tts.shutdown())
        if world > 1:
            torch.distributed.destroy_process_group()
        return

    audio_s_dev = samples_dev / 24000.0
    value = audio_s_dev / dt_dev
    e2e_value = None if args.sweep else (samples_e2e / 24000.0) / dt_e2e

    # ---- roofline of the dominant kernel family (device time by CUDA events inside the timed region)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    tc_peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
    total_ms = sum(v["ms"] for v in prof.values()) or 1.0
    dom_name, dom = max(prof.items(), key=lambda kv: kv[1]["ms"]) if prof else ("none", {"ms": 1, "flops": 0, "bytes": 0, "launches": 1})
    fams = {}
    for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"]):
        gbs = v["bytes"] / (v["ms"] * 1e-3) / 1e9 if v["ms"] else 0.0
        tfs = v["flops"] / (v["ms"] * 1e-3) / 1e12 if v["ms"] else 0.0
        fams[k] = {"ms": round(v["ms"], 3), "share": round(v["ms"] / total_ms, 4), "launches": v["launches"],
                   "GB/s": round(gbs, 1), "TFLOP/s": round(tfs, 2),
                   "frac_of_hbm_peak": round(gbs / hbm_peak, 4), "frac_of_tensor_peak": round(tfs / tc_peak, 4)}
    # which roof binds the dominant family: its algorithmic FLOP/byte against the machine's ridge point
    ridge = tc_peak * 1e12 / (hbm_peak * 1e9)
    ai = dom["flops"] / dom["bytes"] if dom.get("bytes") else 0.0
    tensor_bound = ai >= ridge
    if tensor_bound:
        ach = dom["flops"] / (dom["ms"] * 1e-3) / 1e12
        roof = {"bound": "tensor", "achieved": ach, "peak": tc_peak, "unit": "TFLOP/s", "frac": ach / tc_peak}
    else:
        ach = dom["bytes"] / (dom["ms"] * 1e-3) / 1e9
        roof = {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak}
    roof.update({"kernel": dom_name, "flop_per_byte": ai, "ridge_flop_per_byte": ridge, "avg_launch_us": 1e3 * dom["ms"] / max(1, dom["launches"]), "launches": dom["launches"],
                 "share_of_device_time": dom["ms"] / total_ms, "peak_source": peak_src, "traffic": None,
                 "fp32_tflops": dom["flops"] / (dom["ms"] * 1e-3) / 1e12 if dom["ms"] else None,
                 "families": fams})

    # DRAM traffic of the dominant family, per launch, from the committed ncu capture (profiles/ncu_traffic.json)
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(dom_name)
    except Exception:
        tr = None
    if tr:
        roof["traffic"] = tr["dram_bytes_per_launch"]
        roof["traffic_detail"] = {"unit": "bytes per launch", "algorithmic_bytes_per_launch_at_capture": tr["algorithmic_bytes_per_launch_at_capture"],
                                  "algorithmic_bytes_per_launch_this_run": dom["bytes"] / max(1, dom["launches"]),
                                  "shape": tr["shape"], "note": tr["note"], "source": tr["source"]}

    cpu = None
    if args.gpus == 1 and not args.sweep:
        cpu_reference_sample(dims, state, n_threads, reqs_chunks and [c for ch in reqs_chunks for c in ch], n_chunks=2, max_tokens=8)   # warm
        cpu = cpu_reference_sample(dims, state, n_threads, [c for ch in reqs_chunks for c in ch])

    line = {
        "metric": "audio_seconds_per_second", "value": value, "unit": "audio-s/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt_dev / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": {"bf16": "bf16", "fp16": "f16"}.get(args.precision, "f32"), "data": "synthetic",
        "config": {"workload": workload, "chunks_per_gpu": n_chunks, "tokens_per_chunk": max_tok,
                   "audio_s_per_step": audio_s_dev / args.steps, "geometry": "small (INVALID as a bench number)" if args.small else "XTTSv2 full: GPT-2 30x1024x16h, HiFi-GAN 512ch, random-init",
                   "parallelism": f"dp{args.gpus} (requests sharded, waveform all-gather only)",
                   "gpt_compute": (f"{args.precision} tcgen05 GEMM operands + {args.precision} KV, fp32 accumulate/residual/LN/softmax"
                                   if args.precision != "fp32" else "fp32"),
                   "vocoder_compute": "fp16 tcgen05 implicit-GEMM convs (fp32 accumulate, fp32 residual stream)" if args.precision != "fp32" else "fp32",
                   "l2": "no explicit flush: per-step working set (0.76 GB weights + >5 GB KV + 0.4 GB vocoder activations) >> 126 MB L2",
                   "timing": "CUDA events on the engine stream (first recorded with the device idle after barrier + synchronize, second "
                             "behind the last step's work); max over ranks; e2e: host wall clock around the public API calls",
                   "host_wall_ms_per_step": 1e3 * wall_dev / args.steps,
                   "engine_opts": args.engine_opt,
                   "host_allocator": "glibc mallopt(M_MMAP_THRESHOLD = 1 GiB, M_TRIM_THRESHOLD = max): output arrays reuse heap pages" if malloc_tuned else "default",
                   "vocoder": (f"windows of {args.voc_segment} tokens vocoded on a second stream while the chunk decodes (ragged batches of up to 32 windows)"
                               if args.voc_segment else "whole chunks, vocoded when they end (ragged batches)"),
                   "decode_step": ("per layer: paged attention + one persistent chain kernel (out-proj, LN2, fc+gelu, down-proj, LN1, next QKV)"
                                   if args.decode_chain else f"one launch per GEMM/LayerNorm, {args.microbatches} concurrent row branches"),
                   "roofline_timing": "CUDA events around every launch on the engine stream, in one extra identical step right after the timed ones (decode step: event-record nodes inside the replayed graph, single row branch, no PDL overlap; prefill/vocoder: eager)",
                   "e2e_speakers": "4 reference wavs conditioned on the GPU before the timed region (per-speaker cache, as prepare_for_streaming_generation)"},
        "gpt_tokens_per_s": tokens_dev / dt_dev, "rtf": 1.0 / value,
        "e2e": {"value": e2e_value, "unit": "audio-s/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "api": "TTS.generate_speech_batch([TTSRequest(text, speaker_files=wav bytes)])",
                "ms_per_step": None if args.sweep else 1e3 * dt_e2e / args.steps},
        "gpu_launches": int(st.kernel_launches),
        "clocks": clocks, "roofline": roof,
    }
    # ---- extra arm 4 (N = 1): the PARITY mode — fp32 CUDA-core GEMMs / convs, fp32 KV (greedy token ids bit-exact against
    # the oracle in tests/test_gpu_gpt.py, tests/test_gpu_bench_regime.py) on the same workload, one timed step
    if do_extras and world == 1:
        loop.run_until_complete(tts.shutdown())
        eng32 = XTTSv2Engine(dims, state[0], state[1], device=local, precision="fp32",
                             max_concurrency=min(256, max(8, n_chunks_est)), max_speakers=8)
        ne32 = eng32.native
        spk32 = [tts.loop.run_until_complete(eng32.get_audio_conditioning(b, 60, 30, 4))[0].slot for b in spk_bytes]
        ne32.set_option("d2h_wav", 0)

        def step32(i):
            jobs, sid = [], 0
            for ri, chunks in enumerate(reqs_chunks):
                for ids in chunks:
                    jobs.append((sid, ids, spk32[ri % 4], native.Sampling(temperature=0.75, top_p=0.85, top_k=50, repetition_penalty=5.0,
                                 max_tokens=max_tok, stop_token=dims.gpt.stop_audio_token, seed=SEED + i, seq_seed=sid, vocode=True)))
                    sid += 1
            res = eng32.run_batch_direct(jobs, timeout_s=900, want_wav=False)
            return sum(r.n_samples for (r, _, _, _) in res.values())
        step32(0)
        torch.cuda.synchronize()
        ne32.timer_start()
        n32 = step32(1)
        dt32 = ne32.timer_stop_ms() * 1e-3
        extras["fp32_value"] = n32 / 24000.0 / dt32
        extras["fp32"] = {"value": n32 / 24000.0 / dt32, "unit": "audio-s/s", "steps": 1, "ms_per_step": 1e3 * dt32,
                          "mode": "precision=fp32: CUDA-core fp32 GEMMs and convs, fp32 KV — the mode whose greedy token ids are bit-exact vs the oracle"}
        log(f"fp32 parity mode: {extras['fp32_value']:.1f} audio-s/s")
        tts.loop.run_until_complete(eng32.shutdown())
    line.update(extras)
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if args.sweep:
        line["sweep"] = "option sweep: e2e arm and CPU baseline skipped — not a headline run"
    print(json.dumps(line), flush=True)
    if not (do_extras and world == 1):
        loop.run_until_complete(tts.shutdown())
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
