"""CPU: `auralis_b200.scheduler.TwoPhaseScheduler` against what the REFERENCE's own scheduler
(`common/scheduling/two_phase_scheduler.py`, imported unmodified by oracle/ref_sched.py) did, stored in
tests/golden/scheduler_vs_reference.npz (tests/reference_records.py), scenario by scenario, under the
contract the XTTS engine uses it with — every phase-2 generator yields exactly one item (vLLM FINAL_ONLY, XTTSv2.py:738).
Compared: the items and their order, the exception type and message that reach the caller, how many generators were ever
in flight at once, and which ones were started first.

Known, intended difference (not compared): the reference yields exactly ONE item per sequence index and never finishes a
request whose generators yield more (SURVEY App. B.13); ours yields every item of a generator in order, which the first-audio
early emit relies on."""
import asyncio

import pytest

from auralis_b200.scheduler import TwoPhaseScheduler as Ours
from reference_records import Records

rec = Records("scheduler_vs_reference")


async def _scenario(S, n=5, fail_at=None, conc=2, first_fails=False, slow_gen=None, sched_kw=None):
    sch = S(conc, **(sched_kw or {}))
    started, live, peak = [], [0], [0]

    async def first(x):
        if first_fails:
            raise ValueError("phase one broke")
        return {"parallel_inputs": [{"i": i} for i in range(n)], "request": x}

    async def second(gi):
        i = gi["i"]
        started.append(i); live[0] += 1; peak[0] = max(peak[0], live[0])
        try:
            await asyncio.sleep(1.0 if slow_gen == i else 0.004 * (n - i))       # earlier chunks finish LATER
            if fail_at == i:
                raise RuntimeError(f"boom {i}")
            yield ("item", i)
        finally:
            live[0] -= 1
    out, err = [], None
    try:
        async for item in sch.run(inputs="req", request_id="r1", first_phase_fn=first, second_phase_fn=second):
            out.append(item)
    except BaseException as e:      # noqa: BLE001 — the type is what is compared
        err = (type(e).__name__, str(e))
    try:
        await asyncio.wait_for(sch.shutdown(), 3)               # the reference keeps queue-processor tasks alive until told
    except BaseException:       # noqa: BLE001
        pass
    return out, err, peak[0], sorted(started[:conc])


def _run(S, **kw):
    async def main():
        return await asyncio.wait_for(_scenario(S, **kw), 15)
    return asyncio.new_event_loop().run_until_complete(main())


def _ref_run(**kw):
    from oracle import ref_sched
    return _run(ref_sched.load(), **kw)


def _key(name, kw):
    return name + "[" + ",".join(f"{k}={v}" for k, v in kw.items()) + "]"


@pytest.mark.timeout(120)
@pytest.mark.parametrize("kw", [
    dict(n=1), dict(n=5), dict(n=7, conc=1), dict(n=7, conc=3), dict(n=4, conc=10),
    dict(n=5, fail_at=0), dict(n=5, fail_at=2), dict(n=5, fail_at=4), dict(n=3, first_fails=True),
], ids=lambda kw: ",".join(f"{k}={v}" for k, v in kw.items()))
def test_same_behaviour_as_the_reference_scheduler(kw):
    want = rec(_key("scenario", kw), lambda: _ref_run(**kw))
    got = _run(Ours, **kw)
    assert (got[1] is None) == (want[1] is None)
    if want[1] is None:
        assert got[0] == want[0]                               # items, in order
    else:
        assert got[1] == want[1]                               # exception type and message
        # what was delivered before the error: the reference polls its buffers every 10 ms and checks for errors first
        # (two_phase_scheduler.py:334-350), ours is event-driven — so it may have handed out more of the items that
        # were already complete, never different ones and never out of order
        assert got[0][: len(want[0])] == want[0] and got[0] == [("item", i) for i in range(len(got[0]))]
    assert got[2] == want[2] and got[3] == want[3]             # concurrency peak, first generators started


@pytest.mark.timeout(120)
def test_timeouts_raise_timeout_error_like_the_reference():
    for kw in (dict(n=3, slow_gen=1, sched_kw=dict(request_timeout=0.15)), dict(n=3, slow_gen=1, sched_kw=dict(generator_timeout=0.15))):
        want = rec(_key("timeout", kw), lambda: _ref_run(**kw))
        got = _run(Ours, **kw)
        assert want[1] is not None and got[1] is not None, (want, got)
        assert got[1][0] == want[1][0] == "TimeoutError", (want, got)
        assert got[0][: len(want[0])] == want[0]               # what was delivered before the timeout (see above)
