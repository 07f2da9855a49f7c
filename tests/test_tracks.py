"""Drop-in proof for the caller of the hot path (SURVEY.md 8 a-1 / f-2), CPU only.

The reference's OWN, UNMODIFIED lib/tracks.py (lib/tracks.py:9-38 of yondonfu/ai-rtc-agent) was run with `aiortc` stubbed
(it is not installable offline) and driven by the fake source track below, against this repo's pipeline call contract --
`pipeline(frame)` -- through warm-up, frame dropping and steady state.  tests/golden/make_tracks_golden.py recorded the frames
it returned and the pipeline calls it made in tests/golden/reference_tracks.json; this repo's non-blocking adapter
(host/tracks.py) must make the same pipeline calls in the same order and return the same frames."""
import asyncio
import json
import os

import pytest

REF_TRACKS_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_tracks.json")
DROPS = [0, 1]    # DROP_FRAMES values the reference was recorded with
RECV = 5          # recv() calls per recorded run


class FakeSource:
    """aiortc-like source track: recv() is a coroutine handing out numbered frames."""

    def __init__(self):
        self.n = 0

    async def recv(self):
        await asyncio.sleep(0)
        self.n += 1
        return ("frame", self.n)


class RecordingPipeline:
    """Stands for StreamDiffusionPipeline: records the frames it is called with (lib/tracks.py:24,38 call `pipeline(frame)`)."""

    def __init__(self):
        self.calls = []

    def __call__(self, frame):
        self.calls.append(frame)
        return ("processed", frame[1])


class Ticket:
    def __init__(self, value, polls):
        self.value, self.polls = value, polls

    def done(self):
        self.polls -= 1
        return self.polls < 0

    def result(self):
        return self.value


class AsyncRecordingPipeline(RecordingPipeline):
    """Same, with the non-blocking enqueue() entry of host/pipeline.py; every ticket needs a few polls to complete."""

    def enqueue(self, frame):
        return Ticket(self(frame), polls=3)


def _reference_run(drop):
    """(returned frames, pipeline calls, warm-up counter) of the reference's lib/tracks.py with DROP_FRAMES=drop."""
    with open(REF_TRACKS_GOLDEN) as f:
        gold = json.load(f)
    assert gold["recv_calls"] == RECV
    run = gold["runs"][str(drop)]
    return [tuple(x) for x in run["out"]], [tuple(x) for x in run["calls"]], run["warmup_frame_idx"]


def _drive(track, n):
    async def go():
        return [await track.recv() for _ in range(n)]
    return asyncio.run(go())


@pytest.mark.parametrize("drop", DROPS)
def test_reference_tracks_py_runs_unchanged_and_adapter_matches_it(monkeypatch, drop):
    monkeypatch.delenv("WARMUP_FRAMES", raising=False)
    monkeypatch.setenv("DROP_FRAMES", str(drop))
    # the reference half is recorded data (tests/golden/reference_tracks.json, written by make_tracks_golden.py from the
    # reference's unmodified lib/tracks.py); the two asserts on ref_* below pin that record, the others check this repo's adapter
    ref_out, ref_calls, ref_warmup_idx = _reference_run(drop)
    our_pipe = AsyncRecordingPipeline()
    from ai_rtc_agent_b200.host.tracks import VideoStreamTrack
    our_track = VideoStreamTrack(FakeSource(), our_pipe)
    our_out = _drive(our_track, RECV)
    # warm-up: 10 frames through the pipeline, discarded (lib/tracks.py:21-25); then `drop` source frames skipped per output
    first = 10 + drop + 1
    assert ref_out[0] == ("processed", first)
    assert [f[1] for f in ref_calls[:10]] == list(range(1, 11))
    assert our_out == ref_out
    assert our_pipe.calls == ref_calls
    assert ref_warmup_idx == our_track.warmup_frame_idx == 10


def test_reference_tracks_py_imports_this_repos_pipeline_module(monkeypatch):
    """agent.py:23 does `from lib.pipeline import StreamDiffusionPipeline` next to `from lib.tracks import VideoStreamTrack`:
    both names must resolve in this repo's lib/ package, and the pipeline class must be callable with one frame argument."""
    import inspect
    import lib.pipeline as lp
    import lib.tracks as lt
    assert inspect.iscoroutinefunction(lt.VideoStreamTrack.recv)
    sig = inspect.signature(lp.StreamDiffusionPipeline.__call__)
    assert list(sig.parameters) == ["self", "frame"]
    assert hasattr(lp.StreamDiffusionPipeline, "enqueue")


def test_adapter_yields_to_the_event_loop_while_a_frame_is_in_flight(monkeypatch):
    """The point of 8f-2: while the GPU works on a frame the event loop keeps running other coroutines."""
    monkeypatch.setenv("WARMUP_FRAMES", "2")
    monkeypatch.setenv("DROP_FRAMES", "0")
    from ai_rtc_agent_b200.host.tracks import VideoStreamTrack
    pipe = AsyncRecordingPipeline()
    track = VideoStreamTrack(FakeSource(), pipe)
    assert track.warmup_frames == 2      # int-cast (the reference keeps the env string and would raise on `int < str`)
    ticks = []

    async def other_peer():
        for _ in range(50):
            ticks.append(len(pipe.calls))
            await asyncio.sleep(0)

    async def go():
        t = asyncio.create_task(other_peer())
        out = await track.recv()
        await t
        return out

    out = asyncio.run(go())
    assert out == ("processed", 3)
    assert len(set(ticks)) >= 3, "the other coroutine must have observed the pipeline at several stages"


def test_adapter_accepts_a_plain_callable_pipeline(monkeypatch):
    monkeypatch.setenv("WARMUP_FRAMES", "0")
    from ai_rtc_agent_b200.host.tracks import VideoStreamTrack
    pipe = RecordingPipeline()
    assert _drive(VideoStreamTrack(FakeSource(), pipe), 3) == [("processed", 1), ("processed", 2), ("processed", 3)]
