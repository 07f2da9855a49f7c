"""Records what the original ai-rtc-agent's `lib/tracks.py:VideoStreamTrack` does with the fake source and recording pipeline
of tests/test_tracks.py, into tests/golden/reference_tracks.json:

  python tests/golden/make_tracks_golden.py <checkout of yondonfu/ai-rtc-agent>

The module is executed unmodified, with `aiortc` stubbed (it is only imported for the MediaStreamTrack base class).  For each
DROP_FRAMES value the file holds the frames the track returned, the frames it handed to the pipeline, in order, and its
warm-up counter afterwards; tests/test_tracks.py checks this repo's adapter against that record."""
import importlib.util
import json
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from tests.test_tracks import DROPS, RECV, FakeSource, RecordingPipeline, _drive  # noqa: E402


def load_tracks(checkout: str):
    aiortc = types.ModuleType("aiortc")

    class MediaStreamTrack:
        def __init__(self):
            self._ended = False

    aiortc.MediaStreamTrack = MediaStreamTrack
    sys.modules["aiortc"] = aiortc
    spec = importlib.util.spec_from_file_location("reference_lib_tracks", os.path.join(checkout, "lib", "tracks.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def main(checkout: str):
    mod = load_tracks(checkout)
    os.environ.pop("WARMUP_FRAMES", None)
    runs = {}
    for drop in DROPS:
        os.environ["DROP_FRAMES"] = str(drop)
        pipe = RecordingPipeline()
        track = mod.VideoStreamTrack(FakeSource(), pipe)
        out = _drive(track, RECV)
        runs[str(drop)] = {"out": out, "calls": pipe.calls, "warmup_frame_idx": track.warmup_frame_idx}
    with open(os.path.join(HERE, "reference_tracks.json"), "w") as f:
        json.dump({"recv_calls": RECV, "runs": runs}, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
