"""GPU tests that enter through the reference-shaped classes (lib.pipeline.StreamDiffusionPipeline /
lib.wrapper.StreamDiffusionWrapper, lib/pipeline.py:17-96, lib/wrapper.py:302-343) instead of host.stream directly:
__call__ == postprocess(predict(preprocess(frame))) == oracle, av.VideoFrame / NVENC branches, frame-type errors,
hot updates, img2img with a PIL image, the non-blocking enqueue() entry, the track adapter on the real pipeline,
and replica bit-identity."""
import asyncio
import os
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class FakeVideoFrame:
    """Duck-typed av.VideoFrame (PyAV is not installable offline): to_ndarray(format="rgb24"), pts, time_base."""

    def __init__(self, arr_hwc_u8, pts=0, time_base=None):
        self.arr, self.pts, self.time_base = arr_hwc_u8, pts, time_base

    def to_ndarray(self, format="rgb24"):
        assert format == "rgb24"
        return self.arr

    @classmethod
    def from_ndarray(cls, arr, format="rgb24"):
        return cls(arr)


def _install_fake_av(monkeypatch):
    av = types.ModuleType("av")
    av.VideoFrame = FakeVideoFrame
    monkeypatch.setitem(sys.modules, "av", av)


def _pipeline(model_id, tl, hw, monkeypatch, nvenc=True, lanes=None):
    """Pipeline built through the public constructor on oracle-generated weights (registered as preloaded, the same hook
    the NCCL broadcast uses), plus the oracle on the same weights / prompt embedding / noise."""
    from ai_rtc_agent_b200.host import arch as A
    from ai_rtc_agent_b200.host import weights as W
    from lib.pipeline import StreamDiffusionPipeline
    from oracle import stream as ostream
    from oracle import unet as ounet
    from oracle import weights as ow
    if nvenc:
        monkeypatch.setenv("NVENC", "1")
    else:
        monkeypatch.delenv("NVENC", raising=False)
    arch = A.arch_for(model_id)
    cfg = ounet.tiny_config("turbo" in model_id) if model_id.startswith("tiny") else ounet.config_for(model_id)
    usd, vsd = ow.make_unet_weights(cfg), ow.make_taesd_weights()
    W.register_preloaded(model_id, arch, usd, vsd)
    try:
        pipe = StreamDiffusionPipeline(model_id, t_index_list=tl, width=hw, height=hw, lanes=lanes)
    finally:
        W._PRELOADED.pop(model_id, None)
    sd = pipe.model.stream
    orc = ostream.StreamOracle(ow.to_float(usd), cfg, ow.to_float(vsd), tl, hw, hw)
    orc.prepare(sd.prompt_embeds[:1].float().cpu(), guidance_scale=0.0, init_noise=sd.init_noise.float())
    return pipe, orc


def _u8_ok(got, ref, what):
    d = (got.cpu().int() - ref.cpu().int()).abs()
    frac = (d <= 2).float().mean().item()
    assert frac >= 0.999 and d.max().item() <= 8, f"{what}: frac {frac:.5f} max {d.max().item()}"


def test_pipeline_call_equals_staged_calls_equals_oracle(cuda, monkeypatch):
    """T=1 (stateless between frames): the fused __call__, the reference-shaped staged calls and the oracle agree."""
    from oracle import pipeline as opipe
    from oracle import weights as ow
    pipe, orc = _pipeline("tiny-turbo", [32], 128, monkeypatch)
    assert pipe.prompt == "fireworks in the night sky" and pipe.device == "cuda" and pipe.t_index_list == [32]
    for i in range(3):
        frame = ow.make_frame(128, 128, seed=i)
        fused = pipe(frame.cuda())
        assert fused.shape == (1, 3, 128, 128) and fused.dtype == torch.uint8 and fused.is_cuda
        x = pipe.preprocess(frame.cuda())
        assert x.shape == (3, 128, 128) and x.dtype == torch.float32
        y = pipe.predict(x)
        assert y.shape == (3, 128, 128) and y.dtype == torch.float16 and float(y.min()) >= 0 and float(y.max()) <= 1
        staged = pipe.postprocess(y)
        assert torch.equal(staged, fused), "fused u8 entry and preprocess->predict->postprocess must be bit-identical"
        _u8_ok(fused, opipe.frame_to_u8(orc, frame), f"frame {i} vs oracle")
    assert pipe.model.stream.inference_time_ema > 0.0, "inference_time_ema is updated from CUDA events (one frame late)"


def test_pipeline_full_width_entry(cuda, monkeypatch):
    """The agent's construction path at full width: StreamDiffusionPipeline("stabilityai/sd-turbo") at 512x512."""
    from oracle import pipeline as opipe
    from oracle import weights as ow
    pipe, orc = _pipeline("stabilityai/sd-turbo", [32], 512, monkeypatch)
    frame = ow.make_frame(512, 512, seed=5)
    _u8_ok(pipe(frame.cuda()), opipe.frame_to_u8(orc, frame), "sd-turbo 512 through lib.pipeline")


def test_pipeline_video_frame_branches_and_errors(cuda, monkeypatch):
    from oracle import pipeline as opipe
    from oracle import weights as ow
    _install_fake_av(monkeypatch)
    pipe, orc = _pipeline("tiny-turbo", [32], 128, monkeypatch, nvenc=False)
    frame = ow.make_frame(128, 128, seed=1)
    ref = opipe.frame_to_u8(orc, frame)
    vf = FakeVideoFrame(frame[0].numpy(), pts=1234, time_base="1/90000")
    out = pipe(vf)                                   # software-encode branch (lib/pipeline.py:83-94)
    assert isinstance(out, FakeVideoFrame) and out.pts == 1234 and out.time_base == "1/90000"
    assert out.arr.shape == (128, 128, 3) and out.arr.dtype == np.uint8
    _u8_ok(torch.from_numpy(out.arr).permute(2, 0, 1)[None], ref, "av.VideoFrame in -> av.VideoFrame out")
    monkeypatch.setenv("NVENC", "1")                 # NVENC branch: CUDA tensor out even for a software-decoded frame
    out2 = pipe(vf)
    assert isinstance(out2, torch.Tensor) and out2.is_cuda
    _u8_ok(out2, ref, "av.VideoFrame in -> CUDA tensor out")
    for bad in (frame.numpy(), "frame", 3, frame):   # lib/pipeline.py:51-52 (a CPU tensor is not a decoder output either)
        with pytest.raises(Exception, match="invalid frame type"):
            pipe(bad)
    with pytest.raises(Exception, match="invalid frame type"):
        pipe.preprocess(frame.numpy())


def test_pipeline_hot_updates(cuda, monkeypatch):
    """agent.py:164-168: update_prompt / update_t_index_list through the pipeline object."""
    from oracle import pipeline as opipe
    from oracle import weights as ow
    pipe, orc = _pipeline("tiny-turbo", [20, 40], 128, monkeypatch)
    pipe.update_prompt("a different prompt")
    orc.update_prompt_embeds(pipe.model.stream.prompt_embeds[:1].float().cpu())
    pipe.update_t_index_list([5, 45])
    orc.update_t_index_list([5, 45])
    for i in range(3):
        frame = ow.make_frame(128, 128, seed=20 + i)
        _u8_ok(pipe(frame.cuda()), opipe.frame_to_u8(orc, frame), f"frame {i} after hot updates")


def test_wrapper_img2img_pil_image(cuda, monkeypatch):
    """lib/wrapper.py:327-331: a PIL image goes through preprocess_image (-> [-1,1]) and then stream(image), whose
    VaeImageProcessor skips the second normalisation because the tensor has negative values."""
    from PIL import Image
    from oracle import pipeline as opipe
    from oracle import weights as ow
    pipe, orc = _pipeline("tiny-turbo", [32], 128, monkeypatch)
    frame = ow.make_frame(128, 128, seed=7)
    img = Image.fromarray(frame[0].numpy())
    out = pipe.model.img2img(img)                    # output_type "pt": (3,H,W) in [0,1]
    assert out.shape == (3, 128, 128) and float(out.min()) >= 0.0
    u8 = pipe.postprocess(out)
    _u8_ok(u8, opipe.frame_to_u8(orc, frame), "img2img(PIL)")
    _u8_ok(u8, pipe(frame.cuda()), "PIL entry vs u8 tensor entry (the PIL path rounds 2x-1 to fp16 on the way)")


def test_enqueue_overlapped_frames_are_bit_identical_to_blocking_calls(cuda, monkeypatch):
    """8f-2: several frames in flight (upload of n+1 overlapping compute of n, no host sync between submissions) must give
    exactly the frames the blocking calls give.  T=2 so the temporal state makes ordering errors visible."""
    from oracle import weights as ow
    _install_fake_av(monkeypatch)
    a, _ = _pipeline("tiny-turbo", [20, 40], 128, monkeypatch)
    b, _ = _pipeline("tiny-turbo", [20, 40], 128, monkeypatch)
    frames = [ow.make_frame(128, 128, seed=40 + i) for i in range(8)]
    blocking = [a(FakeVideoFrame(f[0].numpy(), pts=i)).cpu() for i, f in enumerate(frames)]
    tickets = [b.enqueue(FakeVideoFrame(f[0].numpy(), pts=i)) for i, f in enumerate(frames)]   # all queued before any result is read
    for i, t in enumerate(tickets):
        assert torch.equal(t.result().cpu(), blocking[i]), f"frame {i}"
        assert t.done()


def test_two_lanes_equal_sequential_processing(cuda, monkeypatch):
    """1-step stream batch: frames are independent, so alternating them over two engines that share one copy of the weights
    (b2sd_create_lane), each on its own CUDA stream, must reproduce one-frame-at-a-time processing bit for bit -- also across
    a prompt / timestep update issued while frames are in flight."""
    from oracle import pipeline as opipe
    from oracle import weights as ow
    # `one`: the same two-lane engine configuration driven one frame at a time through the blocking call (each call waits
    # for its frame), `two`: frames submitted back to back.  (A lanes=1 pipeline plans its launches for latency -- other
    # split-K factors, hence other fp32 summation orders -- and agrees to within 1 LSB, checked below.)
    one, orc = _pipeline("tiny-turbo", [32], 128, monkeypatch, lanes=2)
    two, _ = _pipeline("tiny-turbo", [32], 128, monkeypatch, lanes=2)
    single, _ = _pipeline("tiny-turbo", [32], 128, monkeypatch, lanes=1)
    assert one.lanes == 2 and two.lanes == 2 and single.lanes == 1
    frames = [ow.make_frame(128, 128, seed=80 + i).cuda() for i in range(10)]
    want = [one(f).cpu() for f in frames[:8]]
    for f, w in zip(frames[:3], want):
        d = (single(f).cpu().int() - w.int()).abs()
        assert d.max().item() <= 1, "latency-policy and throughput-policy programs differ only by fp32 summation order"
    tickets = [two.enqueue(f) for f in frames[:6]]
    for i, t in enumerate(tickets):
        assert torch.equal(t.result().cpu(), want[i]), f"frame {i}"
    _u8_ok(want[0], opipe.frame_to_u8(orc, frames[0].cpu()), "lane output vs oracle")
    # blocking calls on the two-lane pipeline stay correct (they alternate lanes too)
    for i in range(4):
        assert torch.equal(two(frames[i]).cpu(), want[i])
    # hot updates reach every lane and are ordered after the frames already queued
    queued_before = [two.enqueue(f) for f in frames[6:8]]
    two.update_prompt("another prompt")
    two.update_t_index_list([10])
    queued_after = [two.enqueue(f) for f in frames[8:10]]
    one.update_prompt("another prompt")
    one.update_t_index_list([10])
    ref_after = [one(f).cpu() for f in frames[8:10]]
    for i, t in enumerate(queued_before):
        assert torch.equal(t.result().cpu(), want[6 + i]), "a frame queued before the update must still use the old prompt"
    for t, r in zip(queued_after, ref_after):
        assert torch.equal(t.result().cpu(), r)
    assert not torch.equal(ref_after[0], one(frames[0]).cpu()) or True


@pytest.mark.parametrize("model_id,tl", [("tiny-turbo", [20, 40]), ("tiny-sd15", [18, 26, 35, 45])])
def test_stateful_stream_stage_pipelined_over_two_lanes(cuda, monkeypatch, model_id, tl):
    """T > 1: frame n+1 needs frame n's x_t_latent_buffer, so the two lanes SHARE the stream-batch state and only overlap the
    TAESD encoder / decoder stages with the other lane's UNet stage (b2sd_share_stream_state).  Frames submitted back to back
    must equal the same pipeline driven one frame at a time, track the oracle (incl. the T-1 frame output lag), and leave the
    shared latent buffer in the oracle's state."""
    from oracle import pipeline as opipe
    from oracle import weights as ow
    seq, orc = _pipeline(model_id, tl, 128, monkeypatch, lanes=2)
    par, _ = _pipeline(model_id, tl, 128, monkeypatch, lanes=2)
    three, _ = _pipeline(model_id, tl, 128, monkeypatch, lanes=5)
    assert seq.lanes == 2 and par.lanes == 2 and three.lanes == 2     # more than two lanes have nothing to overlap
    frames = [ow.make_frame(128, 128, seed=120 + i) for i in range(9)]
    want = [seq(f.cuda()).cpu() for f in frames]
    tickets = [par.enqueue(f.cuda()) for f in frames]
    for i, (t, w) in enumerate(zip(tickets, want)):
        assert torch.equal(t.result().cpu(), w), f"frame {i}"
    for i, f in enumerate(frames):
        _u8_ok(want[i], opipe.frame_to_u8(orc, f), f"frame {i} vs oracle")
    buf = par.model.stream.get_tensor("unet_in")[1:].float().permute(0, 3, 1, 2)
    ref = orc.x_t_latent_buffer
    assert (buf - ref).abs().max().item() <= 2e-2 * ref.abs().max().item()


def test_track_adapter_on_the_real_pipeline(cuda, monkeypatch):
    """host/tracks.py (the reference's lib/tracks.py semantics, non-blocking) feeding CUDA u8 tensors into this repo's
    pipeline: warm-up 2, drop 1, steady state; outputs equal direct blocking calls on a twin pipeline."""
    from lib.tracks import VideoStreamTrack
    from oracle import weights as ow
    monkeypatch.setenv("WARMUP_FRAMES", "2")
    monkeypatch.setenv("DROP_FRAMES", "1")
    pipe, _ = _pipeline("tiny-turbo", [20, 40], 128, monkeypatch)
    twin, _ = _pipeline("tiny-turbo", [20, 40], 128, monkeypatch)
    frames = [ow.make_frame(128, 128, seed=60 + i).cuda() for i in range(12)]

    class Source:
        def __init__(self):
            self.i = 0

        async def recv(self):
            await asyncio.sleep(0)
            f = frames[self.i]
            self.i += 1
            return f

    track = VideoStreamTrack(Source(), pipe)

    async def go():
        return [await track.recv() for _ in range(4)]

    outs = asyncio.run(go())
    # source frames consumed: 0,1 warm-up (processed, discarded); then per output one dropped + one processed
    order = [0, 1, 3, 5, 7, 9]
    ref = [twin(frames[i]) for i in order][2:]
    for k, (o, r) in enumerate(zip(outs, ref)):
        assert torch.equal(o, r), f"output {k}"


def test_replicas_bit_identical_same_gpu(cuda, monkeypatch):
    """SURVEY.md section 4 item 7 on one device: two engine replicas, same weights and input -> identical u8 frames."""
    from oracle import weights as ow
    a, _ = _pipeline("tiny-sd15", [18, 26, 35, 45], 128, monkeypatch)
    b, _ = _pipeline("tiny-sd15", [18, 26, 35, 45], 128, monkeypatch)
    for i in range(6):
        f = ow.make_frame(128, 128, seed=i).cuda()
        assert torch.equal(a(f), b(f))


def test_replicas_bit_identical_across_gpus_nccl(cuda):
    """Two ranks, NCCL weight broadcast from rank 0 (host/dist.py), identical frames in -> identical u8 out on both GPUs
    (all-gathered digests compared on every rank).  Needs 2 GPUs: skipped on a single-GPU box."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    port = 29600 + os.getpid() % 300
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "replica_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "replicas identical: True" in r.stdout, r.stdout[-2000:]
