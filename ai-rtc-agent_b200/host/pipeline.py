"""Drop-in for the reference's `lib/pipeline.py:StreamDiffusionPipeline` (lib/pipeline.py:17-96): same
module constants, constructor, attributes and methods, so agent.py:23,423 and lib/tracks.py:24,38 run on
it unchanged.

Frames: the reference accepts `nvcv.Tensor` (NVDEC path) or `av.VideoFrame` (software decode).  Neither
package exists offline, so frames are recognised structurally: anything exposing
`__cuda_array_interface__` / `.cuda()` (nvcv.Tensor, torch.Tensor) is a GPU u8 NHWC frame, anything with
`.to_ndarray` is an av.VideoFrame; everything else raises Exception("invalid frame type") like
lib/pipeline.py:51-52.

Fast path: a GPU u8 frame goes through ONE engine call (pre + encode + UNet + decode + post fused,
u8 NHWC in -> u8 NCHW out, nothing leaves HBM).  preprocess / predict / postprocess remain callable
separately with the reference's tensor contracts."""
from __future__ import annotations

import os
from typing import List, Optional

import numpy as np
import torch

from .wrapper import StreamDiffusionWrapper

DEFAULT_PROMPT = "fireworks in the night sky"
DEFAULT_T_INDEX_LIST = [18, 26, 35, 45]
DEFAULT_NUM_INFERENCE_STEPS = 50
DEFAULT_GUIDANCE_SCALE = 0.0
DEFAULT_LANES_ONE_STEP = 8    # frames in flight for a 1-step stream batch (measured with the throughput launch policy: 4 -> 409, 6 -> 470,
                              # 8 -> 483, 10 -> 481, 12 -> 486 fps; p50 submit -> result 10.4 / 13.5 / 16.8 / 17.8 / 18.7 ms; lanes=1: 241 fps, 4.2 ms)
DEFAULT_LANES_STATEFUL = 2    # T > 1: stage pipelining over two lanes that share the stream-batch state


def _is_video_frame(frame) -> bool:
    return hasattr(frame, "to_ndarray") and hasattr(frame, "pts")


def _is_gpu_frame(frame) -> bool:
    if isinstance(frame, torch.Tensor):
        return frame.is_cuda
    return hasattr(frame, "__cuda_array_interface__") or (hasattr(frame, "cuda") and hasattr(frame, "layout"))


def _as_torch_u8_nhwc(frame, device) -> torch.Tensor:
    if isinstance(frame, torch.Tensor):
        t = frame
    elif hasattr(frame, "cuda") and not hasattr(frame, "__cuda_array_interface__"):
        t = torch.as_tensor(frame.cuda(), device=device)  # nvcv.Tensor
    else:
        t = torch.as_tensor(frame, device=device)
    if t.dim() == 3:
        t = t.unsqueeze(0)
    if t.dtype != torch.uint8 or t.shape[-1] != 3:
        raise Exception("invalid frame type")
    return t


class StreamDiffusionPipeline:
    def __init__(self, model_id: str, t_index_list: Optional[List[int]] = None, width: int = 512, height: int = 512,
                 prompt: str = DEFAULT_PROMPT, lanes: Optional[int] = None, *, cfg_type: str = "self",
                 guidance_scale: float = DEFAULT_GUIDANCE_SCALE, delta: float = 1.0, negative_prompt: str = ""):
        """lanes: frames in flight for enqueue() ($B200SD_LANES overrides the default).  With a 1-step stream batch (SD-Turbo)
        consecutive frames are independent: DEFAULT_LANES_ONE_STEP lanes process frame n+1.. while frame n is still on the GPU.
        With T > 1 the stream batch carries state from frame to frame: two lanes share that state and are stage-pipelined (TAESD
        encoder of frame n+1 and decoder of frame n-1 overlap the UNet of frame n).  Both are bit-identical to submitting the
        same frames one at a time.
        cfg_type / guidance_scale / delta / negative_prompt: StreamDiffusion's classifier-free guidance (active when
        guidance_scale > 1 and cfg_type != "none"); the defaults are unguided.  Residual guidance ("self") carries its stock
        noise from frame to frame even with a 1-step stream batch, so such a stream runs on two shared-state lanes too."""
        self.prompt = prompt
        self.t_index_list = list(t_index_list) if t_index_list is not None else DEFAULT_T_INDEX_LIST
        self.device = "cuda"
        self.model = StreamDiffusionWrapper(
            model_id_or_path=model_id,
            device=self.device,
            dtype=torch.float16,
            t_index_list=self.t_index_list,
            frame_buffer_size=1,
            width=width,
            height=height,
            use_lcm_lora=True,
            output_type="pt",
            mode="img2img",
            use_denoising_batch=True,
            use_tiny_vae=True,
            cfg_type=cfg_type,
            engine_dir=os.getenv("TRT_ENGINES_CACHE", "./models/engines"),
        )
        # x_t_latent_buffer (T > 1) or the stock noise of residual guidance chains frame n+1 to frame n
        stateful = len(self.t_index_list) > 1 or (cfg_type == "self" and guidance_scale > 1.0)
        if lanes is None:
            lanes = int(os.getenv("B200SD_LANES", "0")) or (DEFAULT_LANES_STATEFUL if stateful else DEFAULT_LANES_ONE_STEP)
        if stateful:
            lanes = min(lanes, 2)   # three stages, the middle one serial: a third lane has nothing to overlap
        # launch policy = number of frames in flight ($B200SD_POLICY_FRAMES overrides it for profiling: a single lane running the
        # throughput policy's launches gives ncu a clean one-frame launch list)
        self.model.stream.set_concurrency(max(1, int(os.environ.get("B200SD_POLICY_FRAMES", lanes))))
        self.model.prepare(prompt=self.prompt, negative_prompt=negative_prompt, num_inference_steps=DEFAULT_NUM_INFERENCE_STEPS,
                           guidance_scale=guidance_scale, delta=delta)
        sd = self.model.stream
        self._engines = [sd] + [sd.add_lane(share_state=stateful) for _ in range(max(1, lanes) - 1)]
        # one lane: frames run on the caller's stream, exactly as before.  Several lanes: every lane has its own stream (a lane on
        # the caller's stream would order the other lanes' "input ready" events behind its frames and serialise them)
        self._lane_streams = [None] if len(self._engines) == 1 else [torch.cuda.Stream(sd.device) for _ in self._engines]
        self._lane_done = [None] * len(self._engines)     # completion event of the last frame given to each lane
        self._next_lane = 0
        # Every frame's output is a fresh tensor allocated on its lane's stream (the caller owns it and may hold it across calls,
        # SURVEY 8b "Ownership").  Give each lane stream's allocator pool a few output-sized blocks now: the first cudaMalloc a
        # lane needed in the middle of a stream otherwise synchronises the device, i.e. stalls every frame in flight once
        # (seen as a single 2x latency spike, 33 ms instead of 17 ms, some 50-80 frames into a run with 10 frames pending).
        for st in self._lane_streams:
            if st is not None:
                with torch.cuda.stream(st):
                    prime = [torch.empty((1, 3, self.model.height, self.model.width), dtype=torch.uint8, device=sd.device)
                             for _ in range(4)]
                    del prime

    @property
    def lanes(self) -> int:
        return len(self._engines)

    def _quiesce(self):
        """Every lane finishes its queued frames before a prompt / timestep update touches the shared schedule."""
        cur = torch.cuda.current_stream(self.model.stream.device)
        for ev in self._lane_done:
            if ev is not None:
                cur.wait_event(ev)
        return cur

    def _release(self, cur):
        done = torch.cuda.Event()
        done.record(cur)
        for st in self._lane_streams:
            if st is not None:
                st.wait_event(done)

    def update_prompt(self, prompt: str):
        cur = self._quiesce()
        self.model.stream.update_prompt(prompt)
        self._release(cur)

    def update_t_index_list(self, t_index_list: List[int]):
        cur = self._quiesce()
        self.model.update_t_index_list(t_index_list)
        self._release(cur)

    # ---- reference-shaped stages ----------------------------------------------------------------------
    def preprocess(self, frame) -> torch.Tensor:
        """-> (3,H,W) float32 in [0,1] on the GPU (lib/pipeline.py:50-67)."""
        if not _is_gpu_frame(frame) and not _is_video_frame(frame):
            raise Exception("invalid frame type")
        if _is_video_frame(frame):
            t = torch.from_numpy(frame.to_ndarray(format="rgb24")).unsqueeze(0).to(self.device)
        else:
            t = _as_torch_u8_nhwc(frame, self.device)
        return (t.to(torch.float32) * (1.0 / 255.0)).permute(0, 3, 1, 2).squeeze(0)

    def predict(self, frame: torch.Tensor) -> torch.Tensor:
        return self.model(image=frame)

    def postprocess(self, frame: torch.Tensor) -> torch.Tensor:
        """(3,H,W) in [0,1] -> (1,3,H,W) uint8; the cast truncates (lib/pipeline.py:72-74)."""
        return frame.mul(255.0).clamp_(0, 255).to(torch.uint8)[None]

    def __call__(self, frame):
        """lib/pipeline.py:76-96, blocking semantics preserved: the result is complete when the call returns only in the
        software-encode branch (`.cpu()`); with NVENC set the CUDA tensor is returned stream-ordered, like the reference."""
        ticket = self.enqueue(frame)
        if os.getenv("NVENC"):
            ticket.wait(torch.cuda.current_stream(self.model.stream.device))   # stream-ordered result, whichever lane ran it
            return ticket.result(wait=False)
        return ticket.result()

    # ---- non-blocking entry (SURVEY.md 8f-2): everything is queued on CUDA streams and a ticket comes back at once ------
    def enqueue(self, frame) -> "FrameTicket":
        """Queue one frame and return immediately.  GPU frames (NVDEC path) go straight to the engine on the current
        stream.  av.VideoFrame input is staged through a pinned ring and copied on a separate copy stream, so the upload of
        frame n+1 overlaps the compute of frame n; with NVENC unset the download of the result is queued the same way.
        Tickets complete in submission order (one temporal stream per pipeline, like the reference)."""
        if not _is_gpu_frame(frame) and not _is_video_frame(frame):
            raise Exception("invalid frame type")
        dev = self.model.stream.device
        caller = torch.cuda.current_stream(dev)
        lane = self._next_lane
        self._next_lane = (lane + 1) % len(self._engines)
        engine = self._engines[lane]
        compute = self._lane_streams[lane] or caller
        if compute is not caller:
            ready = torch.cuda.Event()
            ready.record(caller)          # whatever produced the frame on the caller's stream
            compute.wait_event(ready)
        if _is_video_frame(frame):
            self._ensure_staging(dev)
            slot = self._slot
            self._slot = (slot + 1) % len(self._pinned_in)
            self._slot_free[slot].synchronize()          # the ring entry's previous upload has been consumed (depth-4 ring)
            arr = frame.to_ndarray(format="rgb24")
            host = self._pinned_in[slot]
            if tuple(arr.shape) != tuple(host.shape[1:]):
                host = self._pinned_in[slot] = torch.empty((1,) + tuple(arr.shape), dtype=torch.uint8).pin_memory()
            host[0].copy_(torch.from_numpy(arr))
            with torch.cuda.stream(self._copy_stream):
                rgb = host.to(dev, non_blocking=True)
                uploaded = torch.cuda.Event()
                uploaded.record(self._copy_stream)
            compute.wait_event(uploaded)
            rgb.record_stream(compute)
        else:
            slot = None
            rgb = _as_torch_u8_nhwc(frame, self.device)
            if compute is not caller:
                rgb.record_stream(compute)
        with torch.cuda.stream(compute):
            post_output = engine.step_u8(rgb)
        if compute is not caller:
            post_output.record_stream(caller)
        if slot is not None:
            self._slot_free[slot].record(compute)
        done = torch.cuda.Event()
        if os.getenv("NVENC"):
            done.record(compute)
            self._lane_done[lane] = done
            return FrameTicket(post_output, done, None, None)
        # software-encode branch (lib/pipeline.py:83-94): hand back an av.VideoFrame with the input's timing
        assert _is_video_frame(frame)
        self._ensure_staging(dev)
        host_out = torch.empty((1, 3, self.model.height, self.model.width), dtype=torch.uint8).pin_memory()
        computed = torch.cuda.Event()
        computed.record(compute)
        with torch.cuda.stream(self._copy_stream):
            self._copy_stream.wait_event(computed)
            host_out.copy_(post_output, non_blocking=True)
            post_output.record_stream(self._copy_stream)
            done.record(self._copy_stream)
        self._lane_done[lane] = done
        return FrameTicket(post_output, done, host_out, frame)

    def _ensure_staging(self, dev) -> None:
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(dev)
            self._pinned_in = [torch.empty((1, self.model.height, self.model.width, 3), dtype=torch.uint8).pin_memory()
                               for _ in range(4)]
            self._slot_free = [torch.cuda.Event() for _ in range(4)]
            self._slot = 0


class FrameTicket:
    """Result handle of StreamDiffusionPipeline.enqueue()."""

    def __init__(self, tensor: torch.Tensor, done: "torch.cuda.Event", host_out: Optional[torch.Tensor], src_frame):
        self._tensor, self._done, self._host_out, self._src = tensor, done, host_out, src_frame

    def done(self) -> bool:
        """True once every GPU operation of this frame (and the download, if any) has finished; never blocks."""
        return self._done.query()

    def wait(self, stream) -> None:
        """Make `stream` wait for this frame (no host synchronisation): later work on it sees the finished tensor."""
        stream.wait_event(self._done)

    def result(self, wait: bool = True):
        """The (1,3,H,W) u8 CUDA tensor (NVENC set) or an av.VideoFrame carrying the input's pts/time_base."""
        if self._host_out is None:
            if wait:
                self._done.synchronize()
            return self._tensor
        try:
            import av
        except ImportError as exc:
            raise RuntimeError("NVENC is unset, so an av.VideoFrame must be returned, but PyAV is not installed; "
                               "set NVENC=1 to receive the CUDA tensor") from exc
        self._done.synchronize()
        hwc = self._host_out.permute(0, 2, 3, 1).squeeze(0).numpy()
        out = av.VideoFrame.from_ndarray(np.ascontiguousarray(hwc))
        out.pts = self._src.pts
        out.time_base = self._src.time_base
        return out
