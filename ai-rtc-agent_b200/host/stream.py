"""`StreamDiffusion` as the reference uses it (imported at lib/wrapper.py:20 from the un-vendored
yondonfu/StreamDiffusion@deepstream), re-implemented over libb200sd.so: the host-side bookkeeping
(LCM timestep table, per-slot scalars, seeded noise, prompt embedding, attributes that
lib/wrapper.py:389-407 pokes at) lives here in Python, everything per-frame runs in the engine.

Supported configuration: img2img, use_denoising_batch=True, frame_buffer_size=1, every cfg_type ("none", "self",
"initialize", "full") at any guidance_scale (lib/pipeline.py:23-42 builds "self" with guidance 0.0, i.e. no guidance)."""
from __future__ import annotations

import ctypes as C
import os
from typing import Callable, Dict, List, Optional

import numpy as np
import torch

from . import capi
from .arch import UNetArch

NUM_TRAIN_TIMESTEPS = 1000
LCM_ORIGINAL_INFERENCE_STEPS = 50
LCM_TIMESTEP_SCALING = 10.0
LCM_SIGMA_DATA = 0.5


# ---- schedule tables (diffusers LCMScheduler with the SD scaled-linear betas) ---------------------------
def scaled_linear_alphas_cumprod(beta_start: float = 0.00085, beta_end: float = 0.012) -> torch.Tensor:
    betas = torch.linspace(beta_start ** 0.5, beta_end ** 0.5, NUM_TRAIN_TIMESTEPS, dtype=torch.float32) ** 2
    return torch.cumprod(1.0 - betas, dim=0)


def lcm_timestep_table(num_inference_steps: int) -> List[int]:
    """LCMScheduler.set_timesteps(N): the 50 'origin' timesteps 19,39,..,999 walked backwards with stride
    50 // N.  N = 50 gives timesteps[i] = 999 - 20 i."""
    stride_train = NUM_TRAIN_TIMESTEPS // LCM_ORIGINAL_INFERENCE_STEPS
    origin = [(i + 1) * stride_train - 1 for i in range(LCM_ORIGINAL_INFERENCE_STEPS)]
    if num_inference_steps > LCM_ORIGINAL_INFERENCE_STEPS:
        raise ValueError("num_inference_steps cannot exceed the 50 LCM origin steps")
    step = LCM_ORIGINAL_INFERENCE_STEPS // num_inference_steps
    return list(reversed(origin))[::step][:num_inference_steps]


def lcm_boundary_scalings(timestep: int):
    scaled = timestep * LCM_TIMESTEP_SCALING
    denom = scaled * scaled + LCM_SIGMA_DATA * LCM_SIGMA_DATA
    return LCM_SIGMA_DATA * LCM_SIGMA_DATA / denom, scaled / denom ** 0.5


def uncond_rows(cfg_type: str, frame_buffer_size: int, batch_size: int) -> int:
    """Unconditional rows a guided UNet batch puts in front of the batch_size text rows (upstream StreamDiffusion.__init__'s
    trt_unet_batch_size): one per frame for "initialize", one per text row for "full", none for "self" / "none"."""
    return {"initialize": frame_buffer_size, "full": batch_size}.get(cfg_type, 0)


class ImageProcessor:
    """The part of diffusers' VaeImageProcessor the reference reaches (lib/wrapper.py:364)."""

    def __init__(self, vae_scale_factor: int = 8):
        self.vae_scale_factor = vae_scale_factor

    def preprocess(self, image, height: Optional[int] = None, width: Optional[int] = None) -> torch.Tensor:
        from PIL import Image
        if isinstance(image, Image.Image):
            if height and width and image.size != (width, height):
                image = image.resize((width, height), Image.LANCZOS)
            arr = np.asarray(image.convert("RGB"), dtype=np.float32) / 255.0
            image = torch.from_numpy(arr).permute(2, 0, 1)
        if isinstance(image, np.ndarray):
            image = torch.from_numpy(image)
        if image.dim() == 3:
            image = image.unsqueeze(0)
        if height and width and (image.shape[-2] != height or image.shape[-1] != width):
            image = torch.nn.functional.interpolate(image, size=(height, width))
        return image if image.min() < 0 else 2.0 * image - 1.0


class StreamDiffusion:
    def __init__(self, arch: UNetArch, unet_sd: Dict[str, torch.Tensor], vae_sd: Dict[str, torch.Tensor],
                 t_index_list: List[int], prompt_encoder: Callable[[str], torch.Tensor],
                 torch_dtype: torch.dtype = torch.float16, width: int = 512, height: int = 512,
                 do_add_noise: bool = True, use_denoising_batch: bool = True, frame_buffer_size: int = 1,
                 cfg_type: str = "self", device: str = "cuda", use_cuda_graph: bool = True,
                 packed_blob: Optional[str] = None, parent: Optional["StreamDiffusion"] = None):
        if frame_buffer_size != 1:
            raise NotImplementedError("frame_buffer_size > 1 is not on the reference's path (lib/pipeline.py:28)")
        if not use_denoising_batch:
            raise NotImplementedError("img2img mode must use denoising batch for now.")
        if torch_dtype != torch.float16:
            raise NotImplementedError("the sm_100a kernels compute in fp16 (fp32 accumulate) like the reference engines")
        self.arch = arch
        self.device = torch.device(device)
        self.dtype = torch_dtype
        self.generator = None
        self.height, self.width = height, width
        self.latent_height, self.latent_width = height // 8, width // 8
        self.frame_bff_size = frame_buffer_size
        self.denoising_steps_num = len(t_index_list)
        self.cfg_type = cfg_type
        self.use_denoising_batch = use_denoising_batch
        self.batch_size = self.denoising_steps_num * frame_buffer_size
        # UNet batch of a guided stream (StreamDiffusion.__init__): initialize adds one unconditional row, full T of them.
        # prepare() sets it to the batch the engine actually runs (T when guidance is off).
        self.trt_unet_batch_size = self.batch_size + uncond_rows(cfg_type, frame_buffer_size, self.batch_size)
        self._uc_rows = 0
        self._uncond: Optional[torch.Tensor] = None
        self.t_list = list(t_index_list)
        self.do_add_noise = do_add_noise
        self.similar_image_filter = False
        self.prev_image_result = None
        self.inference_time_ema = 0.0
        self._ev = None
        self.image_processor = ImageProcessor(8)
        self.prompt_encoder = prompt_encoder
        self.text_encoder = prompt_encoder
        self.unet = self
        self.vae = self
        self._handle = C.c_void_p()
        self._prepared = False
        self._lib = capi.lib()
        cfg = capi.EngineConfig()
        for i in range(4):
            cfg.block_out_channels[i] = arch.block_out_channels[i]
            cfg.heads[i] = arch.heads[i]
            cfg.down_attn[i] = arch.down_attn[i]
        cfg.cross_attention_dim = arch.cross_attention_dim
        cfg.layers_per_block = arch.layers_per_block
        cfg.norm_groups = arch.norm_groups
        cfg.ctx_tokens = arch.ctx_tokens
        cfg.batch = self.batch_size
        cfg.height, cfg.width = height, width
        cfg.do_add_noise = int(do_add_noise)
        cfg.use_cuda_graph = int(use_cuda_graph)
        if not torch.cuda.is_available():
            raise capi.B2Error("no CUDA device: the B200 pipeline has no CPU fallback")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        torch.cuda.set_device(self.device)
        self._ctor = dict(torch_dtype=torch_dtype, width=width, height=height, do_add_noise=do_add_noise,
                          use_denoising_batch=use_denoising_batch, frame_buffer_size=frame_buffer_size, cfg_type=cfg_type,
                          device=device, use_cuda_graph=use_cuda_graph)
        self.lanes: List["StreamDiffusion"] = []     # extra engines over this one's weights (add_lane)
        self._parent = parent
        if parent is not None:
            # a lane: shares the parent's weights in HBM, owns its activations / stream state / CUDA graph
            capi.check(self._lib.b2sd_create_lane(parent._handle, C.byref(cfg), C.byref(self._handle)), "b2sd_create_lane")
            return
        capi.check(self._lib.b2sd_create(C.byref(cfg), C.byref(self._handle)), "b2sd_create")
        if packed_blob is not None:
            # kernel-native weights written by export_packed() / `python -m ai_rtc_agent_b200.pack`: no state dicts, no repacking
            capi.check(self._lib.b2sd_import_packed(self._handle, os.fsencode(packed_blob)), f"b2sd_import_packed({packed_blob})")
        else:
            self._load("", unet_sd)
            self._load("vae.", vae_sd)

    def set_concurrency(self, frames_in_flight: int) -> None:
        """Tell the engine how many frames will be in flight on this GPU (before prepare()): > 1 selects the throughput
        launch policy (b2sd_set_concurrency)."""
        capi.check(self._lib.b2sd_set_concurrency(self._handle, int(frames_in_flight)), "b2sd_set_concurrency")
        self._prepared = False

    def export_packed(self, path: str) -> None:
        """Write the packed-weight blob (after prepare()); the engine-file cache of lib/wrapper.py:593-597, 896-910."""
        self._check()
        tmp = f"{path}.tmp{os.getpid()}"
        capi.check(self._lib.b2sd_export_packed(self._handle, os.fsencode(tmp)), f"b2sd_export_packed({path})")
        os.replace(tmp, path)   # atomic: a concurrently starting replica never sees a half-written blob

    def __del__(self):
        try:
            if getattr(self, "_handle", None) and self._handle.value:
                self._lib.b2sd_destroy(self._handle)
                self._handle = C.c_void_p()
        except Exception:
            pass

    def _load(self, prefix: str, sd: Dict[str, torch.Tensor]) -> None:
        for key, t in sd.items():
            t = t.detach()
            if t.dtype not in (torch.float16, torch.float32):
                t = t.float()
            t = t.contiguous()
            shape = (C.c_int64 * t.dim())(*t.shape)
            capi.check(self._lib.b2sd_load_tensor(self._handle, (prefix + key).encode(), t.data_ptr(),
                                                  0 if t.dtype == torch.float16 else 1, shape, t.dim()),
                       f"b2sd_load_tensor({prefix + key})")

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    # ---- StreamDiffusion.prepare --------------------------------------------------------------------
    @torch.no_grad()
    def prepare(self, prompt: str, negative_prompt: str = "", num_inference_steps: int = 50,
                guidance_scale: float = 1.2, delta: float = 1.0,
                generator: Optional[torch.Generator] = None, seed: int = 2) -> None:
        self.generator = generator if generator is not None else torch.Generator()
        self.generator.manual_seed(seed)
        self.guidance_scale = 1.0 if self.cfg_type == "none" else guidance_scale
        self.delta = delta
        T = self.denoising_steps_num
        guided = self.guidance_scale > 1.0
        cond = self._encode(prompt)
        self._uc_rows = uncond_rows(self.cfg_type, self.frame_bff_size, self.batch_size) if guided else 0
        # residual guidance ("self") needs no negative prompt: its unconditional prediction is delta * stock_noise
        self._uncond = self._encode(negative_prompt) if self._uc_rows else None
        self.trt_unet_batch_size = self.batch_size + self._uc_rows
        # uncond-first layout: initialize [uncond, cond x T], full [uncond x T, cond x T], otherwise [cond x T]
        self.prompt_embeds = self._embeds_rows(cond)
        self.timesteps = lcm_timestep_table(num_inference_steps)
        self.sub_timesteps = [self.timesteps[t] for t in self.t_list]
        self.sub_timesteps_tensor = torch.tensor(self.sub_timesteps, dtype=torch.long, device=self.device)
        self.sub_timesteps_tensor = torch.repeat_interleave(self.sub_timesteps_tensor, repeats=self.frame_bff_size, dim=0)
        self.init_noise = torch.randn((self.batch_size, 4, self.latent_height, self.latent_width),
                                      generator=self.generator).to(dtype=self.dtype)
        self.stock_noise = torch.zeros_like(self.init_noise)
        scal = [lcm_boundary_scalings(t) for t in self.sub_timesteps]
        ac = scaled_linear_alphas_cumprod()
        f16 = lambda v: torch.tensor(v, dtype=torch.float32).to(self.dtype)  # the reference keeps these in fp16
        self.c_skip = f16([s[0] for s in scal]).view(T, 1, 1, 1)
        self.c_out = f16([s[1] for s in scal]).view(T, 1, 1, 1)
        self.alpha_prod_t_sqrt = torch.stack([ac[t].sqrt() for t in self.sub_timesteps]).to(self.dtype).view(T, 1, 1, 1)
        self.beta_prod_t_sqrt = torch.stack([(1 - ac[t]).sqrt() for t in self.sub_timesteps]).to(self.dtype).view(T, 1, 1, 1)
        self._engine_prepare()
        for lane in self.lanes:
            lane._prepare_like(self)

    _SCHEDULE_ATTRS = ("generator", "guidance_scale", "delta", "prompt_embeds", "timesteps", "sub_timesteps", "sub_timesteps_tensor",
                       "init_noise", "stock_noise", "c_skip", "c_out", "alpha_prod_t_sqrt", "beta_prod_t_sqrt", "trt_unet_batch_size",
                       "_uc_rows", "_uncond")

    def _embeds_rows(self, cond: torch.Tensor) -> torch.Tensor:
        rows = cond.repeat(self.batch_size, 1, 1)
        if self._uc_rows:
            rows = torch.cat([self._uncond.repeat(self._uc_rows, 1, 1), rows], dim=0)
        return rows

    def _engine_prepare(self) -> None:
        coef = torch.stack([self.alpha_prod_t_sqrt.flatten(), self.beta_prod_t_sqrt.flatten(),
                            self.c_skip.flatten(), self.c_out.flatten()]).float().contiguous()
        tsteps = torch.tensor(self.sub_timesteps, dtype=torch.float32)
        emb = self.prompt_embeds[self._uc_rows].to(torch.float16).cpu().contiguous()
        noise = self.init_noise.cpu().contiguous()
        unc = self._uncond[0].to(torch.float16).cpu().contiguous() if self._uncond is not None else None
        capi.check(self._lib.b2sd_set_guidance(self._handle, capi.CFG_TYPES[self.cfg_type], float(self.guidance_scale),
                                               float(self.delta), None if unc is None else unc.data_ptr()), "b2sd_set_guidance")
        capi.check(self._lib.b2sd_prepare(self._handle, emb.data_ptr(), tsteps.data_ptr(), coef.data_ptr(),
                                          noise.data_ptr(), self._stream()), "b2sd_prepare")
        self._prepared = True

    def _prepare_like(self, other: "StreamDiffusion") -> None:
        for name in self._SCHEDULE_ATTRS:
            setattr(self, name, getattr(other, name))
        self.t_list = list(other.t_list)
        self._engine_prepare()

    def add_lane(self, share_state: bool = False) -> "StreamDiffusion":
        """Another engine over the same weights, prepared identically (same prompt embedding, schedule and seed-2 noise):
        frames may be alternated between this engine and its lanes on different CUDA streams.  Later prepare() /
        update_prompt() / timestep updates on this object reach every lane.
        share_state=False: the lane is an independent temporal stream (or, for a 1-step stream batch, simply the next frame).
        share_state=True: the lane continues THIS stream -- it shares the stream-batch state and is stage-pipelined with it
        (b2sd_share_stream_state): required for T > 1, where frame n+1 needs frame n's x_t_latent_buffer."""
        self._check()
        lane = StreamDiffusion(self.arch, {}, {}, self.t_list, self.prompt_encoder, parent=self, **self._ctor)
        if share_state:
            capi.check(self._lib.b2sd_share_stream_state(lane._handle, self._handle), "b2sd_share_stream_state")
            self._engine_prepare()          # the owner's frame program is rebuilt as three stages (packed weights are cached)
        lane._prepare_like(self)
        self.lanes.append(lane)
        return lane

    def _encode(self, prompt: str) -> torch.Tensor:
        e = self.prompt_encoder(prompt)
        if e.dim() == 2:
            e = e.unsqueeze(0)
        if e.shape[-2] != self.arch.ctx_tokens or e.shape[-1] != self.arch.cross_attention_dim:
            raise ValueError(f"prompt embedding shape {tuple(e.shape)} != (1,{self.arch.ctx_tokens},{self.arch.cross_attention_dim})")
        return e.to(torch.float16)

    @torch.no_grad()
    def update_prompt(self, prompt: str) -> None:
        """Replaces the conditional rows only.  Upstream StreamDiffusion.update_prompt re-encodes the prompt into batch_size
        rows and so drops the unconditional rows of an initialize / full batch, which then no longer matches the UNet batch;
        here those rows keep the negative prompt of prepare() (a deliberate deviation)."""
        cond = self._encode(prompt)
        self.prompt_embeds = self._embeds_rows(cond)
        emb = cond[0].cpu().contiguous()
        for eng in [self] + self.lanes:
            eng.prompt_embeds = self.prompt_embeds
            capi.check(self._lib.b2sd_set_prompt_embeds(eng._handle, emb.data_ptr(), self._stream()), "b2sd_set_prompt_embeds")

    def sync_timesteps(self) -> None:
        """Push self.sub_timesteps to the engine (called after lib/wrapper.py:389-407 style updates).  As in the
        reference only the timestep embedding changes; alpha/beta/c_skip/c_out keep their prepare() values."""
        t = torch.tensor([float(v) for v in self.sub_timesteps], dtype=torch.float32)
        if t.numel() != self.batch_size:
            raise ValueError(f"t_index_list length {t.numel()} != stream batch {self.batch_size} (static batch, as the "
                             "reference's TensorRT engines)")
        for eng in [self] + self.lanes:
            eng.t_list, eng.sub_timesteps, eng.sub_timesteps_tensor = self.t_list, self.sub_timesteps, self.sub_timesteps_tensor
            capi.check(self._lib.b2sd_set_timesteps(eng._handle, t.data_ptr(), self._stream()), "b2sd_set_timesteps")

    # ---- per frame ---------------------------------------------------------------------------------
    def _check(self):
        if not self._prepared:
            raise RuntimeError("StreamDiffusion.prepare() must be called before frames are processed")

    @torch.no_grad()
    def __call__(self, x: torch.Tensor) -> torch.Tensor:
        """x: (3,H',W') or (1,3,H',W') float tensor in [0,1] on the GPU -> (1,3,H,W) fp16 image in ~[-1,1]."""
        self._check()
        if x.dim() == 3:
            x = x.unsqueeze(0)
        if x.dtype == torch.float32:
            kind = capi.IN_F32_NCHW
        elif x.dtype == torch.float16:
            kind = capi.IN_F16_NCHW
        else:
            raise TypeError(f"unsupported image dtype {x.dtype}")
        x = x.to(self.device)
        # VaeImageProcessor.preprocess (re-run inside the reference's StreamDiffusion.__call__): an image that already has
        # negative values is taken as [-1,1] and NOT normalised again; the encoder's own (x+1)/2 then brings it to [0,1],
        # which is the range the engine's head expects.  Same host sync (`image.min()`) as the reference; the fused u8 entry
        # (step_u8, what lib/pipeline.py's __call__ uses) never comes through here.
        if bool(x.min() < 0):
            x = x * 0.5 + 0.5
        x = x.contiguous()
        out = torch.empty((1, 3, self.height, self.width), dtype=torch.float16, device=self.device)
        t0 = self._tick()
        capi.check(self._lib.b2sd_step_ex(self._handle, x.data_ptr(), kind, x.shape[-2], x.shape[-1], out.data_ptr(),
                                          capi.OUT_F16_NCHW, self._stream()), "b2sd_step_ex")
        self._tock(t0)
        self.prev_image_result = out
        return out

    # ---- inference_time_ema (StreamDiffusion.__call__ times every frame with CUDA events and keeps
    # ema = 0.9 ema + 0.1 dt; external code reads the attribute).  The reference pays a device-wide synchronize per frame for
    # it; here the events are read one frame late, so nothing on the path blocks.
    def _tick(self):
        if self._ev is None:
            self._ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(2)]
            self._ev_pending = None
            self._ev_idx = 0
        if self._ev_pending is not None:
            e0, e1 = self._ev_pending
            if e1.query():
                self.inference_time_ema = 0.9 * self.inference_time_ema + 0.1 * (e0.elapsed_time(e1) / 1000.0)
                self._ev_pending = None
        if self._ev_pending is not None:
            return None            # previous frame still in flight: skip this sample rather than wait
        pair = self._ev[self._ev_idx]
        self._ev_idx ^= 1
        pair[0].record(torch.cuda.current_stream(self.device))
        return pair

    def _tock(self, pair):
        if pair is not None:
            pair[1].record(torch.cuda.current_stream(self.device))
            self._ev_pending = pair

    @torch.no_grad()
    def step_u8(self, frame_nhwc: torch.Tensor) -> torch.Tensor:
        """Fused fast path of lib/pipeline.py:76-96: u8 NHWC (1,H',W',3) CUDA tensor in, u8 NCHW (1,3,H,W) out,
        one engine call, no intermediate tensors."""
        self._check()
        if frame_nhwc.dtype != torch.uint8 or frame_nhwc.dim() != 4 or frame_nhwc.shape[-1] != 3 or not frame_nhwc.is_cuda:
            raise TypeError("expected a CUDA uint8 tensor shaped (1,H,W,3)")
        frame_nhwc = frame_nhwc.contiguous()
        out = torch.empty((1, 3, self.height, self.width), dtype=torch.uint8, device=self.device)
        t0 = self._tick()
        capi.check(self._lib.b2sd_step(self._handle, frame_nhwc.data_ptr(), frame_nhwc.shape[1], frame_nhwc.shape[2],
                                       out.data_ptr(), self._stream()), "b2sd_step")
        self._tock(t0)
        return out

    def step_u8_into(self, frame_nhwc: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
        capi.check(self._lib.b2sd_step(self._handle, frame_nhwc.data_ptr(), frame_nhwc.shape[1], frame_nhwc.shape[2],
                                       out.data_ptr(), self._stream()), "b2sd_step")
        return out

    def get_tensor(self, name: str) -> torch.Tensor:
        """Debug/parity tap of the last step as an fp16 NHWC CPU tensor."""
        n = C.c_int64()
        dims = (C.c_int * 4)()
        capi.check(self._lib.b2sd_get_tensor(self._handle, name.encode(), None, 0, C.byref(n), dims, self._stream()),
                   "b2sd_get_tensor")
        t = torch.empty(tuple(dims), dtype=torch.float16)
        capi.check(self._lib.b2sd_get_tensor(self._handle, name.encode(), t.data_ptr(), n.value, C.byref(n), dims,
                                             self._stream()), "b2sd_get_tensor")
        return t

    def profile(self, frame_nhwc: torch.Tensor, iters: int = 5):
        """Per-launch device times of one frame (eager replay, CUDA events): list of {"name", "ms"}."""
        import json
        self._check()
        out = torch.empty((1, 3, self.height, self.width), dtype=torch.uint8, device=self.device)
        buf = C.create_string_buffer(1 << 20)
        capi.check(self._lib.b2sd_profile(self._handle, frame_nhwc.data_ptr(), frame_nhwc.shape[1], frame_nhwc.shape[2],
                                          out.data_ptr(), iters, buf, len(buf), self._stream()), "b2sd_profile")
        return json.loads(buf.value.decode())

    def profile_kind(self, kind: str, iters: int = 20):
        """Device time of one launch class inside a CUDA graph (only those launches, program order):
        {"ms": per replay, "launches": n, "flops": algorithmic FLOPs per replay}."""
        self._check()
        ms, n, fl = C.c_double(), C.c_int(), C.c_double()
        capi.check(self._lib.b2sd_profile_kind(self._handle, kind.encode(), iters, C.byref(ms), C.byref(n), C.byref(fl),
                                               self._stream()), "b2sd_profile_kind")
        return {"ms": ms.value, "launches": n.value, "flops": fl.value}

    @property
    def launches_per_step(self) -> int:
        return self._lib.b2sd_launches_per_step(self._handle)
