"""Drop-in for the reference's `lib/wrapper.py:StreamDiffusionWrapper` (lib/wrapper.py:34-407): same
constructor keywords and defaults, same validation errors, same methods and externally-read attributes,
with the TensorRT/diffusers model behind it replaced by the sm_100a engine (host/stream.py).

Not carried over (unreachable from lib/pipeline.py:23-42 and listed out-of-scope in SURVEY.md section 8):
ControlNet, safety checker, similar-image filter, DataParallel, txt2img sampling, xformers/sfast/TensorRT
acceleration switches.  Their keywords are accepted; asking for one of those features raises."""
from __future__ import annotations

import logging
from pathlib import Path
from typing import Dict, List, Literal, Optional, Union

import numpy as np
import torch
from PIL import Image

from .prompt import make_prompt_encoder
from .stream import StreamDiffusion, uncond_rows
from .weights import resolve_weights

logger = logging.getLogger(__name__)

torch.set_grad_enabled(False)


class CudaStreamPtr:
    """lib/wrapper.py:29-31: carrier for an externally owned CUDA stream handle."""

    def __init__(self, cuda_stream_handle):
        self.ptr = cuda_stream_handle


def postprocess_image(image: torch.Tensor, output_type: str = "pil"):
    """streamdiffusion.image_utils.postprocess_image: per-sample denormalise to [0,1] then convert."""
    imgs = torch.stack([(img / 2 + 0.5).clamp(0, 1) for img in image])
    if output_type == "latent":
        return image
    if output_type == "pt":
        return imgs
    arr = imgs.float().cpu().permute(0, 2, 3, 1).numpy()
    if output_type == "np":
        return arr
    if output_type == "pil":
        return [Image.fromarray((a * 255).round().astype("uint8")) for a in arr]
    raise ValueError(f"unknown output_type {output_type}")


class StreamDiffusionWrapper:
    def __init__(
        self,
        model_id_or_path: str,
        t_index_list: List[int],
        controlnet_id_or_path: Optional[str] = None,
        controlnet_processor_id: Optional[str] = "hed",
        lora_dict: Optional[Dict[str, float]] = None,
        mode: Literal["img2img", "txt2img"] = "img2img",
        output_type: Literal["pil", "pt", "np", "latent"] = "pil",
        lcm_lora_id: Optional[str] = None,
        vae_id: Optional[str] = None,
        device: Literal["cpu", "cuda"] = "cuda",
        dtype: torch.dtype = torch.float16,
        frame_buffer_size: int = 1,
        width: int = 512,
        height: int = 512,
        warmup: int = 10,
        acceleration: Literal["none", "xformers", "tensorrt"] = "tensorrt",
        do_add_noise: bool = True,
        device_ids: Optional[List[int]] = None,
        use_lcm_lora: bool = True,
        use_tiny_vae: bool = True,
        enable_similar_image_filter: bool = False,
        similar_image_filter_threshold: float = 0.98,
        similar_image_filter_max_skip_frame: int = 10,
        use_denoising_batch: bool = True,
        cfg_type: Literal["none", "full", "self", "initialize"] = "self",
        seed: int = 2,
        use_safety_checker: bool = False,
        engine_dir: Optional[Union[str, Path]] = "engines",
        cuda_stream_handle: Optional[int] = None,
    ):
        self.sd_turbo = "turbo" in model_id_or_path

        # the reference's argument validation (lib/wrapper.py:135-150), same exception types
        if mode == "txt2img":
            if cfg_type != "none":
                raise ValueError(f"txt2img mode accepts only cfg_type = 'none', but got {cfg_type}")
            if use_denoising_batch and frame_buffer_size > 1 and not self.sd_turbo:
                raise ValueError("txt2img mode cannot use denoising batch with frame_buffer_size > 1.")
        if mode == "img2img" and not use_denoising_batch:
            raise NotImplementedError("img2img mode must use denoising batch for now.")

        unsupported = []
        if mode == "txt2img":
            unsupported.append("mode='txt2img'")
        if controlnet_id_or_path is not None:
            unsupported.append("controlnet")
        if use_safety_checker:
            unsupported.append("safety checker")
        if enable_similar_image_filter:
            unsupported.append("similar-image filter")
        if device_ids is not None:
            unsupported.append("DataParallel device_ids (shard streams across GPUs instead, see host/dist.py)")
        if not use_tiny_vae:
            unsupported.append("full AutoencoderKL (only TAESD is on the reference's path)")
        if device != "cuda":
            unsupported.append("device='cpu' (no CPU fallback)")
        if unsupported:
            raise NotImplementedError("not on the hot path this library implements: " + ", ".join(unsupported))

        self.device = device
        self.dtype = dtype
        self.width = width
        self.height = height
        self.mode = mode
        self.output_type = output_type
        self.frame_buffer_size = frame_buffer_size
        self.batch_size = len(t_index_list) * frame_buffer_size if use_denoising_batch else frame_buffer_size
        self.use_denoising_batch = use_denoising_batch
        self.use_safety_checker = use_safety_checker
        self.engine_dir = engine_dir
        self.packed_blob = None
        self._blob_to_write = None
        self.cuda_stream = CudaStreamPtr(cuda_stream_handle) if cuda_stream_handle is not None else None
        self._ext_stream = (torch.cuda.ExternalStream(cuda_stream_handle) if cuda_stream_handle is not None else None)

        self.stream: StreamDiffusion = self._load_model(
            model_id_or_path=model_id_or_path, lora_dict=lora_dict, lcm_lora_id=lcm_lora_id, vae_id=vae_id,
            t_index_list=t_index_list, do_add_noise=do_add_noise, use_lcm_lora=use_lcm_lora, cfg_type=cfg_type)

    # -- model loading: replaces _load_trt_model/_load_model (lib/wrapper.py:409-944) --------------------
    def _load_model(self, model_id_or_path, lora_dict, lcm_lora_id, vae_id, t_index_list, do_add_noise,
                    use_lcm_lora, cfg_type) -> StreamDiffusion:
        """Like the reference (lib/wrapper.py:583-615): first try the cached artefact under `engine_dir` -- there TensorRT engine
        files, here the packed-weight blob -- and on any failure fall through to the full path (load weights, fuse LoRAs),
        after which the blob is written for the next start (lib/wrapper.py:889-910 moves the engines into the cache)."""
        import os
        from . import arch as A
        from . import weights as W
        synthetic_ok = bool(os.getenv(W.ALLOW_SYNTHETIC_ENV)) or model_id_or_path.startswith(("tiny", "synthetic"))
        repo = W.find_local_repo(model_id_or_path)
        have_ckpt = repo is not None and os.path.isdir(os.path.join(repo, "unet"))
        arch = A.arch_for(model_id_or_path)
        kw = dict(torch_dtype=self.dtype, width=self.width, height=self.height, do_add_noise=do_add_noise,
                  use_denoising_batch=self.use_denoising_batch, frame_buffer_size=self.frame_buffer_size, cfg_type=cfg_type,
                  device=self.device)
        blob = None
        # blobs are kept for real checkpoints; seeded synthetic weights (benchmarks, tests) only with B200SD_PACK_CACHE=synthetic
        mode = os.getenv("B200SD_PACK_CACHE", "1")
        use_cache = self.engine_dir is not None and mode != "0" and model_id_or_path not in W._PRELOADED and \
            (have_ckpt or mode == "synthetic")
        if use_cache:
            blob = W.packed_blob_path(self.engine_dir, model_id_or_path, arch.name, use_lcm_lora and not self.sd_turbo, lcm_lora_id,
                                      lora_dict, vae_id, synthetic=not have_ckpt,
                                      variant=W.layout_variant(self._unet_batch(cfg_type), self.height, self.width))
        encoder = make_prompt_encoder(repo if have_ckpt else None, arch.cross_attention_dim, self.device, allow_synthetic=synthetic_ok)
        if blob is not None and os.path.exists(blob) and (have_ckpt or synthetic_ok):
            try:
                sd = StreamDiffusion(arch, {}, {}, t_index_list, encoder, packed_blob=blob, **kw)
                logger.info("loaded packed weights from %s", blob)
                self.packed_blob = blob
                return sd
            except Exception as exc:   # noqa: BLE001 - same policy as lib/wrapper.py:611-615
                logger.warning("packed-weight blob %s unusable (%s); rebuilding from the checkpoint", blob, exc)
        arch, unet_sd, vae_sd, repo = resolve_weights(model_id_or_path, vae_id, lcm_lora_id, use_lcm_lora, lora_dict,
                                                      self.sd_turbo)
        self._blob_to_write = blob
        return StreamDiffusion(arch, unet_sd, vae_sd, t_index_list, encoder, **kw)

    def _unet_batch(self, cfg_type: str) -> int:
        """UNet batch of a guided stream: initialize adds one unconditional row per frame, full one per stream-batch row.  The
        packed layout is chosen for it (those cfg types are used with guidance_scale > 1)."""
        return self.batch_size + uncond_rows(cfg_type, self.frame_buffer_size, self.batch_size)

    def _on_stream(self):
        return torch.cuda.stream(self._ext_stream) if self._ext_stream is not None else _NullCtx()

    def prepare(self, prompt: str, negative_prompt: str = "", t_index_list: List[int] = None,
                num_inference_steps: int = 50, guidance_scale: float = 1.2, delta: float = 1.0) -> None:
        if t_index_list is not None:
            if len(t_index_list) != len(self.stream.t_list):
                raise Exception(
                    f"new and current t_index_list length do not match: {len(t_index_list)} != {len(self.stream.t_list)}")
            self.stream.t_list = t_index_list
        with self._on_stream():
            self.stream.prepare(prompt, negative_prompt, num_inference_steps=num_inference_steps,
                                guidance_scale=guidance_scale, delta=delta)
        if self._blob_to_write is not None:
            # first start from a checkpoint: leave the packed blob behind (the reference moves its freshly built engines into
            # the cache directory, lib/wrapper.py:889-910); failures only cost the next start its speed-up
            import os
            try:
                os.makedirs(os.path.dirname(self._blob_to_write), exist_ok=True)
                self.stream.export_packed(self._blob_to_write)
                self.packed_blob = self._blob_to_write
                logger.info("wrote packed weights to %s", self._blob_to_write)
            except Exception as exc:   # noqa: BLE001
                logger.warning("could not write the packed-weight blob %s: %s", self._blob_to_write, exc)
            self._blob_to_write = None

    def __call__(self, image=None, prompt: Optional[str] = None, t_index_list: Optional[List[int]] = None):
        if self.mode == "img2img":
            return self.img2img(image, prompt, t_index_list)
        return self.txt2img(prompt, t_index_list)

    def txt2img(self, prompt: Optional[str] = None, t_index_list: Optional[List[int]] = None):
        raise NotImplementedError("txt2img is not on the reference's per-frame path (lib/pipeline.py:31)")

    def img2img(self, image, prompt: Optional[str] = None, t_index_list: Optional[List[int]] = None):
        if prompt is not None:
            self.stream.update_prompt(prompt)
        if t_index_list is not None:
            self.update_t_index_list(t_index_list)
        if isinstance(image, (str, Image.Image)):
            image = self.preprocess_image(image)
        with self._on_stream():
            image_tensor = self.stream(image)
        return self.postprocess_image(image_tensor, output_type=self.output_type)

    def preprocess_image(self, image: Union[str, Image.Image]) -> torch.Tensor:
        if isinstance(image, str):
            image = Image.open(image)
        image = image.convert("RGB").resize((self.width, self.height))
        return self.stream.image_processor.preprocess(image, self.height, self.width).to(device=self.device,
                                                                                         dtype=self.dtype)

    def postprocess_image(self, image_tensor: torch.Tensor, output_type: str = "pil"):
        out = postprocess_image(image_tensor, output_type=output_type)
        return out if self.frame_buffer_size > 1 else out[0]

    def update_t_index_list(self, t_index_list: List[int]) -> None:
        """lib/wrapper.py:389-407: swaps the sub-timesteps only."""
        if t_index_list == self.stream.t_list:
            return
        s = self.stream
        s.t_list = t_index_list
        s.sub_timesteps = [s.timesteps[t] for t in t_index_list]
        tt = torch.tensor(s.sub_timesteps, dtype=torch.long, device=self.device)
        s.sub_timesteps_tensor = torch.repeat_interleave(tt, repeats=s.frame_bff_size if s.use_denoising_batch else 1, dim=0)
        s.sync_timesteps()


class _NullCtx:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False
