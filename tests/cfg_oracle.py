"""fp32 restatement of StreamDiffusion's classifier-free guidance (upstream streamdiffusion/pipeline.py: prepare,
predict_x0_batch, unet_step for cfg_type "self" / "initialize" / "full") on top of oracle.stream.StreamOracle, which
restates the unguided path.  With guidance_scale <= 1 or cfg_type "none" everything is StreamOracle's own code.

Semantics (T = stream batch, g = guidance_scale, guidance active when g > 1 and cfg_type != "none"):
  prepare      prompt_embeds uncond first: initialize [uncond, cond x T], full [uncond x T, cond x T], self [cond x T]
  UNet input   initialize cat(x[0:1], x), t likewise; full cat(x, x); self x
  guidance     initialize: stock[0] = eps[0], eps_text = eps[1:];  full: eps_uncond, eps_text = eps.chunk(2)
               self / initialize: eps_uncond = delta * stock;  model_pred = eps_uncond + g (eps_text - eps_uncond)
  stock noise  self / initialize: roll(init_noise, -1) + scheduler_step(model_pred, beta * stock) * alpha_next / beta_next
update_prompt_embeds keeps the uncond rows (upstream drops them and breaks the initialize / full batch: deliberate
deviation).  Test infrastructure only."""
from __future__ import annotations

from typing import Dict, List, Optional

import torch

from oracle import stream as ostream
from oracle import unet as ounet


class CfgStreamOracle(ostream.StreamOracle):
    def prepare(self, prompt_embeds: torch.Tensor, num_inference_steps: int = 50, guidance_scale: float = 1.2,
                delta: float = 1.0, seed: int = 2, init_noise: Optional[torch.Tensor] = None,
                uncond_embeds: Optional[torch.Tensor] = None) -> None:
        """uncond_embeds: the encoded negative prompt (1,77,D), needed by initialize / full with guidance_scale > 1."""
        super().prepare(prompt_embeds, num_inference_steps, guidance_scale, delta, seed, init_noise)
        if self.guided and self.cfg_type in ("initialize", "full"):
            if uncond_embeds is None:
                raise ValueError(f"cfg_type {self.cfg_type!r} with guidance_scale > 1 needs uncond_embeds")
            rows = self.frame_bff_size if self.cfg_type == "initialize" else self.batch_size
            unc = uncond_embeds.float().reshape(1, uncond_embeds.shape[-2], -1).repeat(rows, 1, 1)
            self.prompt_embeds = torch.cat([unc, self.prompt_embeds], 0)

    @property
    def guided(self) -> bool:
        return self.guidance_scale > 1.0 and self.cfg_type != "none"

    def update_prompt_embeds(self, prompt_embeds: torch.Tensor) -> None:
        uc = self.prompt_embeds.shape[0] - self.batch_size
        unc = self.prompt_embeds[:uc]
        super().update_prompt_embeds(prompt_embeds)
        if uc > 0:
            self.prompt_embeds = torch.cat([unc, self.prompt_embeds], 0)

    def unet_step(self, x: torch.Tensor):
        """Returns (x0_batch, eps of every UNet row)."""
        if not self.guided:
            return super().unet_step(x)
        g, cfg, t = self.guidance_scale, self.cfg_type, self.sub_timesteps_tensor
        if cfg == "initialize":
            x_in, t_in = torch.cat([x[0:1], x], 0), torch.cat([t[0:1], t], 0)
        elif cfg == "full":
            x_in, t_in = torch.cat([x, x], 0), torch.cat([t, t], 0)
        else:
            x_in, t_in = x, t
        eps = ostream.unet.unet_forward(self.unet_sd, self.cfg, x_in, t_in, self.prompt_embeds)
        if cfg == "initialize":
            eps_text = eps[1:]
            self.stock_noise = torch.cat([eps[0:1], self.stock_noise[1:]], 0)
        elif cfg == "full":
            eps_uncond, eps_text = eps.chunk(2)
        else:
            eps_text = eps
        if cfg in ("self", "initialize"):
            eps_uncond = self.stock_noise * self.delta
        model_pred = eps_uncond + g * (eps_text - eps_uncond)
        x0 = self.scheduler_step_batch(model_pred, x)
        if cfg in ("self", "initialize"):
            delta_x = self.scheduler_step_batch(model_pred, self.beta_prod_t_sqrt * self.stock_noise)
            one = torch.ones_like(self.alpha_prod_t_sqrt[0:1])
            a_next = torch.cat([self.alpha_prod_t_sqrt[1:], one], 0)
            b_next = torch.cat([self.beta_prod_t_sqrt[1:], one], 0)
            self.stock_noise = torch.cat([self.init_noise[1:], self.init_noise[0:1]], 0) + a_next * delta_x / b_next
        return x0, eps


def build_gpu(cfg: ounet.UNetConfig, unet_sd16: Dict[str, torch.Tensor], vae_sd16: Dict[str, torch.Tensor],
              t_index_list: List[int], hw: int, prompt_embeds: torch.Tensor, init_noise: torch.Tensor, cfg_type: str,
              guidance_scale: float, delta: float = 1.0, uncond_embeds: Optional[torch.Tensor] = None,
              dtype: torch.dtype = torch.float32, device: str = "cuda") -> CfgStreamOracle:
    """oracle.torch_gpu.build with guidance: the restatement on the GPU through torch's library kernels (TF32 off)."""
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    orc = CfgStreamOracle({k: v.float() for k, v in unet_sd16.items()}, cfg, {k: v.float() for k, v in vae_sd16.items()},
                          t_index_list, hw, hw, cfg_type=cfg_type)
    orc.prepare(prompt_embeds.float(), guidance_scale=guidance_scale, delta=delta, init_noise=init_noise.float(),
                uncond_embeds=None if uncond_embeds is None else uncond_embeds.float())
    return orc.to(device, dtype)
