"""Classifier-free guidance (cfg_type none / self / initialize / full) without a GPU: the guided oracle (tests/cfg_oracle.py)
against a literal transcription of upstream StreamDiffusion's prepare / predict_x0_batch / unet_step over a stub UNet, the
unguided path left bit for bit as it was, the committed cfg fixtures, the wrapper's validation and the contraction plans of
a guided UNet batch."""
import os

import numpy as np
import pytest
import torch

from oracle import pipeline as opipe
from oracle import stream as ostream
from oracle import unet as ounet
from oracle import weights as ow
from tests.cfg_oracle import CfgStreamOracle

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
LAT = 8   # latent extent of the stub cases


def stub_unet(sd, cfg, x, t, ctx, taps=None):
    """Depends on each row's input, timestep and context, so a wrong row order or context assignment shows."""
    tt = t.to(x.dtype).view(-1, 1, 1, 1)
    c = ctx.mean(dim=(1, 2)).view(-1, 1, 1, 1) + ctx[:, :4, 0].reshape(-1, 4, 1, 1)
    return 0.6 * x * (1.0 + tt / 1000.0) + 0.3 * torch.sin(3.0 * x + tt / 100.0) + 0.5 * c


class Upstream:
    """streamdiffusion.StreamDiffusion (img2img, use_denoising_batch, frame_buffer_size 1) written out with torch.cat / chunk
    the way upstream states it.  update_prompt keeps the uncond rows (the project's documented deviation)."""

    def __init__(self, T, cfg_type, unet):
        self.T, self.cfg_type, self.unet = T, cfg_type, unet
        self.denoising_steps_num, self.frame_bff_size, self.batch_size = T, 1, T

    def prepare(self, cond, uncond, g, delta, init_noise, sub_timesteps, alpha, beta, c_skip, c_out):
        self.guidance_scale, self.delta = g, delta
        if self.cfg_type == "none":
            self.guidance_scale = 1.0
        self.prompt_embeds = cond.repeat(self.batch_size, 1, 1)
        if self.cfg_type == "full":
            uncond_prompt_embeds = uncond.repeat(self.batch_size, 1, 1)
        elif self.cfg_type == "initialize":
            uncond_prompt_embeds = uncond.repeat(self.frame_bff_size, 1, 1)
        if self.guidance_scale > 1.0 and self.cfg_type in ("initialize", "full"):
            self.prompt_embeds = torch.cat([uncond_prompt_embeds, self.prompt_embeds], dim=0)
        self.x_t_latent_buffer = torch.zeros_like(init_noise[1:]) if self.T > 1 else None
        self.init_noise = init_noise
        self.stock_noise = torch.zeros_like(init_noise)
        self.sub_timesteps_tensor = torch.tensor(sub_timesteps)
        self.alpha_prod_t_sqrt, self.beta_prod_t_sqrt, self.c_skip, self.c_out = alpha, beta, c_skip, c_out

    def update_prompt(self, cond):
        uc = self.prompt_embeds.shape[0] - self.batch_size
        self.prompt_embeds = torch.cat([self.prompt_embeds[:uc], cond.repeat(self.batch_size, 1, 1)], dim=0)

    def scheduler_step_batch(self, model_pred_batch, x_t_latent_batch):
        F_theta = (x_t_latent_batch - self.beta_prod_t_sqrt * model_pred_batch) / self.alpha_prod_t_sqrt
        return self.c_out * F_theta + self.c_skip * x_t_latent_batch

    def unet_step(self, x_t_latent, t_list):
        if self.guidance_scale > 1.0 and (self.cfg_type == "initialize"):
            x_t_latent_plus_uc = torch.concat([x_t_latent[0:1], x_t_latent], dim=0)
            t_list = torch.concat([t_list[0:1], t_list], dim=0)
        elif self.guidance_scale > 1.0 and (self.cfg_type == "full"):
            x_t_latent_plus_uc = torch.concat([x_t_latent, x_t_latent], dim=0)
            t_list = torch.concat([t_list, t_list], dim=0)
        else:
            x_t_latent_plus_uc = x_t_latent
        model_pred = self.unet(None, None, x_t_latent_plus_uc, t_list, self.prompt_embeds)
        self.model_pred = model_pred
        if self.guidance_scale > 1.0 and (self.cfg_type == "initialize"):
            noise_pred_text = model_pred[1:]
            self.stock_noise = torch.concat([model_pred[0:1], self.stock_noise[1:]], dim=0)
        elif self.guidance_scale > 1.0 and (self.cfg_type == "full"):
            noise_pred_uncond, noise_pred_text = model_pred.chunk(2)
        else:
            noise_pred_text = model_pred
        if self.guidance_scale > 1.0 and (self.cfg_type == "self" or self.cfg_type == "initialize"):
            noise_pred_uncond = self.stock_noise * self.delta
        if self.guidance_scale > 1.0 and self.cfg_type != "none":
            model_pred = noise_pred_uncond + self.guidance_scale * (noise_pred_text - noise_pred_uncond)
        else:
            model_pred = noise_pred_text
        denoised_batch = self.scheduler_step_batch(model_pred, x_t_latent)
        if self.guidance_scale > 1.0 and (self.cfg_type == "self" or self.cfg_type == "initialize"):
            scaled_noise = self.beta_prod_t_sqrt * self.stock_noise
            delta_x = self.scheduler_step_batch(model_pred, scaled_noise)
            alpha_next = torch.concat([self.alpha_prod_t_sqrt[1:], torch.ones_like(self.alpha_prod_t_sqrt[0:1])], dim=0)
            delta_x = alpha_next * delta_x
            beta_next = torch.concat([self.beta_prod_t_sqrt[1:], torch.ones_like(self.beta_prod_t_sqrt[0:1])], dim=0)
            delta_x = delta_x / beta_next
            init_noise = torch.concat([self.init_noise[1:], self.init_noise[0:1]], dim=0)
            self.stock_noise = init_noise + delta_x
        return denoised_batch, model_pred

    def predict_x0_batch(self, x_t_latent):
        prev_latent_batch = self.x_t_latent_buffer
        if self.denoising_steps_num > 1:
            x_t_latent = torch.cat((x_t_latent, prev_latent_batch), dim=0)
            self.stock_noise = torch.cat((self.init_noise[0:1], self.stock_noise[:-1]), dim=0)
        x_0_pred_batch, model_pred = self.unet_step(x_t_latent, self.sub_timesteps_tensor)
        if self.denoising_steps_num > 1:
            x_0_pred_out = x_0_pred_batch[-1].unsqueeze(0)
            self.x_t_latent_buffer = (self.alpha_prod_t_sqrt[1:] * x_0_pred_batch[:-1]
                                      + self.beta_prod_t_sqrt[1:] * self.init_noise[1:])
        else:
            x_0_pred_out = x_0_pred_batch
            self.x_t_latent_buffer = None
        return x_0_pred_out


def _pair(cfg_type, T, g, delta, monkeypatch):
    monkeypatch.setattr(ostream.unet, "unet_forward", stub_unet)
    t_list = [18, 26, 35, 45][:T] if T > 1 else [32]
    orc = CfgStreamOracle({}, None, {}, t_list, LAT * 8, LAT * 8, cfg_type=cfg_type)
    gen = torch.Generator().manual_seed(11)
    cond, uncond = torch.randn(1, 77, 16, generator=gen), torch.randn(1, 77, 16, generator=gen)
    orc.prepare(cond, guidance_scale=g, delta=delta, seed=3, uncond_embeds=uncond)
    up = Upstream(T, cfg_type, stub_unet)
    up.prepare(cond, uncond, g, delta, orc.init_noise.clone(), orc.sub_timesteps, orc.alpha_prod_t_sqrt, orc.beta_prod_t_sqrt,
               orc.c_skip, orc.c_out)
    return orc, up, gen


@pytest.mark.parametrize("delta", [0.5, 1.0])
@pytest.mark.parametrize("g", [1.0, 1.5])
@pytest.mark.parametrize("T", [1, 2, 4])
@pytest.mark.parametrize("cfg_type", ["none", "self", "initialize", "full"])
def test_oracle_matches_upstream_transcription(cfg_type, T, g, delta, monkeypatch):
    orc, up, gen = _pair(cfg_type, T, g, delta, monkeypatch)
    assert torch.equal(orc.prompt_embeds, up.prompt_embeds)
    for f in range(5):
        if f == 3:
            new = torch.randn(1, 77, 16, generator=gen)
            orc.update_prompt_embeds(new)
            up.update_prompt(new)
            assert torch.equal(orc.prompt_embeds, up.prompt_embeds)
        x_t = torch.randn(1, 4, LAT, LAT, generator=gen)
        got, ref = orc.predict_x0_batch(x_t), up.predict_x0_batch(x_t)
        assert torch.allclose(got, ref, rtol=1e-5, atol=1e-5), f"x0 frame {f}"
        assert torch.allclose(orc.last["eps"], up.model_pred, rtol=1e-6, atol=1e-6), f"eps frame {f}"
        assert torch.allclose(orc.stock_noise, up.stock_noise, rtol=1e-5, atol=1e-5), f"stock_noise frame {f}"
        if T > 1:
            assert torch.allclose(orc.x_t_latent_buffer, up.x_t_latent_buffer, rtol=1e-5, atol=1e-5), f"buffer frame {f}"
    rows = {"initialize": T + 1, "full": 2 * T}.get(cfg_type, T) if g > 1 and cfg_type != "none" else T
    assert orc.last["eps"].shape[0] == rows and orc.prompt_embeds.shape[0] == rows


def test_guided_self_is_stateful_and_initialize_t1_is_not(monkeypatch):
    """Residual guidance carries stock noise across frames even at T = 1; initialize at T = 1 overwrites it before use."""
    for cfg_type, stateful in (("self", True), ("initialize", False), ("full", False)):
        orc, _, gen = _pair(cfg_type, 1, 1.5, 1.0, monkeypatch)
        x_a, x_b = torch.randn(1, 4, LAT, LAT, generator=gen), torch.randn(1, 4, LAT, LAT, generator=gen)
        fresh = orc.predict_x0_batch(x_b).clone()
        orc2, _, _ = _pair(cfg_type, 1, 1.5, 1.0, monkeypatch)
        orc2.predict_x0_batch(x_a)
        after = orc2.predict_x0_batch(x_b)
        assert torch.equal(fresh, after) != stateful, cfg_type


@pytest.mark.parametrize("cfg_type", ["none", "self", "initialize", "full"])
@pytest.mark.parametrize("g", [0.0, 1.0])
def test_unguided_oracle_is_unchanged(cfg_type, g):
    """guidance_scale <= 1: every cfg_type computes what cfg_type "none" computes, bit for bit, and matches the fixture."""
    cfg = ounet.tiny_config(True)
    usd, vsd = ow.to_float(ow.make_unet_weights(cfg)), ow.to_float(ow.make_taesd_weights())
    emb = ow.make_prompt_embeds(cfg.cross_attention_dim).float()
    neg = ow.make_prompt_embeds(cfg.cross_attention_dim, seed=7).float()
    gold = np.load(os.path.join(GOLDEN, "tiny_turbo_T2.npz"))
    runs = []
    for ct in ("none", cfg_type):
        orc = CfgStreamOracle(usd, cfg, vsd, [20, 40], 128, 128, cfg_type=ct)
        orc.prepare(emb, guidance_scale=g, seed=2, uncond_embeds=neg)
        orc.init_noise = orc.init_noise.half().float()
        outs = []
        for i in range(2):
            outs += [opipe.frame_to_u8(orc, ow.make_frame(128, 128, seed=i)), orc.last["eps"].clone()]
        runs.append(outs)
    for a, b in zip(*runs):
        assert torch.equal(a, b)
    for i in range(2):
        d = np.abs(runs[1][2 * i].numpy().astype(np.int32) - gold["u8"][i:i + 1].astype(np.int32))
        assert d.max() <= 1 and (d > 0).mean() < 1e-3


CFG_CASES = [("cfg_tiny_sd15_T4_self", False, [18, 26, 35, 45], "self"),
             ("cfg_tiny_sd15_T4_initialize", False, [18, 26, 35, 45], "initialize"),
             ("cfg_tiny_sd15_T4_full", False, [18, 26, 35, 45], "full"),
             ("cfg_tiny_turbo_T1_self", True, [32], "self"),
             ("cfg_tiny_turbo_T2_initialize", True, [20, 40], "initialize")]


@pytest.mark.parametrize("name,turbo,tl,cfg_type", CFG_CASES)
def test_oracle_reproduces_cfg_golden(name, turbo, tl, cfg_type):
    path = os.path.join(GOLDEN, name + ".npz")
    assert os.path.getsize(path) < 1 << 20
    gold = np.load(path)
    cfg = ounet.tiny_config(turbo)
    orc = CfgStreamOracle(ow.to_float(ow.make_unet_weights(cfg)), cfg, ow.to_float(ow.make_taesd_weights()), tl, 128, 128,
                          cfg_type=cfg_type)
    orc.prepare(ow.make_prompt_embeds(cfg.cross_attention_dim).float(), guidance_scale=float(gold["guidance_scale"]),
                delta=float(gold["delta"]), seed=2, uncond_embeds=ow.make_prompt_embeds(cfg.cross_attention_dim, seed=7).float())
    orc.init_noise = orc.init_noise.half().float()
    assert list(gold["sub_timesteps"]) == orc.sub_timesteps
    for i in range(3):
        u8 = opipe.frame_to_u8(orc, ow.make_frame(128, 128, seed=i)).numpy()
        d = np.abs(u8.astype(np.int32) - gold["u8"][i:i + 1].astype(np.int32))
        assert d.max() <= 1 and (d > 0).mean() < 1e-3, f"{name} frame {i}: max {d.max()}"
        assert np.allclose(orc.last["eps"].numpy(), gold["eps"][i].astype(np.float32), rtol=2e-3, atol=2e-3)
        assert np.allclose(orc.stock_noise.numpy(), gold["stock_noise"][i].astype(np.float32), rtol=2e-3, atol=2e-3)


@pytest.mark.parametrize("cfg_type", ["initialize", "full"])
def test_wrapper_accepts_initialize_and_full(cfg_type):
    from ai_rtc_agent_b200.host.wrapper import StreamDiffusionWrapper
    with pytest.raises(FileNotFoundError):
        StreamDiffusionWrapper("no/such-model", [1], cfg_type=cfg_type)
    with pytest.raises(ValueError, match="txt2img"):
        StreamDiffusionWrapper("no/such-model", [1], mode="txt2img", cfg_type=cfg_type)


@pytest.mark.parametrize("hw", [512, 768])
@pytest.mark.parametrize("bu", [5, 8])
def test_plans_of_a_guided_unet_batch(bu, hw):
    """Every contraction of the SD-1.5 / SD-Turbo UNets at UNet batch 5 (T = 4, initialize) and 8 (T = 4, full), plus the
    per-row cross-attention K / V^T GEMMs of the prompt program (B_u contexts of 128 rows)."""
    from tests.test_plan import _check, _desc, _plan, _unet_shapes
    latent = hw // 8
    for policy in (1, 2):
        for (b, r, srcs, cout, stride, geglu, allow_swap) in _unet_shapes([320, 640, 1280, 1280], bu, latent):
            d, kb = _desc(b, r, r, srcs, cout, stride=stride, geglu=geglu)
            _check(_plan(d, policy, int(allow_swap)), d, kb, geglu, pairs_ok=policy == 2)
        for D in (768, 1024):
            for Cp in (320, 640, 1280):
                rows = bu * 128
                d, kb = _desc(1, 1, rows, [(D, 1)], Cp)            # K: [B_u*Lpad][Cp]
                _check(_plan(d, policy, 0), d, kb, pairs_ok=policy == 2)
                d, kb = _desc(1, 1, Cp, [(D, 1)], rows)            # V^T: [Cp][B_u*Lpad]
                _check(_plan(d, policy, 0), d, kb, pairs_ok=policy == 2)
