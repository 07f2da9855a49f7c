"""Classifier-free guidance on the B200: the fused scheduler kernel (b2sd_op_lcm_cfg_step) against a torch fp32 restatement,
the engine against the committed cfg fixtures (tests/golden/make_golden_cfg.py) and, at full size, against the guided
oracle's fp32 run on the GPU (tests/cfg_oracle.py); the unguided program left as it was; lanes bit-identical to a single
engine.  Tolerances as in test_engine_gpu.py: eps / stock noise max|d| <= 2e-2 * max|ref|; u8 |d| <= 2 on >= 99.9 % of pixels, max <= 8."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CFG = {"self": 1, "initialize": 2, "full": 3}


def _ref_cfg_step(x, eps, noise, stock, coef, cfg_type, g, delta, do_add_noise):
    """fp32 restatement of StreamDiffusion.predict_x0_batch + unet_step with guidance, rows [T][...]."""
    T = x.shape[0]
    alpha, beta, c_skip, c_out = (coef[k].view(T, 1, 1) for k in range(4))
    step = lambda e, xx: c_out * ((xx - beta * e) / alpha) + c_skip * xx
    s = torch.cat([noise[0:1], stock[:-1]]) if T > 1 else stock.clone()
    u = {"self": 0, "initialize": 1, "full": T}[cfg_type]
    if cfg_type == "initialize":
        s = torch.cat([eps[0:1], s[1:]])
    et = eps[u:]
    eu = eps[:T] if cfg_type == "full" else delta * s
    pred = eu + g * (et - eu)
    x0 = step(pred, x)
    if cfg_type == "full":
        new_stock = s
    else:
        one = torch.ones_like(alpha[0:1])
        an, bn = torch.cat([alpha[1:], one]), torch.cat([beta[1:], one])
        new_stock = torch.cat([noise[1:], noise[0:1]]) + an * step(pred, beta * s) / bn
    new_x = x.clone()
    if T > 1:
        new_x[1:] = alpha[1:] * x0[:-1] + (beta[1:] * noise[1:] if do_add_noise else 0.0)
    return x0[-1], new_x, new_stock


@pytest.mark.parametrize("T", [1, 2, 4])
@pytest.mark.parametrize("cfg_type", ["self", "initialize", "full"])
def test_lcm_cfg_step_op(cuda, cfg_type, T):
    from ai_rtc_agent_b200.host import capi
    lib = capi.lib()
    hw = 24 * 40
    g = torch.Generator().manual_seed(T * 10 + CFG[cfg_type])
    rows = T + {"self": 0, "initialize": 1, "full": T}[cfg_type]
    x = torch.randn(T, hw, 4, generator=g).half()
    eps = torch.randn(rows, hw, 4, generator=g).half()
    noise = torch.randn(T, hw, 4, generator=g).half()
    stock = torch.randn(T, hw, 4, generator=g).half()
    alpha = torch.linspace(0.3, 0.9, T)
    coef = torch.stack([alpha, (1 - alpha ** 2).sqrt(), torch.linspace(0.01, 0.1, T), torch.linspace(0.9, 0.99, T)]).float()
    gs, delta = 1.4, 0.7
    for dan in (1, 0):
        dx, deps, dn, ds, dc = x.cuda(), eps.cuda(), noise.cuda(), stock.cuda(), coef.cuda()
        out = torch.empty(hw, 4, dtype=torch.float16, device="cuda")
        capi.check(lib.b2sd_op_lcm_cfg_step(dx.data_ptr(), deps.data_ptr(), dn.data_ptr(), ds.data_ptr(), dc.data_ptr(),
                                            out.data_ptr(), T, hw, dan, CFG[cfg_type], gs, delta, capi.current_stream_ptr()),
                   "b2sd_op_lcm_cfg_step")
        torch.cuda.synchronize()
        r_out, r_x, r_stock = _ref_cfg_step(x.float(), eps.float(), noise.float(), stock.float(), coef, cfg_type, gs, delta, dan)
        for name, got, ref in (("out", out, r_out), ("x", dx, r_x), ("stock", ds, r_stock)):
            err = (got.float().cpu() - ref).abs().max().item()
            assert err <= 4e-3 * (ref.abs().max().item() + 1.0), f"{cfg_type} T={T} dan={dan}: {name} err {err}"


def _engine(turbo, tl, cfg_type, hw=128, guidance=1.4, delta=0.8, full=False, frames_in_flight=1):
    from ai_rtc_agent_b200.host import arch as A
    from ai_rtc_agent_b200.host.stream import StreamDiffusion
    from oracle import unet as ounet
    from oracle import weights as ow
    if full:
        cfg, arch = (ounet.SD_TURBO, A.SD_TURBO) if turbo else (ounet.SD15, A.SD15)
    else:
        cfg, arch = ounet.tiny_config(turbo), (A.TINY_TURBO if turbo else A.TINY_SD15)
    usd, vsd = ow.make_unet_weights(cfg), ow.make_taesd_weights()
    emb = ow.make_prompt_embeds(cfg.cross_attention_dim)
    neg = ow.make_prompt_embeds(cfg.cross_attention_dim, seed=7)
    sd = StreamDiffusion(arch, usd, vsd, tl, lambda p: neg if p == "negative" else emb, width=hw, height=hw, device="cuda",
                         cfg_type=cfg_type)
    if frames_in_flight > 1:
        sd.set_concurrency(frames_in_flight)
    sd.prepare("p", negative_prompt="negative", guidance_scale=guidance, delta=delta, seed=2)
    return sd, (cfg, usd, vsd, emb, neg)


def _rel(got, ref):
    return (got - ref).abs().max().item() / (ref.abs().max().item() + 1e-12)


@pytest.mark.parametrize("name,turbo,tl,cfg_type", [
    ("cfg_tiny_sd15_T4_self", False, [18, 26, 35, 45], "self"),
    ("cfg_tiny_sd15_T4_initialize", False, [18, 26, 35, 45], "initialize"),
    ("cfg_tiny_sd15_T4_full", False, [18, 26, 35, 45], "full"),
    ("cfg_tiny_turbo_T1_self", True, [32], "self"),
    ("cfg_tiny_turbo_T2_initialize", True, [20, 40], "initialize")])
def test_engine_matches_cfg_golden(cuda, name, turbo, tl, cfg_type):
    from oracle import weights as ow
    gold = np.load(os.path.join(GOLDEN, name + ".npz"))
    sd, _ = _engine(turbo, tl, cfg_type, guidance=float(gold["guidance_scale"]), delta=float(gold["delta"]))
    rows = gold["eps"].shape[1]
    assert sd.trt_unet_batch_size == rows and sd.prompt_embeds.shape[0] == rows
    for i in range(gold["u8"].shape[0]):
        out = sd.step_u8(ow.make_frame(128, 128, seed=i).to(cuda)).cpu().numpy()
        d = np.abs(out.astype(np.int32) - gold["u8"][i:i + 1].astype(np.int32))
        assert (d <= 2).mean() >= 0.999 and d.max() <= 8, f"{name} frame {i}: u8 max {d.max()} frac {(d <= 2).mean():.5f}"
        eps = sd.get_tensor("eps").float().permute(0, 3, 1, 2)
        assert eps.shape[0] == rows
        assert _rel(eps, torch.from_numpy(gold["eps"][i].astype(np.float32))) <= 2e-2, f"{name} frame {i}: eps"
        stock = sd.get_tensor("stock_noise").float().permute(0, 3, 1, 2)
        assert _rel(stock, torch.from_numpy(gold["stock_noise"][i].astype(np.float32))) <= 2e-2, f"{name} frame {i}: stock"


@pytest.mark.parametrize("cfg_type", ["self", "initialize", "full"])
def test_unguided_program_is_unchanged(cuda, cfg_type):
    """guidance <= 1: the same launches and bit-identical frames as cfg_type "none"."""
    from oracle import weights as ow
    base, _ = _engine(False, [18, 26, 35, 45], "none", guidance=1.0)
    for g in (1.0, 0.0):
        sd, _ = _engine(False, [18, 26, 35, 45], cfg_type, guidance=g)
        assert sd.launches_per_step == base.launches_per_step and sd.trt_unet_batch_size == 4
        base.prepare("p", guidance_scale=1.0, seed=2)
        for i in range(3):
            f = ow.make_frame(128, 128, seed=i).cuda()
            assert torch.equal(sd.step_u8(f), base.step_u8(f)), f"{cfg_type} g={g} frame {i}"
    guided, _ = _engine(False, [18, 26, 35, 45], "self", guidance=1.4)
    assert guided.launches_per_step == base.launches_per_step   # residual guidance: the same launch count (fused step)


def _pipeline(model_id, tl, monkeypatch, lanes, **kw):
    from ai_rtc_agent_b200.host import arch as A
    from ai_rtc_agent_b200.host import weights as W
    from lib.pipeline import StreamDiffusionPipeline
    from oracle import unet as ounet
    from oracle import weights as ow
    monkeypatch.setenv("NVENC", "1")
    monkeypatch.setenv("B200SD_POLICY_FRAMES", "2")   # the same launch policy for lanes=1 and lanes=2: outputs comparable bit for bit
    cfg = ounet.tiny_config("turbo" in model_id)
    W.register_preloaded(model_id, A.arch_for(model_id), ow.make_unet_weights(cfg), ow.make_taesd_weights())
    try:
        return StreamDiffusionPipeline(model_id, t_index_list=tl, width=128, height=128, lanes=lanes, **kw)
    finally:
        W._PRELOADED.pop(model_id, None)


@pytest.mark.parametrize("model_id,tl,cfg_type", [("tiny-turbo", [32], "self"), ("tiny-sd15", [18, 26, 35, 45], "initialize")])
def test_guided_lanes_bit_identical_to_one_lane(cuda, monkeypatch, model_id, tl, cfg_type):
    """A guided 1-step "self" stream is stateful (stock noise): it runs on two shared-state stage-pipelined lanes, like T > 1.
    Frames enqueued back to back, with a prompt update while frames are in flight, equal a single engine driven frame by frame."""
    from oracle import weights as ow
    kw = dict(cfg_type=cfg_type, guidance_scale=1.4, delta=0.8, negative_prompt="blurry")
    one = _pipeline(model_id, tl, monkeypatch, 1, **kw)
    two = _pipeline(model_id, tl, monkeypatch, None, **kw)
    assert one.lanes == 1 and two.lanes == 2
    frames = [ow.make_frame(128, 128, seed=140 + i).cuda() for i in range(10)]
    want = []
    for i, f in enumerate(frames):
        if i == 6:
            one.update_prompt("another prompt")
        want.append(one(f).cpu())
    tickets = [two.enqueue(f) for f in frames[:6]]
    two.update_prompt("another prompt")
    tickets += [two.enqueue(f) for f in frames[6:]]
    for i, (t, w) in enumerate(zip(tickets, want)):
        assert torch.equal(t.result().cpu(), w), f"frame {i}"
    s1 = one.model.stream.get_tensor("stock_noise")
    s2 = two.model.stream.get_tensor("stock_noise")
    assert torch.equal(s1, s2) and s1.abs().max().item() > 0


@pytest.mark.parametrize("cfg_type", ["initialize", "self"])
@pytest.mark.parametrize("in_flight", [1, 2])
def test_full_size_sd15_guided_vs_fp32_oracle(cuda, cfg_type, in_flight):
    """SD-1.5 + LCM 4-step at 512x512, guidance 1.4: engine against the oracle's fp32 run on the GPU, latency policy and the
    policy of two stage-pipelined lanes."""
    from oracle import pipeline as opipe
    from oracle import weights as ow
    from tests.cfg_oracle import build_gpu
    tl, hw = [18, 26, 35, 45], 512
    sd, (cfg, usd, vsd, emb, neg) = _engine(False, tl, cfg_type, hw=hw, guidance=1.4, delta=1.0, full=True,
                                            frames_in_flight=in_flight)
    ref = build_gpu(cfg, usd, vsd, tl, hw, emb, sd.init_noise, cfg_type, 1.4, 1.0, uncond_embeds=neg)
    for i in range(4):
        f = ow.make_frame(hw, hw, seed=i).cuda()
        out = sd.step_u8(f).cpu()
        u32 = opipe.frame_to_u8(ref, f).cpu()
        rel = _rel(sd.get_tensor("eps").float().permute(0, 3, 1, 2), ref.last["eps"].float().cpu())
        srel = _rel(sd.get_tensor("stock_noise").float().permute(0, 3, 1, 2), ref.stock_noise.float().cpu())
        d = (out.int() - u32.int()).abs()
        frac = (d <= 2).float().mean().item()
        print(f"{cfg_type} in_flight={in_flight} frame {i}: eps rel {rel:.2e} stock rel {srel:.2e} u8 {frac:.5f}/{d.max().item()}")
        assert rel <= 2e-2 and srel <= 2e-2, f"frame {i}"
        assert frac >= 0.999 and d.max().item() <= 8, f"frame {i}: u8"
