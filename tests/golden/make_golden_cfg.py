"""Regenerates tests/golden/cfg_*.npz (python tests/golden/make_golden_cfg.py) from the guided CPU oracle of
tests/cfg_oracle.py: classifier-free guidance (cfg_type self / initialize / full, guidance_scale GUIDANCE, delta DELTA,
negative prompt = a second seeded embedding) on the seeded tiny models of make_golden.py, 128x128 frames.  Each fixture holds per frame the u8 output, eps of every UNet row
(uncond rows first) and the stock noise after the frame."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import pipeline as opipe  # noqa: E402
from oracle import unet as ounet  # noqa: E402
from oracle import weights as ow  # noqa: E402
from tests.cfg_oracle import CfgStreamOracle  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
# name -> (turbo, t_index_list, cfg_type)
CASES = {
    "cfg_tiny_sd15_T4_self": (False, [18, 26, 35, 45], "self"),
    "cfg_tiny_sd15_T4_initialize": (False, [18, 26, 35, 45], "initialize"),
    "cfg_tiny_sd15_T4_full": (False, [18, 26, 35, 45], "full"),
    "cfg_tiny_turbo_T1_self": (True, [32], "self"),
    "cfg_tiny_turbo_T2_initialize": (True, [20, 40], "initialize"),
}
HW, NFRAMES = 128, 5
GUIDANCE, DELTA = 1.4, 0.8
NEGATIVE_SEED = 7   # ow.make_prompt_embeds(dim, seed=NEGATIVE_SEED) stands for the encoded negative prompt


def run_case(turbo, t_index_list, cfg_type):
    torch.manual_seed(0)
    torch.set_num_threads(4)
    cfg = ounet.tiny_config(turbo)
    usd, vsd = ow.to_float(ow.make_unet_weights(cfg)), ow.to_float(ow.make_taesd_weights())
    orc = CfgStreamOracle(usd, cfg, vsd, t_index_list, HW, HW, cfg_type=cfg_type)
    emb = ow.make_prompt_embeds(cfg.cross_attention_dim)
    neg = ow.make_prompt_embeds(cfg.cross_attention_dim, seed=NEGATIVE_SEED)
    orc.prepare(emb.float(), guidance_scale=GUIDANCE, delta=DELTA, seed=2, uncond_embeds=neg.float())
    orc.init_noise = orc.init_noise.half().float()   # the engine receives fp16 noise
    outs, eps, stock = [], [], []
    for i in range(NFRAMES):
        outs.append(opipe.frame_to_u8(orc, ow.make_frame(HW, HW, seed=i)).numpy())
        eps.append(orc.last["eps"].numpy().astype(np.float16))
        stock.append(orc.stock_noise.numpy().astype(np.float16))
    return {"u8": np.concatenate(outs, 0), "eps": np.stack(eps, 0), "stock_noise": np.stack(stock, 0),
            "sub_timesteps": np.array(orc.sub_timesteps), "guidance_scale": np.float32(GUIDANCE), "delta": np.float32(DELTA)}


if __name__ == "__main__":
    for name, (turbo, tl, cfg_type) in CASES.items():
        d = run_case(turbo, tl, cfg_type)
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **d)
        print(name, {k: v.shape for k, v in d.items()}, os.path.getsize(path), "bytes")
