"""Full-size CPU-oracle fixtures for the SD-1.5 + LCM 4-step configurations (BASELINE.json configs[2] at 512x512 and the
768x768 shape of configs[4]): python tests/golden/make_golden_fullsize.py [512|768] [nframes].

The fp32 CPU oracle needs ~10 s (512) / ~60 s (768) per frame on 8 cores and ~25 GB of host memory at 768 (the explicit
softmax(QK^T) over 9216 tokens, 4 images x 8 heads), too much to run inside the GPU tests; the fixtures hold, per frame, eps of
all four stream-batch slots (fp16, on a 1/EPS_STRIDE grid) and the u8 image on a 1/8 grid, plus the SHA-256 of the seed-2 fp16
init_noise the run used.  The 1/3 grid at 768 keeps that file under 1 MB."""
import hashlib
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import pipeline as opipe  # noqa: E402
from oracle import stream as ostream  # noqa: E402
from oracle import unet as ounet  # noqa: E402
from oracle import weights as ow  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
TL = [18, 26, 35, 45]
STRIDE = 8
EPS_STRIDE = {512: 1, 768: 3}


def main(hw: int, nframes: int):
    es = EPS_STRIDE[hw]
    torch.set_num_threads(os.cpu_count() or 8)
    cfg = ounet.SD15
    usd, vsd = ow.to_float(ow.make_unet_weights(cfg)), ow.to_float(ow.make_taesd_weights())
    orc = ostream.StreamOracle(usd, cfg, vsd, TL, hw, hw)
    orc.prepare(ow.make_prompt_embeds(cfg.cross_attention_dim).float(), guidance_scale=0.0, seed=2)
    orc.init_noise = orc.init_noise.half().float()   # the engine receives fp16 noise
    eps, u8 = [], []
    for i in range(nframes):
        t0 = time.time()
        out = opipe.frame_to_u8(orc, ow.make_frame(hw, hw, seed=i))
        eps.append(orc.last["eps"].numpy()[:, :, ::es, ::es].astype(np.float16))
        u8.append(out.numpy()[:, :, ::STRIDE, ::STRIDE])
        print(f"{hw}: frame {i} {time.time() - t0:.1f} s", flush=True)
    noise_sha = hashlib.sha256(orc.init_noise.numpy().astype(np.float16).tobytes()).hexdigest()
    np.savez_compressed(os.path.join(HERE, f"sd15_T4_{hw}.npz"), eps=np.stack(eps), eps_stride=np.array(es), u8=np.stack(u8),
                        u8_stride=np.array(STRIDE), init_noise_sha256=np.array(noise_sha))


if __name__ == "__main__":
    main(int(sys.argv[1]) if len(sys.argv) > 1 else 512, int(sys.argv[2]) if len(sys.argv) > 2 else 2)
