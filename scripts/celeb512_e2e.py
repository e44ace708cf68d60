"""The celeb512 preset end to end on cuda:0 (test_args/celeb512_adm.txt: ADM UNetModel on 64x64x4 latents, dopri5
atol = rtol = 1e-5, batch 16), synthetic weights: sampling alone, and sampling + the native 512 x 512 VAE decode with the
fused uint8 post-processing, as the --compute_fid loop runs it.  One JSON line; the card and its power limit beside it.
python scripts/celeb512_e2e.py [batch] [reps]"""
import json
import os
import subprocess
import sys
import time
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import lfm_b200  # noqa: E402
from lfm_b200.synthetic import synthetic_unet_state_dict  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return {"gpu": torch.cuda.get_device_name(0), "power_limit": q.stdout.strip() or "unavailable"}


B = int(sys.argv[1]) if len(sys.argv) > 1 else 16
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
dev = torch.device("cuda:0")
with torch.device("meta"):
    net = lfm_b200.UNetModel(image_size=64, in_channels=4, model_channels=256, out_channels=4, num_res_blocks=2,
                             attention_resolutions=(16, 8), channel_mult=(1, 2, 2, 2, 4), num_heads=4,
                             use_scale_shift_norm=True, max_batch=B)
sd = synthetic_unet_state_dict(net, 1)
net = net.to_empty(device="cpu")
net.load_state_dict(sd, strict=True)
net = net.to(dev)
vae = lfm_b200.AutoencoderKL(max_batch=B)
vae.load_state_dict(lfm_b200.synthetic_vae_state_dict(vae, 1), strict=True)
vae = vae.to(dev).eval()
x = torch.randn(B, 4, 64, 64, generator=torch.Generator().manual_seed(0)).to(dev)
args = types.SimpleNamespace(method="dopri5", atol=1e-5, rtol=1e-5, cfg_scale=1.0, compute_nfe=False)


def sample():
    return lfm_b200.sample_from_model(net, x, {}, args)[-1]


def sample_decode():
    return vae.decode_to_uint8(sample() / 0.18215)


def timed(fn):
    fn()                                   # builds the native contexts, warms every shape
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps * 1e3, out


ms_s, _ = timed(sample)
nfe = net.last_stats["nfe"]
ms_sd, u8 = timed(sample_decode)
print(json.dumps({**gpu_info(), "config": f"celeb512 preset: ADM UNetModel dopri5 1e-5, batch {B}, synthetic weights, + VAE decode 512x512",
                  "nfe": nfe, "ms_sampling": round(ms_s, 1), "images_per_s_sampling": round(B / ms_s * 1e3, 2),
                  "ms_sampling_decode": round(ms_sd, 1), "images_per_s_with_decode": round(B / ms_sd * 1e3, 2),
                  "ms_decode_share": round(ms_sd - ms_s, 1), "u8_shape": list(u8.shape), "reps": reps}), flush=True)
