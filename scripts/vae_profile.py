"""Timing of the native VAE decode (lfm_b200.AutoencoderKL, synthetic weights) on cuda:0: ms per batch, images/s, TFLOP/s.
python scripts/vae_profile.py [--side S ...] [batch ...]
  --side: latent side (32 = 256 x 256 images, 64 = 512 x 512); repeat it to time several sizes in one run, on the same card.
  The first line names the card and its power limit.  (Wrap in ncu for a launch list: a decode is ~200 launches.)"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import lfm_b200  # noqa: E402


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["sm_max_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:  # the number is still valid; say why the limit is missing
        info["power_limit"] = f"unavailable ({type(e).__name__})"
    return info


ap = argparse.ArgumentParser()
ap.add_argument("--side", type=int, action="append", help="latent side (default 32)")
ap.add_argument("batches", type=int, nargs="*")
a = ap.parse_args()
dev = torch.device("cuda:0")
print(json.dumps(gpu_info()), flush=True)
vae = lfm_b200.AutoencoderKL(max_batch=16)
vae.load_state_dict(lfm_b200.synthetic_vae_state_dict(vae, 1), strict=True)
vae = vae.to(dev).eval()
for side in a.side or [32]:
    fl = vae.decode_flops_per_image(side)
    # device memory of the native context (weights + the workspace of lfm_finalize(16)): cudaMalloc'd outside torch's allocator
    vae._release()                          # the context of the previous size
    torch.cuda.synchronize()
    free0, reserved0 = torch.cuda.mem_get_info()[0], torch.cuda.memory_reserved()
    vae.decode_to_uint8(torch.zeros(1, 4, side, side, device=dev))
    torch.cuda.synchronize()
    ctx_bytes = free0 - torch.cuda.mem_get_info()[0] - (torch.cuda.memory_reserved() - reserved0)
    print(json.dumps({"latent_side": side, "image_side": 8 * side, "native_context_gb": round(ctx_bytes / 1e9, 2), "max_batch": 16,
                      "gb_per_image": round(ctx_bytes / 16 / 1e9, 3)}), flush=True)
    for B in a.batches or [1, 16, 64]:
        z = torch.randn(B, 4, side, side, device=dev) * 1.1
        for _ in range(2):
            u8 = vae.decode_to_uint8(z)
        torch.cuda.synchronize()
        reps = 5
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = vae.launch_count()
        e0.record()
        for _ in range(reps):
            u8 = vae.decode_to_uint8(z)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        print(json.dumps({"latent_side": side, "image_side": 8 * side, "vae_decode_batch": B, "ms": round(ms, 3),
                          "ms_per_image": round(ms / B, 3), "images_per_s": round(B / ms * 1e3, 1),
                          "tflops": round(B * fl / ms / 1e9, 1), "launches_per_decode": (vae.launch_count() - l0) // reps,
                          "finite": bool(torch.isfinite(vae.decode(z[:1]).sample).all())}), flush=True)
