"""Small end-to-end run for compute-sanitizer (memcheck / racecheck / synccheck): every native family once, at sizes the
instrumented run finishes in minutes - mini DiT (forward with labels, CFG Heun from the step graph, dopri5 from the step
graph, LayerNorm finisher path), mini ADM UNetModel, mini EDM DhariwalUNet (resampling blocks, both attention kernels),
the VAE decoder at 128 x 128 (batched attention GEMMs, 128-pixel conv tiles) with the fused uint8 post-processing, and
at 512 x 512 (vae512: two images; 4096-token attention, four row segments per image row, 2^22 fixed-point statistics).
  compute-sanitizer --tool memcheck  python scripts/sanitizer_run.py [dit unet edm vae vae512]
  compute-sanitizer --tool racecheck python scripts/sanitizer_run.py"""
import os
import sys
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import lfm_b200  # noqa: E402
from lfm_b200.synthetic import synthetic_edm_state_dict, synthetic_state_dict, synthetic_unet_state_dict  # noqa: E402

dev = torch.device("cuda:0")
which = sys.argv[1:] or ["dit", "unet", "edm", "vae", "vae512"]
x = torch.randn(3, 4, 32, 32, device=dev)
res = {}
if "dit" in which:
    net = lfm_b200.DiT(img_resolution=32, patch_size=2, in_channels=4, hidden_size=256, depth=2, num_heads=4, label_dropout=0.1, num_classes=10)
    net.load_state_dict(synthetic_state_dict(net, 3), strict=True)
    net = net.to(dev)
    y = torch.tensor([1, 2, 3], device=dev)
    v = net(torch.tensor([0.3, 0.5, 0.7], device=dev), x, y)
    ynull = torch.full((3,), 10, device=dev)
    out = lfm_b200.karras_sample(net, torch.cat([x, x]), 3, clip_denoised=False, model_kwargs=dict(y=torch.cat([y, ynull]), cfg_scale=1.5),
                                 sigma_min=1e-5, sigma_max=1.0, sampler="heun")
    args = types.SimpleNamespace(method="dopri5", atol=1e-2, rtol=1e-2, cfg_scale=1.0, compute_nfe=False)
    traj = lfm_b200.sample_from_model(net, x, dict(y=y), args)
    res["dit"] = (float(v.abs().mean()), float(out.abs().mean()), float(traj[-1].abs().mean()), net.last_stats)
if "unet" in which:
    un = lfm_b200.UNetModel(image_size=32, in_channels=4, model_channels=128, out_channels=4, num_res_blocks=1, attention_resolutions=(2, 4),
                            channel_mult=(1, 2, 2), num_heads=2, use_scale_shift_norm=True)
    un.load_state_dict(synthetic_unet_state_dict(un, 5), strict=True)
    un = un.to(dev)
    res["unet"] = float(un(torch.tensor(0.4, device=dev), x).abs().mean())
if "edm" in which:
    ed = lfm_b200.DhariwalUNet(img_resolution=32, in_channels=4, out_channels=4, label_dim=5, model_channels=128, channel_mult=(1, 2, 2),
                               num_blocks=1, attn_resolutions=(16, 8))
    ed.load_state_dict(synthetic_edm_state_dict(ed, 7), strict=True)
    ed = ed.to(dev)
    ve = ed.forward_with_cfg(torch.tensor(0.6, device=dev), torch.cat([x[:2], x[:2]]), torch.tensor([0, 4, 0, 0], device=dev), cfg_scale=1.3)
    res["edm"] = float(ve.abs().mean())
if "vae" in which:
    vae = lfm_b200.AutoencoderKL(max_batch=2)
    vae.load_state_dict(lfm_b200.synthetic_vae_state_dict(vae, 2), strict=True)
    vae = vae.to(dev)
    u8 = vae.decode_to_uint8(torch.randn(2, 4, 16, 16, device=dev))
    res["vae"] = float(u8.float().mean())
if "vae512" in which:
    vae = lfm_b200.AutoencoderKL(max_batch=2)
    vae.load_state_dict(lfm_b200.synthetic_vae_state_dict(vae, 2), strict=True)
    vae = vae.to(dev)
    u8 = vae.decode_to_uint8(torch.randn(2, 4, 64, 64, device=dev))
    res["vae512"] = float(u8.float().mean())
torch.cuda.synchronize()
print("ok", res)
