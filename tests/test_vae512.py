"""The native VAE decode of 512 x 512 images (latent side 64: the celeb512 preset, DiT-XL/2 at 512 pixels).

At 512 pixels the decoder's last stage runs on four 128-pixel row segments per image row, the mid-block attention over
4096 tokens, and conv1 of every up_blocks.3 ResBlock takes the GroupNorm statistics of 2^20 elements per (image, group)
in its epilogue - the case the per-slot fixed-point scale of those statistics exists for.

The fp32 oracle (oracle/vae.py) costs ~10 s per 512 x 512 image on the CPU; the GPU tests run it on the device with TF32
off (plain fp32 convolutions and matmuls), which is the same arithmetic up to summation order.
"""
import contextlib
import ctypes
import os

import pytest
import torch
import torch.nn.functional as F

import lfm_b200
from tests._util import rel_l2
from tests.test_gpu_parity import TOL_VAE

SMALL = dict(block_out_channels=(128, 128, 128, 256), layers_per_block=1)   # reduced width, same 512-pixel geometry


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


@contextlib.contextmanager
def _no_tf32():
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        yield
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def oracle_decode(sd, z, cfg, dev, **kw):
    """oracle.vae.vae_decode on the device in fp32 (TF32 off); results on the CPU."""
    from oracle import vae as ovae
    with _no_tf32():
        out = ovae.vae_decode({k: v.to(dev) for k, v in sd.items()}, z.to(dev), cfg, **kw)
    if isinstance(out, tuple):
        return out[0].cpu(), [(p, h) for p, h in out[1]]
    return out.cpu()


def make(cfg_kw, seed, dev, max_batch):
    from oracle import vae as ovae
    cfg = ovae.VAEConfig(**cfg_kw)
    sd = ovae.synthetic_state_dict(cfg, seed)
    vae = lfm_b200.AutoencoderKL(max_batch=max_batch, **cfg_kw)
    vae.load_state_dict(sd, strict=True)
    return vae.to(dev).eval(), sd, cfg


def latents(B, side, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, 4, side, side, generator=g) / 0.18215 * 0.2      # latents / scale_factor, realistic magnitude


def check_vs_oracle(out, z, sd, cfg, dev):
    """-> (fp32 oracle, oracle with bf16-rounded operands)"""
    ref = oracle_decode(sd, z, cfg, dev)
    err = rel_l2(out, ref)
    assert err < TOL_VAE, err
    emul = oracle_decode(sd, z, cfg, dev, emulate_bf16=True)
    noise_floor = rel_l2(emul, ref)                                                  # what bf16 operands cost in exact arithmetic
    assert err < 1.25 * noise_floor + 1e-3, (err, noise_floor)
    return ref, emul


# ------------------------------------------------------------------------------------------------ GPU


@pytest.mark.gpu
def test_vae512_full_width_vs_oracle(dev):
    """sd-vae-ft-mse geometry at latent side 64, two images decoded in chunks of one: parity with the fp32 oracle within
    the bf16-operand noise, determinism, independence of the samples, the fused uint8 post-processing bit for bit."""
    from oracle import vae as ovae
    vae, sd, cfg = make({}, 1, dev, max_batch=1)
    z = latents(2, 64, 164)
    out = vae.decode(z.to(dev)).sample
    assert out.shape == (2, 3, 512, 512) and torch.isfinite(out).all()
    out = out.cpu()
    ref, emul = check_vs_oracle(out, z, sd, cfg, dev)
    assert torch.equal(out, vae.decode(z.to(dev)).sample.cpu())                     # deterministic
    assert rel_l2(vae.decode(z[1:].to(dev)).sample.cpu(), out[1:]) < 1e-5          # samples are independent
    u8 = vae.decode_to_uint8(z.to(dev)).cpu()
    assert u8.dtype == torch.uint8 and u8.shape == (2, 512, 512, 3)
    assert torch.equal(u8, ovae.to_uint8_nhwc(out))
    # grey levels: the shares of pixels off by more than one / two levels are bounded as at 256 pixels.  The largest single
    # deviation is the tail of 4x as many pixels (measured on the B200: 10 levels; 7 for the bf16-operand oracle, which does
    # not round the stored conv1 outputs): bounded at 12 instead of 8.
    d = (u8.int() - ovae.to_uint8_nhwc(ref).int()).abs()
    d_emul = (ovae.to_uint8_nhwc(emul).int() - ovae.to_uint8_nhwc(ref).int()).abs()
    print(f"grey levels vs the fp32 oracle: native max {int(d.max())}, >1 {float((d > 1).float().mean()):.4f}, >2 "
          f"{float((d > 2).float().mean()):.4f}; bf16-operand oracle max {int(d_emul.max())}, >1 {float((d_emul > 1).float().mean()):.4f}")
    assert float((d > 1).float().mean()) < 0.08 and float((d > 2).float().mean()) < 0.01
    assert int(d.max()) <= 12
    # the errors are not concentrated on the seams of the 128-pixel row segments (columns 127 / 128, 255 / 256, 383 / 384)
    seams = [c for c in range(1, 511) if c % 128 in (0, 127)]
    frac_seam, frac_all = float((d[:, :, seams] > 1).float().mean()), float((d > 1).float().mean())
    print(f"share of pixels off by more than one level: seam columns {frac_seam:.4f}, all {frac_all:.4f}")
    assert frac_seam < 1.5 * frac_all + 5e-3


@pytest.mark.gpu
@pytest.mark.parametrize("fuse_out", ["0", "1"])
def test_vae512_reduced_width_odd_batch(dev, monkeypatch, fuse_out):
    """A narrower decoder (128, 128, 128, 256), one ResBlock + 1 per stage, at latent side 64 with an odd batch of three;
    LFM_UNET_FUSE_OUT=1 also takes the statistics of every block output in the epilogue (2^21 elements per group after
    the last upsampler)."""
    monkeypatch.setenv("LFM_UNET_FUSE_OUT", fuse_out)
    vae, sd, cfg = make(SMALL, 4, dev, max_batch=16)
    z = latents(3, 64, 365)
    out = vae.decode(z.to(dev)).sample
    assert out.shape == (3, 3, 512, 512) and torch.isfinite(out).all()
    check_vs_oracle(out.cpu(), z, sd, cfg, dev)


@pytest.mark.gpu
def test_vae512_groupnorm_statistics_headroom(dev):
    """conv1 of the up_blocks.3 ResBlocks scaled by powers of two so that its output rms lands between ~400 and ~1000:
    the sum of squares of one (image, group) of 2^20 elements then exceeds what 2^28 fixed point holds in 63 bits but not
    what the 512-pixel slots' 2^22 holds.  GroupNorm removes the scale (and bf16 keeps a power-of-two multiple exact), so
    the image must stay close to the unscaled decode (a wrapped sum makes it garbage) and match the oracle."""
    from oracle import vae as ovae
    vae, sd, cfg = make(SMALL, 6, dev, max_batch=2)
    z = latents(2, 64, 606)
    base = vae.decode(z.to(dev)).sample.cpu()
    _, feats = oracle_decode(sd, z, cfg, dev, return_features=True)
    prev = dict(zip([p for p, _ in feats[1:]], [h for _, h in feats[:-1]]))     # input of every plan entry but the first
    sdd = {k: v.to(dev) for k, v in sd.items()}
    sd2, overflow_at_2_28 = dict(sd), False
    for j in range(cfg.layers_per_block + 1):
        p = f"decoder.up_blocks.3.resnets.{j}"
        with _no_tf32():
            h = ovae._conv(F.silu(ovae._gn(prev[p].to(dev), sdd, p + ".norm1", cfg)), sdd[p + ".conv1.weight"],
                           sdd[p + ".conv1.bias"], padding=1).double()
        assert h.shape[2] * h.shape[3] * h.shape[1] // 32 == 2 ** 20                  # elements per (image, group)
        k = 2.0 ** round(torch.log2(600.0 / h.pow(2).mean().sqrt()).item())
        assert 400 < k * float(h.pow(2).mean().sqrt()) < 1000
        q = (k * h).pow(2).reshape(h.shape[0], 32, -1).sum(-1)                          # sum of squares per (image, group)
        assert float(q.max()) * 2.0 ** 22 < 2.0 ** 63                                  # the 2^22 slot holds it
        overflow_at_2_28 |= float(q.max()) * 2.0 ** 28 >= 2.0 ** 63                    # 2^28 would have wrapped
        sd2[p + ".conv1.weight"] = sd[p + ".conv1.weight"] * k
        sd2[p + ".conv1.bias"] = sd[p + ".conv1.bias"] * k
    assert overflow_at_2_28
    vae.load_state_dict(sd2, strict=True)
    out = vae.decode(z.to(dev)).sample.cpu()
    assert torch.isfinite(out).all()
    # not bit-identical: eps (1e-6) does not scale with the variance, and the normalised bf16 operand of conv2 rounds
    # differently in places - the decoder amplifies such flips (1.5e-2 for bf16 operand rounding as a whole)
    print(f"scaled vs unscaled decode: rel-L2 {rel_l2(out, base):.2e}")
    assert rel_l2(out, base) < 1e-2
    check_vs_oracle(out, z, sd2, cfg, dev)


@pytest.mark.gpu
def test_vae512_sizes_on_one_module(dev):
    """Latents of side 32, then 64, then 32 again through the same AutoencoderKL (the native context follows the latent
    size): each result equals what a freshly built module gives."""
    vae, sd, _ = make(SMALL, 8, dev, max_batch=2)
    z32, z64 = latents(2, 32, 832), latents(2, 64, 864)
    got = [vae.decode(z.to(dev)).sample.cpu() for z in (z32, z64, z32)]
    for z, g in zip((z32, z64, z32), got):
        fresh, _, _ = make(SMALL, 8, dev, max_batch=2)
        assert torch.equal(g, fresh.decode(z.to(dev)).sample.cpu())
        del fresh


@pytest.mark.gpu
def test_vae512_cli(dev, tmp_path):
    """The CLI at --image_size 512 (DiT-B/2 on 64 x 64 latents, 1024 tokens) with the native decoder and no new flags:
    the image grid, the --compute_fid generation loop with the JPEG sink and the on-device FID, --measure_time."""
    import numpy as np
    from PIL import Image
    from lfm_b200 import cli
    out = str(tmp_path)
    common = ["--model_type", "DiT-B/2", "--image_size", "512", "--num_in_channels", "4", "--num_classes", "1", "--label_dropout", "0.",
              "--method", "euler", "--step_size", "0.5", "--synthetic_init", "3", "--synthetic_vae", "2", "--out_dir", out,
              "--device", "cuda:0", "--dataset", "celeba_512", "--exp", "t"]
    assert cli.main(common + ["--batch_size", "2"]) == 0
    img = Image.open(os.path.join(out, "samples_celeba_512_euler_1e-05_1e-05.jpg"))
    assert img.size == (1024, 512)                                   # 2 images of 512 x 512 in one row
    stat, log = os.path.join(out, "stat.npy"), os.path.join(out, "fid.log")
    feats = np.random.RandomState(0).rand(64, 2048)
    np.save(stat, {"mu": feats.mean(0), "sigma": np.cov(feats, rowvar=False)}, allow_pickle=True)
    assert cli.main(common + ["--batch_size", "2", "--n_sample", "2", "--compute_fid", "--synthetic_inception", "1",
                              "--real_img_dir", stat, "--output_log", log]) == 0
    d = os.path.join(out, "generated_samples", "celeba_512", "expt_ep1000_meuler_s40")
    files = sorted(os.listdir(d), key=lambda f: int(f.split(".")[0]))
    assert files == ["0.jpg", "1.jpg"]
    assert all(Image.open(os.path.join(d, f)).size == (512, 512) for f in files)
    fid = float(open(log).read().strip().split("FID = ")[1])
    assert np.isfinite(fid) and fid > 0
    assert cli.main(common + ["--measure_time", "--measure_reps", "2"]) == 0


# ------------------------------------------------------------------------------------------------ CPU


def _vae_desc(latent_size, boc=(128, 256, 512, 512)):
    from lfm_b200 import _lib
    return _lib.VaeDesc(latent_size, 4, 3, len(boc), (ctypes.c_int32 * 8)(*boc), 2, 32)


def test_vae512_create_validation_without_gpu():
    """lfm_create_vae accepts latent side 64 (its only failure here is the missing device) and still refuses 128, whose
    mid-block attention would run over 16384 tokens."""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from lfm_b200 import _lib, build
    build.build()
    lib = _lib.load()
    ctx = ctypes.c_void_p()
    assert lib.lfm_create_vae(ctypes.byref(_vae_desc(64)), 0, ctypes.byref(ctx)) != 0
    assert "no CUDA device" in _lib.last_error()
    assert lib.lfm_create_vae(ctypes.byref(_vae_desc(128)), 0, ctypes.byref(ctx)) != 0
    assert "16384 tokens" in _lib.last_error()
    assert lib.lfm_create_vae(ctypes.byref(_vae_desc(64, (128, 256, 512, 512, 512))), 0, ctypes.byref(ctx)) != 0
    assert "exceeds 512" in _lib.last_error()
