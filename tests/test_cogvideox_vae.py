"""CogVideoX 3-D causal VAE decoder (SURVEY 8 row f4) against outputs of the reference's UNMODIFIED cp_enc_dec.py
(oracle/cogvideox_vae.py: context-parallel size 1, SafeConv3d = Conv3d), stored by oracle/make_golden_reference.py."""
import pytest
import torch

from star_b200.utils.synth import synth_state_dict
from tests.util import assert_close, load_golden, rel_l2, sample_flat

SMALL = dict(ch=32, ch_mult=(1, 2, 2, 4), num_res_blocks=1)          # 32..128 channels, same topology as the shipped decoder


def decoder_weights(manifest, seed=3):
    sd = synth_state_dict(manifest, seed=seed)
    for k in sd:                                    # conv_y multiplies the normalised features: keep it O(1), not O(1/sqrt(16))
        if ".conv_y.conv.bias" in k:
            sd[k] = sd[k] + 1.0
    return sd


def _decoder(kw, device="cpu", dtype=torch.float16):
    from star_b200.cogvideox.vae3d import ContextParallelDecoder3D
    mine = ContextParallelDecoder3D(**kw)
    mine.load_state_dict(decoder_weights({k: tuple(v.shape) for k, v in mine.state_dict().items()}))
    return mine.to(device=device, dtype=dtype).eval()


def _encoder(kw, seed=6, device="cpu", dtype=torch.float16):
    from star_b200.cogvideox.vae3d import ContextParallelEncoder3D
    mine = ContextParallelEncoder3D(**kw)
    mine.load_state_dict(synth_state_dict({k: tuple(v.shape) for k, v in mine.state_dict().items()}, seed=seed))
    return mine.to(device=device, dtype=dtype).eval()


def decoder_host_input():
    return torch.randn(1, 16, 7, 4, 6, generator=torch.Generator().manual_seed(0))


def encoder_host_inputs():
    x = torch.rand(1, 3, 9, 32, 48, generator=torch.Generator().manual_seed(3)) * 2 - 1
    even = torch.rand(1, 3, 8, 16, 16, generator=torch.Generator().manual_seed(4)) * 2 - 1      # even T: plain pair pooling
    return x, even


def _patch(monkeypatch):
    from oracle import kernel_ref as KR
    from star_b200 import ops
    for name in dir(KR):
        if not name.startswith("_") and callable(getattr(KR, name)) and hasattr(ops, name):
            monkeypatch.setattr(ops, name, getattr(KR, name))


def test_state_dict_layout_matches_reference():
    from star_b200.cogvideox.vae3d import ContextParallelDecoder3D
    gold = load_golden("reference_cpu.pt")
    with torch.device("meta"):
        mine = ContextParallelDecoder3D()
    got = {k: tuple(v.shape) for k, v in mine.state_dict().items()}
    assert got == gold["vae_dec_manifest"]
    assert sum(torch.Size(s).numel() for s in got.values()) == gold["vae_dec_params"]


def test_decoder_host_graph_on_emulated_kernels(monkeypatch):
    """3 + 2 + 2 latent frames through the reference's chunk protocol (sample_sr.py:212-227): odd / even clip lengths, the
    first-frame split of SpatialNorm3D and Upsample3D, and the causal-conv context carried between chunks."""
    gold = load_golden("reference_cpu.pt")
    _patch(monkeypatch)
    mine = _decoder(SMALL)
    z = decoder_host_input()
    got = mine.decode_latent(z)
    assert got.shape == (1, 3, 25, 32, 48) and got.dtype == torch.float16
    assert rel_l2(sample_flat(got), gold["vae_dec_out"]) < 3e-3
    assert not mine._cache                                                    # the last chunk clears the context
    # a chunk decoded alone (clear cache) replicates its first frame instead of using context
    assert rel_l2(sample_flat(mine(z[:, :, 3:5].contiguous())), gold["vae_dec_alone"]) < 3e-3
    assert rel_l2(sample_flat(got[:, :, 9:17]), gold["vae_dec_alone"]) > 1e-2  # ... and that differs from the chunked result


def test_encoder_host_graph_on_emulated_kernels(monkeypatch):
    """9 frames of 32x48 -> moments (1, 32, 3, 4, 6): odd clip lengths through both time-compressing DownSample3D levels
    (9 -> 5 -> 3), the (0,1,0,1)-padded stride-2 convs, clip-wide GroupNorm, first-frame replication of the causal convs"""
    from star_b200.cogvideox.vae3d import ContextParallelEncoder3D
    gold = load_golden("reference_cpu.pt")
    _patch(monkeypatch)
    with torch.device("meta"):
        assert {k: tuple(v.shape) for k, v in ContextParallelEncoder3D().state_dict().items()} == gold["vae_enc_manifest"]
    mine = _encoder(SMALL)
    x, even = encoder_host_inputs()
    got = mine(x)
    assert got.shape == gold["vae_enc_out"].shape == (1, 32, 3, 4, 6)
    assert rel_l2(got, gold["vae_enc_out"]) < 3e-3
    assert rel_l2(mine(even), gold["vae_enc_even_out"]) < 3e-3
    torch.manual_seed(0)
    z = mine.encode(x)
    torch.manual_seed(0)
    mean, logvar = got.float().chunk(2, dim=1)
    assert torch.allclose(z.float(), mean + torch.exp(0.5 * logvar.clamp(-30, 20)) * torch.randn_like(got[:, :16], dtype=torch.float32), atol=1e-2)


def test_spatial_norm_index_rule():
    """row -> latent-row map of star_groupnorm_mod == F.interpolate(nearest) with the reference's first-frame split"""
    import torch.nn.functional as F
    from oracle.kernel_ref import spatial_norm_src_index
    for (T, Tl) in ((9, 3), (5, 3), (3, 3), (8, 2), (4, 2), (2, 2), (1, 1)):
        H, W, Hl, Wl = 8, 12, 4, 6
        zq = torch.arange(Tl * Hl * Wl, dtype=torch.float32).reshape(1, 1, Tl, Hl, Wl)
        if T > 1 and T % 2 == 1:
            a = F.interpolate(zq[:, :, :1], size=(1, H, W), mode="nearest")
            b = F.interpolate(zq[:, :, 1:], size=(T - 1, H, W), mode="nearest")
            want = torch.cat([a, b], dim=2)
        else:
            want = F.interpolate(zq, size=(T, H, W), mode="nearest")
        got = spatial_norm_src_index(T, H, W, Tl, Hl, Wl, "cpu")
        assert torch.equal(got, want.reshape(-1).long())


# ---------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def env():
    from star_b200 import ops
    from oracle import kernel_ref as KR
    return ops, KR


@pytest.mark.gpu
@pytest.mark.parametrize("T,H,W,Cin,Cout,res", [(3, 12, 20, 64, 128, False), (9, 30, 44, 128, 128, True), (2, 60, 90, 256, 128, True),
                                                 (8, 17, 23, 64, 3, False), (3, 60, 90, 512, 512, True)])
def test_conv3d_causal(env, T, H, W, Cin, Cout, res):
    ops, KR = env
    g = torch.Generator(device="cuda").manual_seed(T * 100 + Cin)
    xp = torch.randn((T + 2) * H * W, Cin, device="cuda", generator=g).half()
    w = (torch.randn(Cout, 3, 3, 3, Cin, device="cuda", generator=g) * (27 * Cin) ** -0.5).half()
    b = (torch.randn(Cout, device="cuda", generator=g) * 0.1).half()
    r = torch.randn(T * H * W, Cout, device="cuda", generator=g).half() if res else None
    if Cout == 3:
        out = torch.zeros(T * H * W, 8, device="cuda", dtype=torch.float16)
        ops.conv3d_causal(xp, w, T, H, W, b, out=out[:, :3])
        got = out[:, :3]
        assert (out[:, 3:] == 0).all()
    else:
        got = ops.conv3d_causal(xp, w, T, H, W, b, residual=r)
    assert_close(got, KR.conv3d_causal(xp, w, T, H, W, b, residual=r), what="conv3d_causal")


@pytest.mark.gpu
@pytest.mark.parametrize("T,Tl,H,W,Hl,Wl,C", [(9, 3, 32, 48, 4, 6, 128), (8, 2, 32, 48, 4, 6, 256), (3, 3, 60, 90, 60, 90, 512),
                                               (5, 3, 24, 36, 12, 18, 512), (4, 2, 16, 16, 8, 8, 32), (2, 2, 12, 18, 4, 6, 64), (9, 3, 480, 720, 60, 90, 128)])
def test_groupnorm_mod(env, T, Tl, H, W, Hl, Wl, C):
    ops, KR = env
    g = torch.Generator(device="cuda").manual_seed(T + C)
    x = (torch.randn(T * H * W, C, device="cuda", generator=g) * 2 + 0.5).half()
    gam, bet = (1 + 0.1 * torch.randn(C, device="cuda", generator=g)).half(), (0.1 * torch.randn(C, device="cuda", generator=g)).half()
    mod = torch.randn(Tl * Hl * Wl, 2 * C, device="cuda", generator=g).half()
    got = ops.groupnorm_mod(x, gam, bet, mod[:, :C], mod[:, C:], T, H, W, Tl, Hl, Wl, 1e-6, True)
    assert_close(got, KR.groupnorm_mod(x, gam, bet, mod[:, :C], mod[:, C:], T, H, W, Tl, Hl, Wl, 1e-6, True), what="groupnorm_mod")


def decoder_gpu_input():
    return torch.randn(1, 16, 5, 16, 24, generator=torch.Generator().manual_seed(1))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,tol", [(torch.float16, 3e-3), (torch.bfloat16, 1.6e-2)])
def test_decoder_vs_reference_gpu(dtype, tol):
    """full-width decoder (ch 128, 3 res blocks per level), 3 + 2 latent frames at 16x24 -> 17 frames of 128x192, against the
    reference's own file in fp32 (TF32 off) and beside the reference run in the same 16-bit dtype, both on the B200"""
    gold = load_golden("reference_gpu.pt")["vae_dec"]
    mine = _decoder({}, device="cuda", dtype=dtype)
    got = mine.decode_latent(decoder_gpu_input().cuda().to(dtype))
    assert got.shape == (1, 3, 17, 128, 192)
    err, err_ref = rel_l2(sample_flat(got), gold["out"]), gold["err_ref"][str(dtype)]
    print(f"[cogvideox vae {dtype}] star {err:.2e}  reference-in-{dtype} {err_ref:.2e}")
    assert torch.isfinite(got.float()).all()
    assert err < tol and err < 1.5 * err_ref + 1e-3


@pytest.mark.gpu
@pytest.mark.parametrize("T,HW,C", [(9, 640, 128), (8, 1000, 256), (2, 77, 64), (49, 120, 128)])
def test_time_avgpool2(env, T, HW, C):
    ops, KR = env
    x = torch.randn(T * HW, C, device="cuda", generator=torch.Generator(device="cuda").manual_seed(T)).half()
    got, want = ops.time_avgpool2(x, T, HW), KR.time_avgpool2(x, T, HW)
    assert got.shape == want.shape and torch.equal(got, want)                  # one rounding of an exact fp32 sum


def encoder_gpu_input():
    return torch.rand(1, 3, 17, 96, 128, generator=torch.Generator().manual_seed(2)) * 2 - 1


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,tol", [(torch.float16, 3e-3), (torch.bfloat16, 1.6e-2)])
def test_encoder_vs_reference_gpu(dtype, tol):
    """full-width encoder (ch 128, 3 res blocks per level), 17 frames of 96x128 -> moments (1, 32, 5, 12, 16)"""
    gold = load_golden("reference_gpu.pt")["vae_enc"]
    mine = _encoder({}, device="cuda", dtype=dtype)
    got = mine(encoder_gpu_input().cuda().to(dtype))
    err, err_ref = rel_l2(sample_flat(got), gold["out"]), gold["err_ref"][str(dtype)]
    print(f"[cogvideox vae encoder {dtype}] star {err:.2e}  reference-in-{dtype} {err_ref:.2e}")
    assert got.shape == (1, 32, 5, 12, 16) and torch.isfinite(got.float()).all()
    assert err < tol and err < 1.5 * err_ref + 1e-3
