"""CPU suite (no GPU): the oracle against the golden vectors produced by the real reference
(oracle/make_golden.py, oracle/make_golden_reference.py)."""
import json
import os

import pytest
import torch

from tests.util import SMALL_KW, make_inputs, rel_l2

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def small_sd():
    from star_b200.utils.synth import synth_state_dict
    from star_b200.video_to_video.modules.unet_v2v import ControlledV2VUNet
    with torch.device("meta"):
        net = ControlledV2VUNet(**SMALL_KW)
    return synth_state_dict({k: tuple(v.shape) for k, v in net.state_dict().items()}, seed=1)


def test_unet_restatement_matches_golden(small_sd):
    """oracle/unet_ref.py (fp32) == real reference output, all three recorded shapes."""
    from oracle.unet_ref import UNetCfg, controlled_unet_forward
    gold = torch.load(os.path.join(GOLD, "unet_small.pt"))
    assert gold["kw"] == SMALL_KW and gold["weight_seed"] == 1
    for c in gold["cases"]:
        x, hint, y = make_inputs(c["seed"], c["B"], c["F"], c["H"], c["W"])
        out = controlled_unet_forward(small_sd, x, torch.tensor(c["t"]), y, hint, UNetCfg(**SMALL_KW))
        assert rel_l2(out, c["out_fp32"]) < 2e-5, c


def live_reference_inputs():
    x, hint, y = make_inputs(42, 1, 3, 10, 16)
    return x, torch.tensor([123]), y, hint


def test_unet_restatement_matches_live_reference(small_sd):
    """oracle/unet_ref.py (fp32) == the reference's own ControlledV2VUNet at a fourth input shape"""
    from oracle.unet_ref import UNetCfg, controlled_unet_forward
    x, t, y, hint = live_reference_inputs()
    out = controlled_unet_forward(small_sd, x, t, y, hint, UNetCfg(**SMALL_KW))
    assert rel_l2(out, torch.load(os.path.join(GOLD, "reference_cpu.pt"))["unet_out"]) < 2e-5


def test_state_dict_layout_matches_live_reference():
    """2 247 tensors, same names and shapes as the reference's ControlledV2VUNet() (manifest written from it)."""
    from star_b200.video_to_video.modules.unet_v2v import ControlledV2VUNet
    man = json.load(open(os.path.join(GOLD, "state_dict_manifest.json")))
    with torch.device("meta"):
        mine = ControlledV2VUNet()
    a = {k: list(v.shape) for k, v in mine.state_dict().items()}
    assert a == man and len(a) == 2247


def test_state_dict_layout_matches_manifest():
    from star_b200.video_to_video.modules.unet_v2v import ControlledV2VUNet
    man = json.load(open(os.path.join(GOLD, "state_dict_manifest.json")))
    with torch.device("meta"):
        mine = ControlledV2VUNet()
    a = {k: list(v.shape) for k, v in mine.state_dict().items()}
    assert a == man and len(a) == 2247
    assert sum(torch.Size(s).numel() for s in man.values()) == 2041121910      # SURVEY 8c [probe]


def test_unet_host_graph_on_emulated_kernels(small_sd, monkeypatch):
    """Host logic of the product (weight repacking, op order, layouts) with every C-ABI op replaced
    by its torch reference (oracle/kernel_ref.py): must reproduce the golden output to fp16
    accuracy.  The CUDA kernels themselves are checked op by op in test_kernels_gpu.py."""
    from oracle import kernel_ref as KR
    from star_b200 import ops
    from star_b200.video_to_video.modules.unet_v2v import ControlledV2VUNet
    for name in dir(KR):
        if not name.startswith("_") and callable(getattr(KR, name)) and hasattr(ops, name):
            monkeypatch.setattr(ops, name, getattr(KR, name))
    with torch.device("meta"):
        net = ControlledV2VUNet(**SMALL_KW)
    net.load_state_dict(small_sd, assign=True)
    net = net.half().eval()
    gold = torch.load(os.path.join(GOLD, "unet_small.pt"))
    for c in gold["cases"][:2]:
        x, hint, y = make_inputs(c["seed"], c["B"], c["F"], c["H"], c["W"])
        out = net(x, torch.tensor(c["t"]), y, hint=hint)
        assert out.dtype == torch.float16
        err = rel_l2(out, c["out_fp32"])
        # fp16 storage between ops: same error class as the reference's own fp16-autocast path
        assert err < 1.5 * c["ref_fp16_rel_err"] and err < 4e-3, (err, c["ref_fp16_rel_err"])


def test_cfg_pair_forward_equals_two_forwards_on_emulated_kernels(small_sd, monkeypatch):
    """forward_cfg_pair (shared text-independent prefix) == two forward() calls, bit for bit (host graph on the emulated kernels);
    the sampler's denoise() takes the pair path and reproduces the two-call result exactly."""
    from oracle import kernel_ref as KR
    from star_b200 import ops
    from star_b200.video_to_video.diffusion.diffusion_sdedit import GaussianDiffusion
    from star_b200.video_to_video.diffusion.schedules_sdedit import noise_schedule
    from star_b200.video_to_video.modules.unet_v2v import ControlledV2VUNet
    for name in dir(KR):
        if not name.startswith("_") and callable(getattr(KR, name)) and hasattr(ops, name):
            monkeypatch.setattr(ops, name, getattr(KR, name))
    with torch.device("meta"):
        net = ControlledV2VUNet(**SMALL_KW)
    net.load_state_dict(small_sd, assign=True)
    net = net.half().eval()
    x, hint, y = make_inputs(0, 1, 3, 10, 8)
    _, _, ny = make_inputs(1, 1, 3, 10, 8)
    t = torch.tensor([500])
    a, b = net(x, t, y, hint=hint), net(x, t, ny, hint=hint)
    pa, pb = net.forward_cfg_pair(x, t, (y, ny), hint=hint)
    assert torch.equal(a, pa) and torch.equal(b, pb) and not torch.equal(a, b)
    d = GaussianDiffusion(noise_schedule(schedule="logsnr_cosine_interp", n=1000, zero_terminal_snr=True, scale_min=2.0, scale_max=4.0))
    kw = [{"y": y}, {"y": ny}, {"hint": hint}]
    x0_pair = d.denoise(x, t, None, net, kw, guide_scale=7.5, guide_rescale=0.2)[-2]

    class TwoCalls(torch.nn.Module):                    # hides forward_cfg_pair: the reference's two-call structure
        def forward(self, *a, **k):
            return net(*a, **k)
    x0_two = d.denoise(x, t, None, TwoCalls(), kw, guide_scale=7.5, guide_rescale=0.2)[-2]
    assert torch.equal(x0_pair, x0_two)


def test_product_has_no_cpu_fallback():
    from star_b200 import lib, ops
    x = torch.zeros(8, 64, dtype=torch.float16)
    with pytest.raises(lib.StarError):
        ops.linear(x, x)


def test_uneven_chunks_host_graph_vs_oracle(small_sd, monkeypatch):
    """A 36-frame clip with max_chunk_len 16 -> chunks (0,16), (8,24), (16,36): the last one is 1.25x long (as the
    (32,72) chunk of BASELINE config 3).  Product (host graph on emulated kernels, fp16 storage) against the fp32 oracle
    UNet through the same sampler, CFG 7.5, identical noise."""
    from oracle import kernel_ref as KR
    from oracle.unet_ref import UNetCfg, controlled_unet_forward
    from star_b200 import ops
    from star_b200.video_to_video.diffusion.diffusion_sdedit import GaussianDiffusion
    from star_b200.video_to_video.diffusion.schedules_sdedit import noise_schedule
    from star_b200.video_to_video.modules.unet_v2v import ControlledV2VUNet
    from star_b200.video_to_video.video_to_video_model import make_chunks
    for name in dir(KR):
        if not name.startswith("_") and callable(getattr(KR, name)) and hasattr(ops, name):
            monkeypatch.setattr(ops, name, getattr(KR, name))
    chunks = make_chunks(36, 0, 16)
    assert chunks == [(0, 16), (8, 24), (16, 36)]
    with torch.device("meta"):
        net = ControlledV2VUNet(**SMALL_KW)
    net.load_state_dict(small_sd, assign=True)
    net = net.half().eval()
    cfg = UNetCfg(**SMALL_KW)

    def oracle_model(xt, t, y=None, hint=None, hint_chunk=None, variant_info=None):
        return controlled_unet_forward(small_sd, xt, t, y, hint_chunk if hint_chunk is not None else hint, cfg)

    x, hint, y = make_inputs(5, 1, 36, 10, 8)
    _, _, ny = make_inputs(6, 1, 36, 10, 8)
    diff = GaussianDiffusion(noise_schedule(schedule="logsnr_cosine_interp", n=1000, zero_terminal_snr=True, scale_min=2.0,
                                            scale_max=4.0))
    outs = []
    for model in (oracle_model, net):
        g = torch.Generator().manual_seed(3)
        outs.append(diff.sample_sr(noise=x.clone(), model=model, model_kwargs=[{"y": y}, {"y": ny}, {"hint": hint}],
                                   guide_scale=7.5, guide_rescale=0.2, solver="dpmpp_2m_sde", solver_mode="normal", steps=2,
                                   t_max=899, t_min=0, discretization="trailing", chunk_inds=list(chunks),
                                   noise_sampler=lambda a, b: torch.randn(x.shape, generator=g)).float())
    err = rel_l2(outs[1], outs[0])
    assert outs[1].shape == (1, 4, 36, 10, 8) and err < 1e-2, err          # CFG 7.5 amplifies the fp16 error (cf. test_unet_gpu)
