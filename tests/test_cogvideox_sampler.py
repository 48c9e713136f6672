"""CogVideoX sampling loop (VPSDEDPMPP2MSampler + DynamicCFG + DiscreteDenoiser / VideoScaling) against outputs of the reference's
UNMODIFIED sgm/modules/diffusionmodules files (oracle/cogvideox_sampler.py), stored by oracle/make_golden_reference.py."""
import pytest
import torch

from tests.util import load_golden, rel_l2, sample_flat


class FakeDiT(torch.nn.Module):
    """cheap deterministic stand-in with the DiffusionTransformer call signature: (2B, T, 32, h, w) -> (2B, T, 16, h, w)"""

    def __init__(self):
        super().__init__()
        self.calls = []

    def forward(self, x, timesteps=None, context=None, y=None, **kw):
        self.calls.append(float(timesteps[0]))
        noisy, lq = x.float().chunk(2, dim=2)
        t = timesteps.float().view(-1, 1, 1, 1, 1) / 1000.0
        c = context.float().mean(dim=(1, 2)).view(-1, 1, 1, 1, 1)
        return torch.tanh(0.8 * noisy - 0.3 * lq + 0.1 * noisy.mean(dim=1, keepdim=True)) * (1.0 + 0.2 * c) + 0.05 * t * lq


def test_step_plan_matches_reference_tables():
    from star_b200.cogvideox.sampling import StepPlan
    gold, tables = load_golden("reference_cpu.pt")["sampler"], load_golden("cogvideox_path.pt")
    acs, timesteps = tables["acs"], tables["timesteps"]
    plan = StepPlan()
    assert gold["num_sigmas"] == 51 and torch.equal(plan.alphas_cumprod_sqrt, acs)
    assert plan.timesteps == timesteps
    for i, st in enumerate(plan.steps):                                   # quantised sigma of the denoiser, guidance scale
        assert st.c_skip == float(tables["sigma_q"][i]) and st.timestep == timesteps[-(i + 1)]
        assert st.cfg_scale == tables["cfg"][i]
    assert [st.last for st in plan.steps] == [False] * 49 + [True]


@pytest.mark.parametrize("steps", [50, 6])
def test_sampler_matches_reference(steps):
    from oracle.make_golden_cogvideox import sampler_inputs
    from star_b200.cogvideox.sampling import VPSDEDPMPP2MSampler
    gold = load_golden("reference_cpu.pt")["sampler"]["runs"][steps]
    lq, randn, cond, uc = sampler_inputs()
    net_m = FakeDiT()
    mine = VPSDEDPMPP2MSampler(num_steps=steps, dtype=torch.float32)
    torch.manual_seed(123)
    got = mine(net_m, randn.clone(), cond, uc=uc, lq=torch.cat((lq, lq), 0))
    assert net_m.calls == gold["calls"] and len(net_m.calls) == steps
    assert got.shape == gold["out"].shape == randn.shape
    assert rel_l2(got, gold["out"]) < 2e-5
    # random-stream consumption: 1 draw in the first step, 2 in every later one but the last (sampling.py:635,:641)
    after = torch.randn(4)
    torch.manual_seed(123)
    for _ in range(2 * steps - 3):
        torch.randn_like(randn)
    assert torch.equal(after, torch.randn(4))


def pipeline_nets(dit_kw, vae_kw, dtype, device):
    """star_b200 DiT, 3-D VAE encoder / decoder with the weights of the stored reference runs, and the text context"""
    from tests.test_cogvideox import dit_inputs, dit_net
    from tests.test_cogvideox_vae import _decoder, _encoder
    return dit_net(dit_kw, dtype, device), _encoder(vae_kw, device=device, dtype=dtype), \
        _decoder(vae_kw, device=device, dtype=dtype), dit_inputs(dit_kw)[2].to(device)


def pipeline_lq(F, H, W):
    """LQ clip (1, F, 3, H, W), already upsampled"""
    return torch.rand(1, F, 3, H, W, generator=torch.Generator().manual_seed(9)) * 2 - 1


def test_cogvideox_pipeline_host_graph_on_emulated_kernels(monkeypatch):
    """LQ frames -> frames through 3-D VAE encode + DiT + sampler + 3-D VAE decode (reduced sizes, 4 steps) against the same chain of
    reference modules"""
    from oracle import kernel_ref as KR
    from star_b200 import ops
    from star_b200.cogvideox import sample_sr
    from tests.test_cogvideox import SMALL_DIT
    from tests.test_cogvideox_vae import SMALL
    gold = load_golden("reference_cpu.pt")["pipeline"]
    for name in dir(KR):
        if not name.startswith("_") and callable(getattr(KR, name)) and hasattr(ops, name):
            monkeypatch.setattr(ops, name, getattr(KR, name))
    net, enc, dec, ctx = pipeline_nets(SMALL_DIT, SMALL, torch.float16, "cpu")
    cond, uc = {"crossattn": ctx[:1]}, {"crossattn": torch.zeros_like(ctx[:1])}
    got, z = sample_sr(net, dec, cond, uc, lq=pipeline_lq(9, 64, 96), encoder=enc, num_steps=4, seed=77)
    assert got.shape == (1, 9, 3, 64, 96)
    assert rel_l2(sample_flat(z), gold["z"]) < 1e-2 and rel_l2(sample_flat(got), gold["frames"]) < 1e-2


FULL_WIDTH_PIPELINE_DIT = dict(num_layers=2, hidden_size=3072, num_attention_heads=48, num_frames=17, latent_height=16, latent_width=24,
                               text_length=226, text_hidden_size=4096, lora_r=64, time_embed_dim=512)


@pytest.mark.gpu
def test_cogvideox_pipeline_gpu():
    """the same chain on the B200 kernels: full-width DiT (2 layers), full-width 3-D VAE decoder, 6 sampler steps, fp16"""
    from star_b200.cogvideox import sample_sr
    gold = load_golden("reference_gpu.pt")["pipeline"]
    net, enc, dec, ctx = pipeline_nets(FULL_WIDTH_PIPELINE_DIT, {}, torch.float16, "cuda")
    cond, uc = {"crossattn": ctx[:1]}, {"crossattn": torch.zeros_like(ctx[:1])}
    got, z = sample_sr(net, dec, cond, uc, lq=pipeline_lq(17, 128, 192).cuda(), encoder=enc, num_steps=6, seed=5)
    e_z, e_x = rel_l2(sample_flat(z), gold["z"]), rel_l2(sample_flat(got), gold["frames"])
    print(f"[cogvideox pipeline fp16, 6 steps] latent rel-L2 {e_z:.2e}, frames rel-L2 {e_x:.2e}")
    assert got.shape == (1, 17, 3, 128, 192) and torch.isfinite(got).all()
    assert e_z < 2e-2 and e_x < 2e-2


# ---------------------------------------------------------------------------------------------------- 2 ranks (gloo, CPU)
def _split_worker(rank, world, port, q):
    import os
    import torch.distributed as dist
    from star_b200.cogvideox.sampling import VPSDEDPMPP2MSampler, split_cfg_pair
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        g = torch.Generator().manual_seed(0)
        lq = torch.randn(1, 3, 16, 6, 8, generator=g)
        randn = torch.randn(1, 3, 16, 6, 8, generator=g)
        cond, uc = {"crossattn": torch.randn(1, 226, 32, generator=g)}, {"crossattn": torch.zeros(1, 226, 32)}
        net = FakeDiT()
        torch.manual_seed(123)
        out = VPSDEDPMPP2MSampler(num_steps=6, dtype=torch.float32)(split_cfg_pair(net), randn, cond, uc=uc, lq=torch.cat((lq, lq), 0))
        q.put((rank, out.numpy(), len(net.calls)))
    finally:
        dist.destroy_process_group()


def test_cfg_pair_split_two_ranks_equals_single():
    """CogVideoX multi-GPU axis: the CFG pair over 2 ranks (one all-gather per step) == the batch-2 run, bit for bit, on both ranks"""
    import socket
    import torch.multiprocessing as mp
    from star_b200.cogvideox.sampling import VPSDEDPMPP2MSampler
    g = torch.Generator().manual_seed(0)
    lq = torch.randn(1, 3, 16, 6, 8, generator=g)
    randn = torch.randn(1, 3, 16, 6, 8, generator=g)
    cond, uc = {"crossattn": torch.randn(1, 226, 32, generator=g)}, {"crossattn": torch.zeros(1, 226, 32)}
    torch.manual_seed(123)
    single = VPSDEDPMPP2MSampler(num_steps=6, dtype=torch.float32)(FakeDiT(), randn, cond, uc=uc, lq=torch.cat((lq, lq), 0))
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_split_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=120) for _ in procs], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, out, ncalls in res:
        assert ncalls == 6                                                     # one single-branch forward per step and rank
        assert torch.equal(torch.from_numpy(out), single)
