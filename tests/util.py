import torch


def rel_l2(got, ref):
    got, ref = got.float(), ref.float()
    return ((got - ref).norm() / ref.norm().clamp_min(1e-12)).item()


def assert_close(got, ref, rel=2e-3, max_rel=2e-2, what=""):
    """fp16-output comparison: relative L2 error and max-abs error relative to max|ref|."""
    assert got.shape == ref.shape, f"{what}: shape {tuple(got.shape)} vs {tuple(ref.shape)}"
    g, r = got.float(), ref.float()
    assert torch.isfinite(g).all(), f"{what}: non-finite values in result"
    e = rel_l2(g, r)
    m = ((g - r).abs().max() / r.abs().max().clamp_min(1e-12)).item()
    assert e <= rel and m <= max_rel, f"{what}: rel-L2 {e:.3e} (tol {rel:.1e}), max-abs/max|ref| {m:.3e} (tol {max_rel:.1e})"
    return e, m


def sample_flat(t, n=4096, seed=0):
    """A fixed, seeded sample of n elements of t (flattened): large golden outputs are stored as this sample."""
    idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(seed))[:n]
    return t.reshape(-1)[idx.to(t.device)].float().cpu()


def load_golden(name):
    """A golden file of tests/golden/ (outputs of the unmodified reference, see oracle/make_golden*.py)."""
    import os
    return torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name))


SMALL_KW = dict(dim_mult=[1, 2, 1, 4], num_res_blocks=1)     # reduced ControlledV2VUNet used by fast tests


def make_inputs(seed, B, F, H, W):
    """Seeded CPU inputs of one denoiser call: latent x, LR-latent hint, text embedding y."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, 4, F, H, W, generator=g)
    hint = 0.5 * torch.randn(B, 4, F, H, W, generator=g)
    y = torch.randn(B, 77, 1024, generator=g)
    return x, hint, y


def synth_model(kw, seed, device="cpu", half=True):
    """star_b200 ControlledV2VUNet with the deterministic synthetic checkpoint (seed)."""
    from star_b200.utils.synth import synth_state_dict
    from star_b200.video_to_video.modules.unet_v2v import ControlledV2VUNet
    with torch.device("meta"):
        net = ControlledV2VUNet(**kw)
    manifest = {k: tuple(v.shape) for k, v in net.state_dict().items()}
    sd = synth_state_dict(manifest, seed=seed)
    net.load_state_dict(sd, assign=True)
    net.eval()
    if half:
        net = net.half()
    if device != "cpu":
        net = net.to(device)
    return net, sd


class FakeDenoiser(torch.nn.Module):
    """Cheap stand-in for the UNet with the same call signature (sampler tests)."""

    def __init__(self):
        super().__init__()
        self.calls = []

    def forward(self, x, t, y=None, hint=None, hint_chunk=None, variant_info=None):
        self.calls.append(int(t[0]))
        h = hint_chunk if hint_chunk is not None else hint
        return torch.tanh(x * 0.7 + 0.3 * h) * (1 + 0.1 * y.mean()) + 0.01 * x.mean(dim=2, keepdim=True)
