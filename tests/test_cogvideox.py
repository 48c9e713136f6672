"""CogVideoX-5B DiT layer (STAR's patched block).  PARITY UNPINNED: the oracle (oracle/cogvideox_ref.py) restates
STAR's layer_forward on top of sat's default leaf modules, which are not in the reference tree."""
import pytest
import torch

from tests.util import load_golden, rel_l2, sample_flat


def _setup(cfg_kw, seed=3):
    from oracle.cogvideox_ref import DiTCfg, layer_manifest, rope_tables
    from star_b200.utils.synth import synth_state_dict
    cfg = DiTCfg(**cfg_kw)
    sd = synth_state_dict(layer_manifest(cfg), seed=seed)
    cos, sin = rope_tables(cfg)
    g = torch.Generator().manual_seed(0)
    S = cfg.text_length + cfg.frames * cfg.height * cfg.width
    hidden = torch.randn(2, S, cfg.hidden, generator=g)
    emb = torch.randn(2, 512, generator=g)
    return cfg, sd, cos, sin, hidden, emb


def test_dit_layer_host_graph_on_emulated_kernels(monkeypatch):
    from oracle import kernel_ref as KR
    from oracle.cogvideox_ref import dit_layer_forward
    from star_b200 import ops
    from star_b200.cogvideox import DiTLayer
    for name in dir(KR):
        if not name.startswith("_") and callable(getattr(KR, name)) and hasattr(ops, name):
            monkeypatch.setattr(ops, name, getattr(KR, name))
    cfg, sd, cos, sin, hidden, emb = _setup(dict(hidden=256, heads=4, text_length=10, frames=3, height=6, width=5))
    ref = dit_layer_forward(sd, hidden, emb, cfg, cos, sin)
    layer = DiTLayer(sd, cfg.hidden, cfg.heads, cfg.text_length, cfg.frames, cfg.height, cfg.width, cfg.ln_eps,
                     cfg.qk_ln_eps, cos, sin, device="cpu")
    assert rel_l2(layer.forward(hidden, emb), ref) < 2e-3


def test_rope_tables_shape():
    from oracle.cogvideox_ref import DiTCfg, rope_tables
    cos, sin = rope_tables(DiTCfg())
    assert cos.shape == (13 * 30 * 45, 64) and torch.allclose(cos ** 2 + sin ** 2, torch.ones_like(cos), atol=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg_kw", [dict(hidden=256, heads=4, text_length=10, frames=3, height=6, width=5),
                                    dict(hidden=3072, heads=48, text_length=226, frames=2, height=6, width=10)])
def test_dit_layer_gpu(cfg_kw):
    """full-width layer (3072 / 48 heads / 226 text tokens) at a short sequence, and a small layer"""
    from oracle.cogvideox_ref import dit_layer_forward
    from star_b200.cogvideox import DiTLayer
    cfg, sd, cos, sin, hidden, emb = _setup(cfg_kw)
    ref = dit_layer_forward(sd, hidden, emb, cfg, cos, sin)
    layer = DiTLayer(sd, cfg.hidden, cfg.heads, cfg.text_length, cfg.frames, cfg.height, cfg.width, cfg.ln_eps,
                     cfg.qk_ln_eps, cos, sin, device="cuda")
    out = layer.forward(hidden.cuda(), emb.cuda())
    torch.cuda.synchronize()
    err = rel_l2(out.cpu(), ref)
    print(f"DiT layer {cfg_kw}: rel-L2 vs fp32 oracle {err:.3e}")
    assert err < 3e-3


# ------------------------------------------------------------------------------------------------------------------
# Whole DiffusionTransformer (patch embed, text proj, time embed, N layers with LoRA, final LayerNorm, final layer,
# unpatchify) against outputs of the REFERENCE'S OWN FILES executed behind the sat shim (oracle/cogvideox_sat.py), stored
# by oracle/make_golden_reference.py in tests/golden/reference_cpu.pt and reference_gpu.pt.
SMALL_DIT = dict(num_layers=2, hidden_size=128, num_attention_heads=2, num_frames=9, latent_height=8, latent_width=12,
                 text_length=6, text_hidden_size=32, lora_r=8, time_embed_dim=64)
FULL_WIDTH_DIT = dict(num_layers=2, hidden_size=3072, num_attention_heads=48, num_frames=9, latent_height=16, latent_width=20,
                      text_length=226, text_hidden_size=4096, lora_r=64, time_embed_dim=512)
# reference state-dict entries star_b200's DiffusionTransformer recomputes instead of loading (rope tables)
DIT_DERIVED = ("mixins.pos_embed.freqs_", "transformer.position_embeddings.weight")


def dit_weights(manifest, seed=4):
    """synthetic non-zero weights for a DiffusionTransformer state-dict manifest {key: shape}"""
    from star_b200.utils.synth import synth_tensor
    sd = {}
    for k, shape in manifest.items():
        t = synth_tensor(k, shape, seed)
        if k.endswith("temp_local.conv1.weight") or k.endswith("spa_local.conv1.weight"):
            t = t * 0.5
        if ".matrix_B." in k:                              # LoRA B is zero-initialised by sat: make the merge matter
            t = t * 8.0
        sd[k] = t
    return sd


def dit_inputs(kw):
    """seeded (x, timesteps, context) of one DiT call"""
    g = torch.Generator().manual_seed(1)
    frames = (kw["num_frames"] - 1) // 4 + 1
    x = torch.randn(2, frames, 32, kw["latent_height"], kw["latent_width"], generator=g)
    ctx = torch.randn(2, kw["text_length"], kw["text_hidden_size"], generator=g)
    return x, torch.tensor([731, 12]), ctx


def dit_net(kw, dtype, device):
    """star_b200 DiffusionTransformer with dit_weights"""
    from star_b200.cogvideox import DiffusionTransformer
    net = DiffusionTransformer(**kw, dtype=dtype)
    net.load_state_dict(dit_weights({k: v.shape for k, v in net.state_dict().items()}))
    return net.to(device)


def _emulate(monkeypatch):
    from oracle import kernel_ref as KR
    from star_b200 import ops
    for name in dir(KR):
        if not name.startswith("_") and callable(getattr(KR, name)) and hasattr(ops, name):
            monkeypatch.setattr(ops, name, getattr(KR, name))


def test_dit_model_host_graph_vs_reference_files(monkeypatch):
    """CPU: star_b200's host graph (im2col patch embed, LoRA merge, adaLN folding, layer stack, final layer, unpatchify) on the
    emulated kernels against the reference's unmodified DiffusionTransformer (sat shimmed); same state-dict layout."""
    gold = load_golden("reference_cpu.pt")
    _emulate(monkeypatch)
    net = dit_net(SMALL_DIT, torch.float16, "cpu")
    assert {k: tuple(v.shape) for k, v in net.state_dict().items()} == \
           {k: s for k, s in gold["dit_manifest"].items() if not k.startswith(DIT_DERIVED)}
    x, t, ctx = dit_inputs(SMALL_DIT)
    got = net(x, timesteps=t, context=ctx)
    want = gold["dit_out"]
    assert got.shape == want.shape == (2, 3, 16, 8, 12)
    err = rel_l2(got, want)
    print(f"DiT model host graph vs reference files: rel-L2 {err:.3e}")
    assert err < 3e-3


RESTATED_LAYER_DIT = dict(SMALL_DIT, num_layers=1, lora_r=0)


def restated_layer_inputs():
    """(hidden, emb) of the one-layer check below: text 6 + 3 x 4 x 6 patches, hidden 128"""
    g = torch.Generator().manual_seed(2)
    return torch.randn(2, 6 + 72, 128, generator=g), torch.randn(2, 64, generator=g)


def test_restated_layer_oracle_is_pinned_to_reference_files():
    """oracle/cogvideox_ref.py (the line-by-line restatement the layer tests use) == the reference's layer_forward"""
    from oracle.cogvideox_ref import DiTCfg, dit_layer_forward
    from star_b200.cogvideox import DiffusionTransformer, rope_tables
    with torch.device("meta"):
        manifest = {k: v.shape for k, v in DiffusionTransformer(**RESTATED_LAYER_DIT, dtype=torch.float16).state_dict().items()}
    sd = dit_weights(manifest)
    cfg = DiTCfg(hidden=128, heads=2, text_length=6, frames=3, height=4, width=6)
    lsd = {"adaLN_modulation.1.weight": sd["mixins.adaln_layer.adaLN_modulations.0.1.weight"],
           "adaLN_modulation.1.bias": sd["mixins.adaln_layer.adaLN_modulations.0.1.bias"]}
    for k, v in sd.items():
        if k.startswith("transformer.layers.0."):
            lsd[k[len("transformer.layers.0."):]] = v
    for n in ("query", "key"):
        lsd[n + "_layernorm.weight"] = sd[f"mixins.adaln_layer.{n}_layernorm_list.0.weight"]
        lsd[n + "_layernorm.bias"] = sd[f"mixins.adaln_layer.{n}_layernorm_list.0.bias"]
    hidden, emb = restated_layer_inputs()
    cos, sin = rope_tables(3, 4, 6, 64)
    got = dit_layer_forward(lsd, hidden, emb, cfg, cos, sin)
    assert rel_l2(sample_flat(got), load_golden("reference_cpu.pt")["dit_layer_out"]) < 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,tol", [(torch.float16, 4e-3), (torch.bfloat16, 2.5e-2)])
def test_dit_model_gpu_vs_reference_files(dtype, tol):
    """GPU: the whole (reduced-depth, full-width) DiT on the fp16 and bf16 kernel libraries vs the reference files in fp32;
    the error of the reference's own low-precision path (module.to(dtype), as sample_sr.py runs it) on the B200 bounds it."""
    gold = load_golden("reference_gpu.pt")["dit"]
    net = dit_net(FULL_WIDTH_DIT, dtype, "cuda")
    x, t, ctx = (v.cuda() for v in dit_inputs(FULL_WIDTH_DIT))
    got = net(x, timesteps=t, context=ctx).float().cpu()
    err, err_ref = rel_l2(sample_flat(got), gold["out"]), gold["err_ref"][str(dtype)]
    print(f"DiT model [{dtype}] 2 layers x 3072: rel-L2 vs reference fp32 {err:.3e} (reference's own {dtype} path: {err_ref:.3e})")
    assert torch.isfinite(got).all() and err < tol and err < 2.0 * err_ref + 1e-3
