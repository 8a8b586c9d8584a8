"""Pin the CPU oracle (oracle/*.py) against the UNMODIFIED reference.

The reference ships no tests or golden vectors (SURVEY.md §4), so its own code run on CPU in fp32 is the pin: what it
returned on these inputs is stored in tests/golden/reference_pins.npz (tests/golden/make_reference_pins.py), and the
inputs, sampler noise included, are drawn again here from the same seeds."""
import json
import os

import numpy as np
import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_pins.npz")


@pytest.fixture(scope="module")
def ref():
    return np.load(GOLDEN)


def _noise(shapes):
    """The noise the reference drew in the stored run: the same global-RNG draws, in order."""
    return [torch.randn(tuple(int(d) for d in s)) for s in shapes]


def test_quantiser_and_gfq_vs_reference(ref):
    from oracle import quant as oq
    torch.manual_seed(0)
    h = torch.randn(2, 32, 5, 7)
    h[0, 0, 0, 0] = 0.0
    assert np.array_equal(ref["gfq_quant"].astype(np.float32), oq.sign_quantize(h.numpy()))
    mine = oq.gfq_indices(h.numpy(), 4)
    for g in range(4):
        assert np.array_equal(ref["gfq_idx"][g], mine[g])
    # VQModel.encode's rule and torch.sign
    cb = torch.tensor([1.0])
    assert np.array_equal(torch.where(h > 0, cb, -cb).numpy(), oq.sign_quantize(h.numpy()))
    x = torch.tensor([0.0, -0.0, float("nan"), 2.0, -3.0])
    assert np.array_equal(torch.sign(x).numpy(), oq.sign_lfq(x.numpy()))


@pytest.mark.parametrize("swiglu,pn", [(True, 16), (True, 64), (False, 4)])
def test_head_and_sampler_vs_reference(ref, swiglu, pn):
    from bitdance_b200.head import head_spec
    from bitdance_b200.synth import synth_state_dict
    from oracle import head as oh
    key = f"head_{int(swiglu)}_{pn}"
    spec = {k: tuple(v) for k, v in json.loads(str(ref[key + "_spec"])).items()}
    assert spec == head_spec(32, 96, 128, 4, 2, swiglu)
    sd = synth_state_dict(spec, seed=1, std=0.05)
    torch.manual_seed(0)
    R = 4
    x, t, c = torch.randn(R, pn, 32), torch.rand(R), torch.randn(R, pn, 96)
    with torch.no_grad():
        assert (torch.from_numpy(ref[key + "_net"]) - oh.head_forward(sd, x, t, c)).abs().max().item() < 2e-5
        for cfg_scale in (1.0, 3.0):
            noise = _noise(ref[f"{key}_noise_shapes_{cfg_scale:g}"])
            mine = oh.euler_maruyama(sd, c, cfg_scale, 6, noise)
            assert (torch.from_numpy(ref[f"{key}_sample_{cfg_scale:g}"]) - mine).abs().max().item() < 2e-4


def test_llm_vs_transformers():
    from transformers import Qwen3Config, Qwen3ForCausalLM
    from bitdance_b200.llm import llm_spec
    from bitdance_b200.synth import synth_state_dict
    from oracle import llm as ol
    from oracle.ref_harness import shim_transformers
    shim_transformers()
    c = dict(hidden_size=128, intermediate_size=256, num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2,
             head_dim=64, rms_norm_eps=1e-6, rope_theta=1e6)
    hf = Qwen3ForCausalLM(Qwen3Config(vocab_size=64, max_position_embeddings=512, tie_word_embeddings=False, **c)).eval()
    spec = {k: tuple(v.shape) for k, v in hf.state_dict().items()}
    assert all(spec[k] == v for k, v in llm_spec(c).items())
    sd = synth_state_dict(spec, seed=3, std=0.05)
    hf.load_state_dict(sd)
    torch.manual_seed(0)
    B, pn = 2, 16
    xs = [torch.randn(B, 9, 128), torch.randn(B, pn, 128), torch.randn(B, pn, 128)]
    cache = [None] * 2
    with torch.no_grad():
        o = hf.model(inputs_embeds=xs[0], use_cache=True)
        pkv = o.past_key_values
        assert (o.last_hidden_state - ol.decoder_forward(sd, c, xs[0], cache, causal=True)).abs().max() < 2e-5
        for x in xs[1:]:
            mask = torch.ones(B, 1, pn, pn + pkv[0][0].shape[2], dtype=torch.bool)
            o = hf.model(inputs_embeds=x, past_key_values=pkv, use_cache=True, attention_mask=mask)
            pkv = o.past_key_values
            assert (o.last_hidden_state - ol.decoder_forward(sd, c, x, cache, causal=False)).abs().max() < 2e-5


def test_autoencoder_vs_reference(ref):
    from bitdance_b200.ae import ae_spec
    from bitdance_b200.synth import synth_state_dict
    from oracle import ae as oa
    dd = dict(double_z=False, z_channels=32, in_channels=3, out_ch=3, ch=32, ch_mult=[1, 2, 2], num_res_blocks=2)
    spec = {k: tuple(v) for k, v in json.loads(str(ref["ae_spec"])).items()}
    assert spec == ae_spec(dd)
    sd = synth_state_dict(spec, seed=2, std=0.05)
    torch.manual_seed(0)
    x = torch.rand(2, 3, 32, 48) * 2 - 1
    q_ref, d_ref = torch.from_numpy(ref["ae_quant"]).float(), torch.from_numpy(ref["ae_decoded"])
    with torch.no_grad():
        q, _ = oa.encode(sd, x)
        assert torch.equal(q, q_ref)                       # token grid: bit-exact
        assert (oa.decoder_forward(sd, q) - d_ref).abs().max().item() < 1e-4


def test_pipeline_vs_reference(ref):
    """Whole gen_image: tiny Qwen3 + head + projector + tokenizer, stub tokenizer, CFG on, 2 images."""
    from transformers import Qwen3Config, Qwen3ForCausalLM
    from bitdance_b200.synth import synth_state_dict
    from oracle import pipeline as op
    pn, S, B, guidance = 16, 4, 2, 3.0
    c = dict(hidden_size=128, intermediate_size=256, num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2,
             head_dim=64, rms_norm_eps=1e-6, rope_theta=1e6)
    hf = Qwen3ForCausalLM(Qwen3Config(vocab_size=200, max_position_embeddings=2048, tie_word_embeddings=False, **c))
    sd_llm = synth_state_dict({k: tuple(v.shape) for k, v in hf.state_dict().items()}, seed=3, std=0.05)
    specs = {k: {n: tuple(v) for n, v in d.items()} for k, d in json.loads(str(ref["pipeline_specs"])).items()}
    sd_head = synth_state_dict(specs["head"], seed=1, std=0.05)
    sd_ae = synth_state_dict(specs["ae"], seed=2, std=0.05)
    sd_proj = synth_state_dict(specs["proj"], seed=4, std=0.05)

    class Tok:
        special = {"<|vision_start|>": 150}

        def encode(self, s):
            return [ord(ch) % 100 for ch in s][:12] if s == "cond" else [7, 8, 9]

        def convert_tokens_to_ids(self, t):
            if t in self.special:
                return self.special[t]
            if t.startswith("<|res_"):
                return 151 + int(t[6:-2]) % 20
            return 172 + int(t[8:-2])  # <|query_i|>

    Himg = Wimg = 32  # 8 x 8 latent = 64 tokens = 4 AR steps
    img_ref = torch.from_numpy(ref["pipeline_image"])
    torch.manual_seed(11)
    noise = _noise(ref["pipeline_noise_shapes"])
    steps = 64 // pn
    assert len(noise) == steps * (S + 1)
    per_step = [noise[i * (S + 1):(i + 1) * (S + 1)] for i in range(steps)]
    tok = Tok()
    start = [tok.convert_tokens_to_ids("<|vision_start|>"), tok.convert_tokens_to_ids("<|res_8|>"),
             tok.convert_tokens_to_ids("<|res_8|>")] + [tok.convert_tokens_to_ids(f"<|query_{i}|>") for i in range(1, pn)]
    with torch.no_grad():
        tokens, img = op.gen_image(sd_llm=sd_llm, cfg_llm=c, embed=sd_llm["model.embed_tokens.weight"], sd_head=sd_head,
                                   sd_proj=sd_proj, sd_ae=sd_ae, cond_ids=tok.encode("cond"), uncond_ids=tok.encode("u"),
                                   start_ids=start, h=8, w=8, pn=pn, num_images=B, guidance=guidance, S=S,
                                   noise=per_step, head_dim=128)
    assert img.shape == img_ref.shape == (B, 3, Himg, Wimg)
    assert (img - img_ref).abs().max().item() < 1e-3 * max(1.0, img_ref.abs().max().item())


def test_imagenet_sample_vs_reference(ref):
    """SURVEY.md section 8 row a16: oracle/imagenet.py::sample against the unmodified ``BitDance.sample``
    (imagenet_gen/src/model_parallel.py:372-419) — tiny dims, CFG on with the linear ramp, noise replayed from the
    reference's own torch.randn calls. Harness-side shims of the stored run (no arithmetic under test changes): the
    460 M-parameter VAE is replaced by a stub whose decode is the identity (the tokenizer is pinned separately),
    torch.compile is disabled (CPU), the tensors the reference zero-initialises are re-randomised (SURVEY.md F8)."""
    from oracle import imagenet as oi
    cfg = dict(dim=64, n_layer=2, n_head=2, resolution=64, down_size=16, patch_size=1, cls_token_num=4, parallel_num=4,
               num_classes=10, latent_dim=16, parallel_mode="patch")
    # the reference module's parameters, in its order, re-randomised as in the stored run
    g = torch.Generator().manual_seed(1)
    sd = {}
    for n, shape in json.loads(str(ref["imagenet_params"])):
        if len(shape) >= 2:
            sd[n] = torch.randn(shape, generator=g) * 0.08
        elif "norm" in n:
            sd[n] = 1.0 + 0.1 * torch.randn(shape, generator=g)
        else:
            sd[n] = torch.randn(shape, generator=g) * 0.05
    cls_ids = torch.tensor([3, 7])
    S = 4
    torch.manual_seed(5)
    rec = _noise(ref["imagenet_noise_shapes"])
    steps = (cfg["resolution"] // 16) ** 2 // cfg["parallel_num"]
    assert len(rec) == steps * (S + 1)
    noise = [rec[i * (S + 1):(i + 1) * (S + 1)] for i in range(steps)]
    with torch.no_grad():
        tokens, grid = oi.sample(sd, cfg, cls_ids, S, 3.0, noise)
    ref_grid = torch.from_numpy(ref["imagenet_grid"]).float()
    assert grid.shape == ref_grid.shape == (2, 16, 4, 4)
    agree = (grid == ref_grid).float().mean().item()
    assert agree == 1.0, f"token grid agreement {agree}"
    # buffers
    fc, mask, h, w = oi.make_buffers(cfg)
    assert torch.equal(fc, torch.from_numpy(ref["imagenet_freqs_cis"]))
    assert torch.equal(mask, torch.from_numpy(ref["imagenet_attn_mask"]))


def test_vt_forward_host_logic_vs_reference(ref):
    """SURVEY.md section 8 row a4: the image-list bucketing / flattening of ``VQModel.vt_forward`` and
    ``vt_forward_maxpad`` (autoencoder.py:402-511) is host logic re-expressed in the API mirror; both versions are driven
    with the same stand-in ``encode`` (the convolutional encoder is pinned separately) and must agree exactly."""
    import types
    import torch.nn.functional as F
    from bitdance_b200.modeling.vision_encoder.autoencoder import VQModel as Mine

    def fake_encode(x, f=16, C=8):
        p = F.avg_pool2d(x, f)                                    # [B, 3, H/f, W/f]
        feats = torch.cat([p * (k + 1) for k in range(C // 3 + 1)], dim=1)[:, :C]
        return torch.where(torch.sin(37.0 * feats) > 0, 1.0, -1.0)

    torch.manual_seed(0)
    sizes = [(64, 64), (96, 64), (64, 64), (128, 96), (96, 64), (64, 64), (64, 64)]
    imgs = [torch.randn(1, 3, h, w) for h, w in sizes]
    stub = types.SimpleNamespace(encode=lambda x: fake_encode(x))
    for ps in (1, 2):
        a = torch.from_numpy(ref[f"vt_forward_ps{ps}"]).float()
        b = Mine.vt_forward(stub, imgs, max_bs=2, ps=ps)
        assert a.shape == b.shape and torch.equal(a, b)
    # maxpad: stride 32 with a stride-32 stand-in encoder; includes a "long" image and every normal bucket boundary
    sizes2 = [(384, 256), (416, 384), (1024, 512), (512, 512), (1056, 320), (768, 800), (96, 1536)]
    imgs2 = [torch.randn(1, 3, h, w) for h, w in sizes2]
    stub2 = types.SimpleNamespace(encode=lambda x: fake_encode(x, f=32))
    a = torch.from_numpy(ref["vt_forward_maxpad"]).float()
    b = Mine.vt_forward_maxpad(stub2, imgs2, max_bs=2)
    assert a.shape == b.shape and torch.equal(a, b)
