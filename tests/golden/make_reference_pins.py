#!/usr/bin/env python
"""Generate tests/golden/reference_pins.npz: what the UNMODIFIED reference (CPU, fp32) returns on the inputs of the pin
tests in tests/test_oracle_vs_reference.py, tests/test_imagenet_cpu.py, tests/test_interleaved_cpu.py and
tests/test_interleaved_vs_reference.py (the last needs the reference's whole source tree: its mllm.py imports ``data``).

  python tests/golden/make_reference_pins.py    # where oracle/ref_harness.py finds the reference

Inputs are not stored: the tests draw them again from the same seeds (weights, images). Of the sampler noise the file keeps
the shapes of the draws, and this script asserts that drawing those shapes again gives exactly what the reference consumed.
The reference ships no golden vectors (SURVEY.md §4): these are the pinned outputs of its own code."""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_pins.npz")


def capture_noise(fn):
    rec = []
    o1, o2 = torch.randn, torch.randn_like
    torch.randn = lambda *a, **k: (rec.append(o1(*a, **k)) or rec[-1])
    torch.randn_like = lambda a, **k: (rec.append(o2(a, **k)) or rec[-1])
    try:
        out = fn()
    finally:
        torch.randn, torch.randn_like = o1, o2
    return out, [r.clone() for r in rec]


def redraw(shapes):
    """The tests' replay of a captured noise sequence: the same global-RNG draws, in order."""
    return [torch.randn(s) for s in shapes]


def replayable(fn):
    """fn()'s output and the shapes of its noise draws, after checking that redraw(shapes) from the same RNG state gives
    back exactly the noise fn consumed."""
    state = torch.get_rng_state()
    out, noise = capture_noise(fn)
    after = torch.get_rng_state()
    shapes = [tuple(n.shape) for n in noise]
    torch.set_rng_state(state)
    assert all(torch.equal(a, b) for a, b in zip(noise, redraw(shapes)))
    torch.set_rng_state(after)
    return out, np.array(shapes)


def quantiser(ref, g):
    sys.path.insert(0, os.path.join(ref.root, "imagenet_gen"))
    from src.gfq import GFQ
    torch.manual_seed(0)
    h = torch.randn(2, 32, 5, 7)
    h[0, 0, 0, 0] = 0.0
    quant, _, idx_list = GFQ(dim=32, num_codebooks=4).eval()(h)
    g["gfq_quant"] = quant.numpy().astype(np.int8)
    g["gfq_idx"] = np.stack([i.numpy().astype(np.int32) for i in idx_list])


def head(ref, g):
    from bitdance_b200.synth import synth_state_dict
    for swiglu, pn in [(True, 16), (True, 64), (False, 4)]:
        cfg = dict(ch_target=32, ch_cond=96, ch_latent=128, depth_latent=4, depth_adanln=2, parallel_num=pn, use_swiglu=swiglu)
        m = ref.fh.DiffHead(**cfg).eval()
        m.load_state_dict(synth_state_dict({k: tuple(v.shape) for k, v in m.state_dict().items()}, seed=1, std=0.05))
        key = f"head_{int(swiglu)}_{pn}"
        g[key + "_spec"] = np.array(json.dumps({k: list(v.shape) for k, v in m.state_dict().items()}))
        torch.manual_seed(0)
        x, t, c = torch.randn(4, pn, 32), torch.rand(4), torch.randn(4, pn, 96)
        g[key + "_net"] = m.net(x, t, c).numpy()
        for cfg_scale in (1.0, 3.0):
            out, shapes = replayable(lambda: m.sample(c, cfg=cfg_scale, num_sampling_steps=6))
            g[f"{key}_sample_{cfg_scale:g}"] = out.numpy()
            g[f"{key}_noise_shapes_{cfg_scale:g}"] = shapes


def autoencoder(ref, g):
    from bitdance_b200.synth import synth_state_dict
    dd = dict(double_z=False, z_channels=32, in_channels=3, out_ch=3, ch=32, ch_mult=[1, 2, 2], num_res_blocks=2)
    m = ref.ae.VQModel(dd).eval()
    m.load_state_dict(synth_state_dict({k: tuple(v.shape) for k, v in m.state_dict().items()}, seed=2, std=0.05))
    g["ae_spec"] = np.array(json.dumps({k: list(v.shape) for k, v in m.state_dict().items()}))
    torch.manual_seed(0)
    x = torch.rand(2, 3, 32, 48) * 2 - 1
    q = m.encode(x)
    g["ae_quant"] = q.numpy().astype(np.int8)
    g["ae_decoded"] = m.decode(q).numpy()


def pipeline(ref, g):
    from transformers import Qwen3Config, Qwen3ForCausalLM
    from bitdance_b200.synth import synth_state_dict
    pn, S, B, guidance = 16, 4, 2, 3.0
    c = dict(hidden_size=128, intermediate_size=256, num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2,
             head_dim=64, rms_norm_eps=1e-6, rope_theta=1e6)
    hf = Qwen3ForCausalLM(Qwen3Config(vocab_size=200, max_position_embeddings=2048, tie_word_embeddings=False, **c)).eval()
    hf.load_state_dict(synth_state_dict({k: tuple(v.shape) for k, v in hf.state_dict().items()}, seed=3, std=0.05))
    head = ref.fh.DiffHead(ch_target=32, ch_cond=128, ch_latent=128, depth_latent=2, depth_adanln=2, parallel_num=pn,
                           use_swiglu=True).eval()
    head.load_state_dict(synth_state_dict({k: tuple(v.shape) for k, v in head.state_dict().items()}, seed=1, std=0.05))
    dd = dict(double_z=False, z_channels=32, in_channels=3, out_ch=3, ch=32, ch_mult=[1, 2, 2], num_res_blocks=1)
    ae = ref.ae.VQModel(dd).eval()
    ae.load_state_dict(synth_state_dict({k: tuple(v.shape) for k, v in ae.state_dict().items()}, seed=2, std=0.05))
    proj = ref.mu.MLPconnector(32, 128, "gelu_pytorch_tanh").eval()
    proj.load_state_dict(synth_state_dict({k: tuple(v.shape) for k, v in proj.state_dict().items()}, seed=4, std=0.05))

    class Tok:
        special = {"<|vision_start|>": 150}

        def encode(self, s):
            return [ord(ch) % 100 for ch in s][:12] if s == "cond" else [7, 8, 9]

        def convert_tokens_to_ids(self, t):
            if t in self.special:
                return self.special[t]
            if t.startswith("<|res_"):
                return 151 + int(t[6:-2]) % 20
            return 172 + int(t[8:-2])

    pipe = object.__new__(ref.t2i.BitDanceT2IPipeline)
    pipe.device, pipe.tokenizer, pipe.llm_model = "cpu", Tok(), hf
    pipe.hidden_size, pipe.ae, pipe.vision_head, pipe.embed_vision_mlp = 128, ae, head, proj
    pipe.vae_patch_size, pipe.parallel_num, pipe.ps = 4, pn, 4
    pipe.build_pos_embed(max_len=1024)
    torch.manual_seed(11)
    img, shapes = replayable(lambda: pipe.gen_image("cond", "uncond", guidance_scale=guidance, num_sampling_steps=S,
                                                      max_length=64, num_images=B, image_size=[32, 32]))
    g["pipeline_image"] = img.numpy()
    g["pipeline_specs"] = np.array(json.dumps({k: {n: list(v.shape) for n, v in mod.state_dict().items()}
                                               for k, mod in (("head", head), ("ae", ae), ("proj", proj))}))
    g["pipeline_noise_shapes"] = shapes


def imagenet(ref, g):
    import torch.nn as nn
    sys.path.insert(0, os.path.join(ref.root, "imagenet_gen"))
    from src import model_parallel as mp

    class _VaeStub(nn.Module):
        def __init__(self, *a, **k):
            super().__init__()

        def decode(self, x):
            return x

    real_vq = mp.VQModel
    mp.VQModel = _VaeStub
    try:
        torch.manual_seed(0)
        model = mp.BitDance(dim=64, n_layer=2, n_head=2, diff_layers=2, diff_dim=64, diff_adanln_layers=1, latent_dim=16,
                            down_size=16, patch_size=1, resolution=64, diff_batch_mul=1, cls_token_num=4,
                            num_classes=10, parallel_num=4, parallel_mode="patch").eval()
    finally:
        mp.VQModel = real_vq
    params = [(n, tuple(p.shape)) for n, p in model.named_parameters()]
    assert [n for n, _ in params] == [k for k in model.state_dict()]   # the state dict holds parameters only
    gen = torch.Generator().manual_seed(1)
    for n, p in model.named_parameters():
        if p.dim() >= 2:
            p.copy_(torch.randn(p.shape, generator=gen) * 0.08)
        elif "norm" in n:
            p.copy_(1.0 + 0.1 * torch.randn(p.shape, generator=gen))
        else:
            p.copy_(torch.randn(p.shape, generator=gen) * 0.05)
    torch.manual_seed(5)
    grid, shapes = replayable(lambda: model.sample(torch.tensor([3, 7]), 4, cfg_scale=3.0, cfg_schedule="linear"))
    g["imagenet_params"] = np.array(json.dumps(params))
    g["imagenet_grid"] = grid.numpy().astype(np.int8)
    g["imagenet_noise_shapes"] = shapes
    g["imagenet_freqs_cis"] = model.freqs_cis.numpy()
    g["imagenet_attn_mask"] = model.attn_mask[0, 0].numpy()
    # tests/test_imagenet_cpu.py: the parameter names and shapes of the small test model
    kw = dict(dim=128, n_layer=2, n_head=2, diff_layers=2, diff_dim=128, diff_adanln_layers=1, latent_dim=32, down_size=16,
              patch_size=1, resolution=64, diff_batch_mul=1, cls_token_num=4, num_classes=10, parallel_num=4,
              parallel_mode="patch")
    with torch.device("meta"):
        small = mp.BitDance(**kw)
    g["imagenet_small_spec"] = np.array(json.dumps({k: list(v.shape) for k, v in small.state_dict().items()}))


def vt_forward(ref, g):
    import types
    import torch.nn.functional as F

    def fake_encode(x, f=16, C=8):
        p = F.avg_pool2d(x, f)
        feats = torch.cat([p * (k + 1) for k in range(C // 3 + 1)], dim=1)[:, :C]
        return torch.where(torch.sin(37.0 * feats) > 0, 1.0, -1.0)

    torch.manual_seed(0)
    sizes = [(64, 64), (96, 64), (64, 64), (128, 96), (96, 64), (64, 64), (64, 64)]
    imgs = [torch.randn(1, 3, h, w) for h, w in sizes]
    stub = types.SimpleNamespace(encode=lambda x: fake_encode(x))
    for ps in (1, 2):
        g[f"vt_forward_ps{ps}"] = ref.ae.VQModel.vt_forward(stub, imgs, max_bs=2, ps=ps).numpy().astype(np.int8)
    sizes2 = [(384, 256), (416, 384), (1024, 512), (512, 512), (1056, 320), (768, 800), (96, 1536)]
    imgs2 = [torch.randn(1, 3, h, w) for h, w in sizes2]
    stub2 = types.SimpleNamespace(encode=lambda x: fake_encode(x, f=32))
    g["vt_forward_maxpad"] = ref.ae.VQModel.vt_forward_maxpad(stub2, imgs2, max_bs=2).numpy().astype(np.int8)


def sampler(ref, g):
    """tests/test_interleaved_cpu.py: top_k_top_p_filtering (as the mask of kept logits) and sample_codebook (tokens)."""
    r = ref.mu
    gen = torch.Generator().manual_seed(0)
    keep, tok_s, tok_a = [], [], []
    for trial in range(120):
        B, V = 3, int(torch.randint(5, 400, (1,), generator=gen))
        logits = torch.randn(B, V, generator=gen) * float(torch.rand(1, generator=gen) * 5 + 0.1)
        if trial % 3 == 0:
            logits = (logits * 2).round() / 2
        k = int(torch.randint(0, V + 50, (1,), generator=gen))
        p = 1.0 if trial % 5 == 0 else float(torch.rand(1, generator=gen))
        mk = int(torch.randint(1, 4, (1,), generator=gen))
        b = r.top_k_top_p_filtering(logits.clone(), k, p, min_tokens_to_keep=mk)
        kept = b > -float("inf")
        assert torch.equal(b, logits.masked_fill(~kept, -float("inf")))
        keep.append(kept.reshape(-1).numpy())
        emb = torch.nn.Embedding(V, 8)
        torch.manual_seed(trial)
        tb, eb = r.sample_codebook(logits.clone(), "text", emb, True, 0.7, k, p)
        assert torch.equal(eb, emb(tb))
        tok_s.append(tb.reshape(-1).numpy())
        tok_a.append(r.sample_codebook(logits.clone(), "text", emb, False, 1.0, k, p)[0].reshape(-1).numpy())
    g["sampler_keep"] = np.packbits(np.concatenate(keep))
    g["sampler_tokens_sampled"] = np.stack(tok_s).astype(np.int32)
    g["sampler_tokens_argmax"] = np.stack(tok_a).astype(np.int32)
    strs = ["<|im_start|>user\nhi<|im_end|>\n<|im_start|>assistant\n", "no markers", "<|im_start|>user\nunterminated",
            "a<|im_start|>user\nx<|im_end|>\nb<|im_start|>user\ny<|im_end|>\n", ""]
    g["remove_first_user_block"] = np.array(json.dumps({s: r.remove_first_user_block(s) for s in strs}))


def interleaved(ref, g):
    """MLLModel.forward_inference_block_causal on the "tiny" weights of bitdance_b200.synthetic.tiny_state_dicts(), fp32:
    the plan [user text, model image] and the editing plan [user text, user image, model image]."""
    from torch import nn
    from oracle import ref_harness as rh
    from oracle import ref_runner as rr
    from bitdance_b200.synthetic import synthetic_tokenizer, tiny_state_dicts
    mllm = rh.import_reference_mllm()
    pipe, _ = rr.build_pipeline("tiny", "cpu")
    sds = tiny_state_dicts()
    missing = pipe.llm_model.load_state_dict(sds["llm"], strict=False)
    assert set(missing.missing_keys) <= {"lm_head.weight"} and not missing.unexpected_keys
    pipe.llm_model.float()
    pipe.vision_head.load_state_dict(sds["head"])
    pipe.ae.load_state_dict(sds["ae"])
    pipe.embed_vision_mlp.load_state_dict(sds["proj"])
    tok, _ = synthetic_tokenizer(512, 16)
    for alias, t in (("im_start", "<|im_start|>"), ("im_end", "<|im_end|>"), ("start_of_image", "<|vision_start|>"),
                     ("end_of_image", "<|vision_end|>")):
        setattr(tok, alias + "_id", tok.convert_tokens_to_ids(t))      # data/data_utils.py:95-109
    for i in range(1, 161):
        setattr(tok, f"res_{i}_id", tok.convert_tokens_to_ids(f"<|res_{i}|>"))
    for i in range(1, 16):
        setattr(tok, f"query_{i}_id", tok.convert_tokens_to_ids(f"<|query_{i}|>"))

    class _Cfg(dict):
        __getattr__ = dict.__getitem__

    M = mllm.MLLModel
    m = M.__new__(M)
    nn.Module.__init__(m)
    m.config = _Cfg(vit_patch_size=pipe.vae_patch_size, head=_Cfg(vision_pred=_Cfg(parallel_num=16)),
                    encoder=_Cfg(vt_forward_func="group", max_bs=32))
    m.tokenizer, m.llm_model, m.vision_head_type = tok, pipe.llm_model, "diffusion_parallel_x"
    m.vision_diffusion_head, m.embed_vision_mlp, m.vision_encoder = pipe.vision_head, pipe.embed_vision_mlp, pipe.ae
    m.parallel_num, m.ps, m.hidden_size = 16, 4, 256
    m.register_buffer("pos_embed_1d", m._get_1d_sincos_pos_embed(128, 64), persistent=False)
    m.eval()
    text = "<|im_start|>user\na photo of the red cat<|im_end|>\n<|im_start|>assistant\n"
    user, model = {"from": "user"}, {"from": "model"}
    torch.manual_seed(5)
    out, shapes = replayable(lambda: m.forward_inference_block_causal(
        [dict(type="text", **user), dict(type="image", **model)], [text], [], max_length_vision=64, sample_steps=3,
        image_size=[32, 32], cfg_scale=3.0))
    assert out["generated_text"] == []
    g["interleaved_t2i_image"] = out["generated_image"][0].numpy()
    g["interleaved_t2i_noise_shapes"] = shapes
    src = torch.rand(1, 3, 32, 32, generator=torch.Generator().manual_seed(1)) * 2 - 1
    plan = [dict(type="text", **user), dict(type="image", **user), dict(type="image", **model)]
    torch.manual_seed(7)
    out, shapes = replayable(lambda: m.forward_inference_block_causal(
        plan, [text], [src.clone()], max_length_vision=64, sample_steps=3, image_size=[32, 32], cfg_scale=3.0))
    g["interleaved_edit_image"] = out["generated_image"][0].numpy()
    g["interleaved_edit_noise_shapes"] = shapes
    g["interleaved_edit_source_latent"] = m.encode_image([src.clone()])[0].float().numpy()


def main():
    from oracle import ref_harness as rh
    ref = rh.import_reference()
    ref.root = rh.REF
    import torch._dynamo
    torch._dynamo.config.disable = True
    g = {}
    with torch.no_grad():
        for fn in (quantiser, head, autoencoder, pipeline, imagenet, vt_forward, sampler, interleaved):
            fn(ref, g)
    np.savez_compressed(OUT, **g)
    print(OUT, os.path.getsize(OUT))


if __name__ == "__main__":
    main()
