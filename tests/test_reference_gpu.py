"""The oracle's autocast-bf16 mode (``rnd=bf16`` — what every GPU parity test compares against) pinned against the UNMODIFIED
reference running on a B200 under the real ``torch.autocast("cuda", bfloat16)`` (the reference's deployment, t2i_pipeline.py:130),
and the native engine against that same reference run end to end. What the reference returned on the B200 is stored in
tests/golden/reference_gpu_pins.npz (tests/golden/make_reference_gpu_pins.py); weights and inputs are drawn again here from
the same seeds. Only the engine test needs a GPU: the oracle pins compare stored device outputs with CPU arithmetic."""
import os

import numpy as np
import pytest
import torch

@pytest.fixture(scope="module")
def ref():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_gpu_pins.npz"))


def _noise(ref, key):
    flat, out, o = torch.from_numpy(ref[key]), [], 0
    for s in ref[key + "_shapes"]:
        n = int(np.prod(s))
        out.append(flat[o:o + n].view(*(int(d) for d in s)))
        o += n
    return out


def _ulps(a, b):
    """max |a - b| in units of the bf16 spacing at max|b|"""
    scale = b.abs().max().item()
    return (a - b).abs().max().item() / (2.0 ** -8 * max(scale, 1e-6))


def test_head_network_cuda_autocast_vs_oracle_bf16(ref):
    from bitdance_b200.head import head_spec
    from bitdance_b200.synth import synth_state_dict
    from oracle import head as oh
    sd = synth_state_dict(head_spec(32, 256, 256, 4, 2, True), seed=1, std=0.05)
    torch.manual_seed(0)
    R, pn = 4, 16
    x, t, c = torch.randn(R, pn, 32), torch.rand(R), torch.randn(R, pn, 256)
    out = torch.from_numpy(ref["head_net"])
    with torch.no_grad():
        o_bf = oh.head_forward(sd, x, t, c, rnd=oh.bf16)
        o_32 = oh.head_forward(sd, x, t, c, rnd=oh.ident)
    e_bf, e_32 = (out - o_bf).abs().max().item(), (out - o_32).abs().max().item()
    print(f"reference head under CUDA autocast vs oracle: rnd=bf16 max err {e_bf:.4f} ({_ulps(out, o_bf):.1f} bf16 ulps), "
          f"rnd=ident (fp32) {e_32:.4f}")
    assert _ulps(out, o_bf) <= 6.0          # same rounding points, different accumulation order (cuBLAS vs torch CPU)
    assert e_bf <= e_32 + 1e-3              # the bf16 policy explains the reference's output at least as well as exact math


def test_tokenizer_cuda_autocast_vs_oracle_bf16(ref):
    from bitdance_b200.ae import ae_spec
    from bitdance_b200.synth import synth_state_dict
    from oracle import ae as oa
    dd = dict(double_z=False, z_channels=32, in_channels=3, out_ch=3, ch=32, ch_mult=[1, 2, 2], num_res_blocks=2)
    sd = synth_state_dict(ae_spec(dd), seed=2, std=0.05)
    torch.manual_seed(0)
    x = torch.rand(2, 3, 32, 48) * 2 - 1
    lat, q = torch.from_numpy(ref["ae_latent"]), torch.from_numpy(ref["ae_quant"]).float()
    dec = torch.from_numpy(ref["ae_decoded"])
    with torch.no_grad():
        q_o, lat_o = oa.encode(sd, x, rnd=oa.bf16)
        dec_o = oa.decoder_forward(sd, q, rnd=oa.bf16)
    e_lat = (lat - lat_o).abs().max().item()
    print(f"reference tokenizer under CUDA autocast vs oracle rnd=bf16: latent err {e_lat:.4f} (scale {lat_o.abs().max().item():.2f}), "
          f"token agreement {(q == q_o).float().mean().item():.4f}, decode err {(dec - dec_o).abs().max().item():.4f}")
    assert e_lat < 2e-2 * lat_o.abs().max().item() + 1e-3
    safe = lat_o.abs() > e_lat + 1e-3
    assert torch.equal(q[safe], q_o[safe])
    assert (dec - dec_o).abs().max().item() < 3e-2 * dec_o.abs().max().item() + 1e-2


def test_llm_cuda_autocast_vs_oracle_bf16(ref):
    """bf16 Qwen3 on the GPU exactly as the pipeline drives it: causal prefill (bf16 stream), first block with the all-ones
    mask, then an AR block whose inputs_embeds are fp32 (bf16 MLP output + fp32 pos-embed, t2i_pipeline.py:253)."""
    from transformers import Qwen3Config, Qwen3ForCausalLM
    from bitdance_b200.synth import synth_state_dict
    from oracle import llm as ol
    c = dict(hidden_size=256, intermediate_size=512, num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2,
             head_dim=128, rms_norm_eps=1e-6, rope_theta=1e6)
    hf = Qwen3ForCausalLM(Qwen3Config(vocab_size=64, max_position_embeddings=512, tie_word_embeddings=False, **c))
    spec = {k: tuple(v.shape) for k, v in hf.state_dict().items()}
    sd = {k: v.to(torch.bfloat16).float() for k, v in synth_state_dict(spec, seed=3, std=0.05).items()}
    torch.manual_seed(0)
    B, pn = 2, 16
    x0 = torch.randn(B, 9, 256).to(torch.bfloat16).float()
    x1 = torch.randn(B, pn, 256).to(torch.bfloat16).float()
    x2 = torch.randn(B, pn, 256)                                   # fp32 AR input
    cache = [None] * 2
    errs = []
    with torch.no_grad():
        r0 = ol.decoder_forward(sd, c, x0, cache, causal=True, rnd=ol.bf16, stream_f32=False)
        errs.append(((torch.from_numpy(ref["llm_h0"]) - r0).abs().max() / r0.abs().max()).item())
        for i, (x, f32) in enumerate(((x1, False), (x2, True)), 1):
            r = ol.decoder_forward(sd, c, x, cache, causal=False, rnd=ol.bf16, stream_f32=f32)
            errs.append(((torch.from_numpy(ref[f"llm_h{i}"]) - r).abs().max() / r.abs().max()).item())
    print("reference Qwen3 (transformers, bf16, CUDA autocast) vs oracle rnd=bf16, rel err prefill / block / fp32-stream AR block:",
          [round(e, 4) for e in errs])
    assert max(errs) < 3e-2


@pytest.mark.gpu
def test_engine_vs_unmodified_reference_gen_image_on_gpu(ref):
    """The whole ``gen_image`` of the reference on this GPU (tiny models, CUDA autocast, its own torch.randn draws recorded)
    against the native engine fed the same token ids and the same noise: first-block tokens agree, decoded images are close."""
    from oracle import ref_runner as rr
    from bitdance_b200.synthetic import MODELS, engine_from_state_dicts, tiny_state_dicts
    pn = MODELS["tiny"]["parallel_num"]
    sds = tiny_state_dicts()          # the weights the stored reference run was loaded with
    S, guidance, B, px = 3, 3.0, 1, 32
    img_ref = torch.from_numpy(ref["gen_image"])
    rec = _noise(ref, "gen_image_noise")
    steps = 64 // pn
    assert len(rec) == steps * (S + 1)
    noise = [torch.stack(rec[i * (S + 1):(i + 1) * (S + 1)]).float().contiguous() for i in range(steps)]
    eng = engine_from_state_dicts(sds, "tiny", "cuda")
    it = iter(noise)
    eng.head.draw_noise = lambda b, p, s: next(it).cuda().contiguous()
    tok = rr.StubTokenizer(MODELS["tiny"]["llm"]["vocab_size"])   # the reference pipeline's tokenizer in that run
    emb = sds["llm"]["model.embed_tokens.weight"]
    bf = lambda ids: emb[ids].to(torch.bfloat16).cuda()
    h = w = px // 4                                             # vae_patch_size of the tiny tokenizer
    start = [tok.convert_tokens_to_ids("<|vision_start|>"), tok.convert_tokens_to_ids(f"<|res_{h}|>"),
             tok.convert_tokens_to_ids(f"<|res_{w}|>")] + [tok.convert_tokens_to_ids(f"<|query_{i}|>") for i in range(1, pn)]
    tokens, _ = eng.gen_tokens(bf(tok.encode("cond")), bf(tok.encode("uncond")), bf(start), h=h, w=w, num_images=B,
                               guidance_scale=guidance, num_sampling_steps=S)
    img = eng.decode(tokens, h, w).float().cpu()
    d = (img - img_ref).abs()
    print(f"engine vs the unmodified reference gen_image on this GPU: image |diff| max {d.max().item():.3f} mean "
          f"{d.mean().item():.4f} (scale {img_ref.abs().max().item():.2f})")
    # pixels only: a token that flips in the chaotic sampler changes its 4 x 4-pixel neighbourhood (measured mean 7.6 %)
    assert d.mean().item() < 0.15 * img_ref.abs().max().item()
