#!/usr/bin/env python
"""Generate tests/golden/reference_gpu_pins.npz: what the UNMODIFIED reference returns on a B200 under
``torch.autocast("cuda", bfloat16)`` (its deployment, t2i_pipeline.py:130) on the inputs of tests/test_reference_gpu.py and
tests/test_imagenet_gpu.py::test_imagenet_vs_unmodified_reference_on_gpu. Weights and inputs are drawn again by the tests
from the same seeds; the sampler noise the reference drew on the device is stored.

  python tests/golden/make_reference_gpu_pins.py [OUT]    # on a GPU, where oracle/ref_harness.py finds the reference
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_gpu_pins.npz")


def capture_noise(fn):
    rec = []
    o1, o2 = torch.randn, torch.randn_like
    torch.randn = lambda *a, **k: (rec.append(o1(*a, **k)) or rec[-1])
    torch.randn_like = lambda a, **k: (rec.append(o2(a, **k)) or rec[-1])
    try:
        out = fn()
    finally:
        torch.randn, torch.randn_like = o1, o2
    return out, [r.float().cpu() for r in rec]


def store_noise(g, key, noise):
    """draws of different shapes: flattened one after the other, with their shapes"""
    g[key] = torch.cat([n.reshape(-1) for n in noise]).numpy()
    g[key + "_shapes"] = np.array([tuple(n.shape) for n in noise])


def head(ref, g):
    from bitdance_b200.head import head_spec
    from bitdance_b200.synth import synth_state_dict
    m = ref.fh.DiffHead(ch_target=32, ch_cond=256, ch_latent=256, depth_latent=4, depth_adanln=2, parallel_num=16,
                        use_swiglu=True).eval()
    m.load_state_dict(synth_state_dict(head_spec(32, 256, 256, 4, 2, True), seed=1, std=0.05))
    m = m.cuda()
    torch.manual_seed(0)
    x, t, c = torch.randn(4, 16, 32), torch.rand(4), torch.randn(4, 16, 256)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        g["head_net"] = m.net(x.cuda(), t.cuda(), c.cuda()).float().cpu().numpy()


def tokenizer(ref, g):
    from bitdance_b200.ae import ae_spec
    from bitdance_b200.synth import synth_state_dict
    dd = dict(double_z=False, z_channels=32, in_channels=3, out_ch=3, ch=32, ch_mult=[1, 2, 2], num_res_blocks=2)
    m = ref.ae.VQModel(dd).eval()
    m.load_state_dict(synth_state_dict(ae_spec(dd), seed=2, std=0.05))
    m = m.cuda()
    torch.manual_seed(0)
    x = torch.rand(2, 3, 32, 48) * 2 - 1
    with torch.autocast("cuda", dtype=torch.bfloat16):
        g["ae_latent"] = m.encoder(x.cuda()).float().cpu().numpy()
        q = m.encode(x.cuda()).float()
        g["ae_quant"] = q.cpu().numpy().astype(np.int8)
        g["ae_decoded"] = m.decode(q).float().cpu().numpy()


def llm(ref, g):
    from transformers import Qwen3Config, Qwen3ForCausalLM
    from bitdance_b200.synth import synth_state_dict
    c = dict(hidden_size=256, intermediate_size=512, num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2,
             head_dim=128, rms_norm_eps=1e-6, rope_theta=1e6)
    hf = Qwen3ForCausalLM(Qwen3Config(vocab_size=64, max_position_embeddings=512, tie_word_embeddings=False, **c)).eval()
    spec = {k: tuple(v.shape) for k, v in hf.state_dict().items()}
    hf.load_state_dict({k: v.to(torch.bfloat16).float() for k, v in synth_state_dict(spec, seed=3, std=0.05).items()})
    hf = hf.to(torch.bfloat16).cuda()
    torch.manual_seed(0)
    B, pn = 2, 16
    x0 = torch.randn(B, 9, 256).to(torch.bfloat16).float()
    x1 = torch.randn(B, pn, 256).to(torch.bfloat16).float()
    x2 = torch.randn(B, pn, 256)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        o = hf.model(inputs_embeds=x0.to(torch.bfloat16).cuda(), use_cache=True)
        pkv = o.past_key_values
        g["llm_h0"] = o.last_hidden_state.float().cpu().numpy()
        for i, (x, f32) in enumerate(((x1, False), (x2, True)), 1):
            mask = torch.ones(B, 1, pn, pn + pkv[0][0].shape[2], dtype=torch.bool, device="cuda")
            o = hf.model(inputs_embeds=x.cuda() if f32 else x.to(torch.bfloat16).cuda(), past_key_values=pkv,
                         use_cache=True, attention_mask=mask)
            pkv = o.past_key_values
            g[f"llm_h{i}"] = o.last_hidden_state.float().cpu().numpy()


def gen_image(ref, g):
    """The reference's whole gen_image on the "tiny" weights of bitdance_b200.synthetic.tiny_state_dicts()."""
    from oracle import ref_runner as rr
    from bitdance_b200.synthetic import tiny_state_dicts
    pipe, _ = rr.build_pipeline("tiny", "cuda")
    sds = tiny_state_dicts()
    missing = pipe.llm_model.load_state_dict(sds["llm"], strict=False)
    assert set(missing.missing_keys) <= {"lm_head.weight"} and not missing.unexpected_keys
    pipe.vision_head.load_state_dict(sds["head"])
    pipe.ae.load_state_dict(sds["ae"])
    pipe.embed_vision_mlp.load_state_dict(sds["proj"])
    torch.manual_seed(11)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        img, noise = capture_noise(lambda: pipe.gen_image("cond", "uncond", guidance_scale=3.0, num_sampling_steps=3,
                                                          max_length=64, num_images=1, image_size=[32, 32]))
    g["gen_image"] = img.float().cpu().numpy()
    store_noise(g, "gen_image_noise", noise)


def imagenet(ref, g):
    import torch._dynamo
    import torch.nn as nn
    from oracle import ref_harness as rh
    from bitdance_b200.imagenet import imagenet_spec
    from bitdance_b200.synth import synth_state_dict
    sys.path.insert(0, rh.REF + "/imagenet_gen")
    torch._dynamo.config.disable = True
    from src import model_parallel as mp

    class _VaeStub(nn.Module):
        def __init__(self, *a, **k):
            super().__init__()

        def decode(self, x):
            return x

    real = mp.VQModel
    mp.VQModel = _VaeStub
    try:
        m = mp.BitDance(dim=128, n_layer=2, n_head=2, diff_layers=2, diff_dim=128, diff_adanln_layers=1, latent_dim=32,
                        down_size=16, patch_size=1, resolution=64, diff_batch_mul=1, cls_token_num=4, num_classes=10,
                        parallel_num=4, parallel_mode="patch").eval()
    finally:
        mp.VQModel = real
    cfg = dict(dim=128, n_layer=2, n_head=2, diff_layers=2, diff_dim=128, diff_adanln_layers=1, latent_dim=32, down_size=16,
               patch_size=1, resolution=64, cls_token_num=4, num_classes=10, parallel_num=4, parallel_mode="patch")
    missing = m.load_state_dict(synth_state_dict(imagenet_spec(cfg), seed=4, std=0.08), strict=False)
    assert not missing.unexpected_keys and all(k.startswith("vae.") for k in missing.missing_keys)
    m = m.cuda()
    torch.manual_seed(11)
    with torch.amp.autocast("cuda", dtype=torch.bfloat16):
        grid, noise = capture_noise(lambda: m.sample(torch.tensor([3, 7, 1]).cuda(), 4, cfg_scale=3.0,
                                                     cfg_schedule="linear"))
    g["imagenet_grid"] = grid.float().cpu().numpy().astype(np.int8)
    store_noise(g, "imagenet_noise", noise)


def main(out):
    from oracle import ref_harness as rh
    ref = rh.import_reference()
    g = {}
    with torch.no_grad():
        for fn in (head, tokenizer, llm, gen_image, imagenet):
            fn(ref, g)
    np.savez_compressed(out, **g)
    print(out, os.path.getsize(out), {k: v.shape for k, v in g.items()})


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else OUT)
