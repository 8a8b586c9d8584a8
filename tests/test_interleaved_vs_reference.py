"""Interleaved text+image inference against the UNMODIFIED reference ``MLLModel.forward_inference_block_causal``
(modeling/mllm.py:696-897), on CPU in fp32 with the tiny model of ``bitdance_b200.synthetic.tiny_state_dicts()``.

What can be pinned and is, against the reference's outputs stored in tests/golden/reference_pins.npz
(tests/golden/make_reference_pins.py; the sampler noise is drawn again here from the same seeds):
  * plan [user text, model image] == ``oracle/pipeline.py::gen_image(cond, remove_first_user_block(cond))`` — the
    equivalence the mirror's image item rests on (it hands the accumulated context to the same block generator);
  * plan [user text, user image, model image] (editing) == ``oracle/pipeline.py::gen_image`` fed with the context the MIRROR's
    bookkeeping builds (start tokens + the reference's encode_image of the source + <|vision_end|> in BOTH streams,
    unconditional text = remove_first_user_block): pins that bookkeeping against the reference's.
What cannot: the reference's TEXT branch raises — without a cache at mllm.py:798 (``past_key_values[0][0]`` of None), after a
generated image on the second token (a 2-D ``(1, hidden)`` tensor fed back as ``inputs_embeds``, :857 -> rotary shape
error). Both are asserted by the last test, which runs the reference itself and needs its whole source tree (its
``mllm.py`` imports the reference's ``data`` package), as the evidence for DESIGN.md section 2c's "text loop parity-unpinned"."""
import os

import numpy as np
import pytest
import torch
from torch import nn

TEXT = "<|im_start|>user\na photo of the red cat<|im_end|>\n<|im_start|>assistant\n"
U, M_ = {"from": "user"}, {"from": "model"}
S, GUIDANCE, PN = 3, 3.0, 16


class _Cfg(dict):
    __getattr__ = dict.__getitem__


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_pins.npz"))


@pytest.fixture(scope="module")
def tiny():
    """the weights and tokenizer of the stored reference runs"""
    from bitdance_b200.synthetic import MODELS, synthetic_tokenizer, tiny_state_dicts
    sds = tiny_state_dicts()
    tok, _ = synthetic_tokenizer(512, PN)
    cfg = {k: v for k, v in MODELS["tiny"]["llm"].items() if k != "vocab_size"}
    return sds, tok, cfg


def _noise(shapes):
    """the reference's draws in the stored run, in order, from the same global-RNG state; grouped per AR step"""
    rec = [torch.randn(tuple(int(d) for d in s)) for s in shapes]
    steps = 64 // PN
    assert len(rec) == steps * (S + 1)
    return [rec[i * (S + 1):(i + 1) * (S + 1)] for i in range(steps)]


def _oracle_image(tiny, cond, uncond, noise):
    from oracle import pipeline as op
    sds, tok, cfg = tiny
    ids = lambda ts: [tok.convert_tokens_to_ids(t) for t in ts]
    start = ids(["<|vision_start|>", "<|res_8|>", "<|res_8|>"] + [f"<|query_{i}|>" for i in range(1, PN)])
    with torch.no_grad():
        _, img = op.gen_image(sd_llm=sds["llm"], cfg_llm=cfg, embed=sds["llm"]["model.embed_tokens.weight"],
                              sd_head=sds["head"], sd_proj=sds["proj"], sd_ae=sds["ae"], cond_ids=None, uncond_ids=None,
                              cond_emb=cond, uncond_emb=uncond, start_ids=start, h=8, w=8, pn=PN, num_images=1,
                              guidance=GUIDANCE, S=S, noise=noise, head_dim=128)
    return img


def test_reference_t2i_plan_is_gen_image(golden, tiny):
    from bitdance_b200.modeling.utils import remove_first_user_block
    sds, tok, _ = tiny
    embed = sds["llm"]["model.embed_tokens.weight"]
    E = lambda s: embed[torch.tensor(tok.encode(s))]
    torch.manual_seed(5)
    noise = _noise(golden["interleaved_t2i_noise_shapes"])
    img = _oracle_image(tiny, E(TEXT), E(remove_first_user_block(TEXT)), noise)
    img_ref = torch.from_numpy(golden["interleaved_t2i_image"])
    assert img.shape == img_ref.shape == (1, 3, 32, 32)
    err = (img - img_ref).abs().max().item()
    assert err < 1e-3 * max(1.0, img_ref.abs().max().item()), err


def test_reference_editing_plan_vs_oracle_with_mirror_bookkeeping(golden, tiny):
    from bitdance_b200.modeling.utils import remove_first_user_block
    sds, tok, _ = tiny
    torch.manual_seed(7)
    noise = _noise(golden["interleaved_edit_noise_shapes"])
    # the context as bitdance_b200/modeling/mllm.py builds it, around the reference's encode_image of the source image
    embed = sds["llm"]["model.embed_tokens.weight"]
    E = lambda ids: embed[torch.tensor(list(ids))]
    start3 = [tok.convert_tokens_to_ids(t) for t in ("<|vision_start|>", "<|res_8|>", "<|res_8|>")]
    pre = torch.from_numpy(golden["interleaved_edit_source_latent"])
    assert pre.shape == (64, 256)
    end = E([tok.convert_tokens_to_ids("<|vision_end|>")])
    cond = torch.cat([E(tok.encode(TEXT)), E(start3), pre, end])
    uncond = torch.cat([E(tok.encode(remove_first_user_block(TEXT))), E(start3), pre, end])
    img = _oracle_image(tiny, cond, uncond, noise)
    img_ref = torch.from_numpy(golden["interleaved_edit_image"])
    assert img.shape == img_ref.shape == (1, 3, 32, 32)
    err = (img - img_ref).abs().max().item()
    assert err < 1e-3 * max(1.0, img_ref.abs().max().item()), err


@pytest.fixture(scope="module")
def world():
    from oracle import ref_harness as rh
    if not os.path.isdir(os.path.join(rh.REF, "data")):
        pytest.skip("runs the reference itself: needs its whole source tree (modeling/mllm.py imports data.data_utils)")
    from bitdance_b200.synthetic import synthetic_tokenizer
    from oracle import ref_runner as rr
    rh.import_reference()
    mllm = rh.import_reference_mllm()
    torch.manual_seed(0)
    pipe, info = rr.build_pipeline("tiny", "cpu")
    pipe.llm_model.float()                                   # exact-math pin: everything fp32
    tok, _ = synthetic_tokenizer(512, 16)
    for alias, t in (("im_start", "<|im_start|>"), ("im_end", "<|im_end|>"), ("start_of_image", "<|vision_start|>"),
                     ("end_of_image", "<|vision_end|>")):
        setattr(tok, alias + "_id", tok.convert_tokens_to_ids(t))      # data/data_utils.py:95-109
    for i in range(1, 161):
        setattr(tok, f"res_{i}_id", tok.convert_tokens_to_ids(f"<|res_{i}|>"))
    for i in range(1, 16):
        setattr(tok, f"query_{i}_id", tok.convert_tokens_to_ids(f"<|query_{i}|>"))
    pipe.tokenizer = tok
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
    return m, pipe, tok


@pytest.mark.reference
def test_reference_text_branch_raises(world):
    m, pipe, tok = world
    with torch.no_grad():
        # no cache yet: mllm.py:798 subscripts past_key_values = None before the first pass
        with pytest.raises(TypeError):
            m.forward_inference_block_causal([dict(type="text", **U), dict(type="text", **M_)], [TEXT], [], max_length_text=4)
        # after a generated image (a cache exists): the first token is sampled, then its (1, hidden) embedding is fed back
        # as inputs_embeds (mllm.py:857) and the decoder fails on the rotary shapes
        with pytest.raises(RuntimeError):
            m.forward_inference_block_causal([dict(type="text", **U), dict(type="image", **M_), dict(type="text", **U),
                                              dict(type="text", **M_)], [TEXT, "the blue dog"], [], max_length_text=4,
                                             max_length_vision=64, sample_steps=2, image_size=[32, 32], cfg_scale=3.0)
