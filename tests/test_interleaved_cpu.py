"""Interleaved text+image inference (SURVEY.md section 8f-4), CPU side:

  * the mirrored sampler (``top_k_top_p_filtering`` / ``sample_codebook`` / ``remove_first_user_block``) bit-exactly against the
    UNMODIFIED reference functions (modeling/utils.py:64-124, 206-216) on random logits incl. ties and degenerate settings;
  * the host bookkeeping of ``MLLModel.forward_inference_block_causal`` (mllm.py:696-897) over a STUB engine (no CUDA, no
    kernels): which embeddings reach the image generator for which plan, the persistent conditional cache, the
    context reset on ``<|im_end|>``, the literal re-feed after a cut-off text, the unsupported plans.
"""
import types

import pytest
import torch


def test_sampler_mirrors_vs_reference():
    """Against the reference functions' outputs stored in tests/golden/reference_pins.npz (tests/golden/make_reference_pins.py):
    the logits top_k_top_p_filtering keeps (it sets every other one to -inf) and the tokens sample_codebook draws."""
    import json
    import os
    import numpy as np
    import bitdance_b200.modeling.utils as mu
    golden = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_pins.npz"))
    keep_all = np.unpackbits(golden["sampler_keep"]).astype(bool)
    off = 0
    g = torch.Generator().manual_seed(0)
    for trial in range(120):
        B, V = 3, int(torch.randint(5, 400, (1,), generator=g))
        logits = torch.randn(B, V, generator=g) * float(torch.rand(1, generator=g) * 5 + 0.1)
        if trial % 3 == 0:
            logits = (logits * 2).round() / 2           # ties at the k-th value / at the nucleus edge
        k = int(torch.randint(0, V + 50, (1,), generator=g))
        p = 1.0 if trial % 5 == 0 else float(torch.rand(1, generator=g))
        mk = int(torch.randint(1, 4, (1,), generator=g))
        a = mu.top_k_top_p_filtering(logits.clone(), k, p, min_tokens_to_keep=mk)
        keep = torch.from_numpy(keep_all[off:off + B * V].reshape(B, V))
        off += B * V
        assert torch.equal(a, logits.masked_fill(~keep, -float("inf"))), (trial, k, p, mk)
        emb = torch.nn.Embedding(V, 8)
        torch.manual_seed(trial)
        ta, ea = mu.sample_codebook(logits.clone(), "text", emb, True, 0.7, k, p)
        tb = torch.from_numpy(golden["sampler_tokens_sampled"][trial]).long().view_as(ta)
        assert torch.equal(ta, tb) and torch.equal(ea, emb(tb))
        ta, _ = mu.sample_codebook(logits.clone(), "text", emb, False, 1.0, k, p)
        assert torch.equal(ta, torch.from_numpy(golden["sampler_tokens_argmax"][trial]).long().view_as(ta))
    for s, want in json.loads(str(golden["remove_first_user_block"])).items():
        assert mu.remove_first_user_block(s) == want


def test_filtering_properties():
    """No reference needed: top-k keeps >= k entries (ties), the nucleus keeps the crossing token, the argmax always
    survives, the input is not modified."""
    from bitdance_b200.modeling.utils import top_k_top_p_filtering
    torch.manual_seed(1)
    x = torch.randn(4, 50)
    keep = x.clone()
    y = top_k_top_p_filtering(x, top_k=7, top_p=1.0)
    assert torch.equal(x, keep)
    assert ((y > -float("inf")).sum(-1) == 7).all()
    y = top_k_top_p_filtering(x, top_k=0, top_p=0.5)
    pr = torch.softmax(x, -1)
    for b in range(4):
        kept = y[b] > -float("inf")
        assert kept[x[b].argmax()]
        mass = pr[b][kept].sum().item()
        smallest = pr[b][kept].min().item()
        assert mass > 0.5 >= mass - smallest - 1e-6    # minimal prefix whose mass exceeds top_p
    y = top_k_top_p_filtering(torch.zeros(1, 9), top_k=3, top_p=1.0)
    assert (y == 0).all()                                # all tied with the k-th value: nothing removed


# ----------------------------------------------------------------------------------------------------------------------
# host bookkeeping over a stub engine
# ----------------------------------------------------------------------------------------------------------------------
D, V, PN, VPS = 8, 40, 4, 4
IM_START, IM_END, VSTART, VEND = 30, 31, 32, 33


class StubTok:
    im_start_id, im_end_id, start_of_image_id, end_of_image_id = IM_START, IM_END, VSTART, VEND

    def __getattr__(self, name):           # res_{n}_id, query_{i}_id
        if name.startswith("res_") and name.endswith("_id"):
            return 34
        if name.startswith("query_") and name.endswith("_id"):
            return 35 + int(name[6:-3]) % 4
        raise AttributeError(name)

    def encode(self, s):
        return [ord(c) % 29 for c in s]

    def convert_ids_to_tokens(self, ids, skip_special_tokens=False):
        return [None if (skip_special_tokens and i >= 30) else f"t{i}" for i in ids]

    def convert_tokens_to_string(self, toks):
        return " ".join(toks)


class StubLlm:
    """records every forward; 'hidden' = running mean of everything in the cache (so the output depends on the cache)"""

    def __init__(self):
        self.rope_cos = torch.zeros(4096, 1)
        self.calls = []

    def new_cache(self, R, max_tokens):
        return types.SimpleNamespace(rows=[], max_tokens=max_tokens, R=R)

    def forward(self, x, cache, r0, R, *, causal, **kw):
        assert causal and x.dim() == 3 and x.shape[0] == 1 and x.dtype == torch.bfloat16
        self.calls.append(x.shape[1])
        out = []
        for i in range(x.shape[1]):
            cache.rows.append(x[0, i].float())
            assert len(cache.rows) <= cache.max_tokens
            out.append(torch.stack(cache.rows).mean(0))
        return torch.stack(out)[None].to(torch.bfloat16)


def make_stub(script):
    """script: the token ids the (stub) lm_head makes the argmax, in order."""
    from bitdance_b200.modeling.mllm import MLLModel
    torch.manual_seed(0)
    emb = torch.nn.Embedding(V, D)
    emb.weight.data = emb.weight.data.to(torch.bfloat16)
    it = iter(script)

    def lm_head(h):
        lg = torch.zeros(1, V)
        lg[0, next(it)] = 50.0
        return lg

    llm = StubLlm()
    gen_calls = []

    def gen_tokens(cond, uncond, start, **kw):
        gen_calls.append((cond.clone(), None if uncond is None else uncond.clone(), start.clone(), kw))
        hw = kw["h"] * kw["w"]
        return torch.ones(1, hw, 32), torch.zeros(1, hw, 1, dtype=torch.int32)

    eng = types.SimpleNamespace(pn=PN, ps=2, D=D, pos_1d=torch.zeros(64, D // 2), llm=llm, gen_tokens=gen_tokens,
                                ae=types.SimpleNamespace(decode_tokens=lambda t, h, w, ps: torch.zeros(1, 3, h * VPS, w * VPS)))
    m = MLLModel.from_components(tokenizer=StubTok(), llm_model=types.SimpleNamespace(model=types.SimpleNamespace(embed_tokens=emb),
                                                                                    lm_head=lm_head),
                                 engine=eng, vision_encoder=None, vision_diffusion_head=None, embed_vision_mlp=None,
                                 vit_patch_size=VPS, device="cpu")
    m.encode_image = lambda imgs: (torch.full(((imgs[0].shape[-2] // VPS) * (imgs[0].shape[-1] // VPS), D), 0.5), None)
    return m, emb, llm, gen_calls


def E(emb, ids):
    return emb(torch.tensor(ids))


def test_plan_t2i_and_editing_contexts():
    m, emb, llm, gen = make_stub([])
    text = "<|im_start|>user\nab<|im_end|>\n<|im_start|>assistant\n"
    un = "<|im_start|>assistant\n"
    plan = [dict(type="text", **{"from": "user"}), dict(type="image", **{"from": "model"})]
    out = m.forward_inference_block_causal(plan, [text], [], max_length_vision=16, image_size=[16, 16], cfg_scale=3.0,
                                           sample_steps=2)
    assert out["generated_text"] == [] and out["generated_image"][0].shape == (1, 3, 16, 16)
    cond, uncond, start, kw = gen[0]
    tok = m.tokenizer
    assert torch.equal(cond, E(emb, tok.encode(text))) and torch.equal(uncond, E(emb, tok.encode(un)))
    assert torch.equal(start, E(emb, [VSTART, 34, 34] + [35 + i % 4 for i in range(1, PN)]))   # [pn + 2, D]
    assert kw["h"] == kw["w"] == 4 and kw["num_images"] == 1 and kw["guidance_scale"] == 3.0 and kw["num_sampling_steps"] == 2
    # editing: text, user image (start + content + end in BOTH streams), image from the model; no CFG -> uncond None
    m, emb, llm, gen = make_stub([])
    plan = [dict(type="text", **{"from": "user"}), dict(type="image", **{"from": "user"}), dict(type="image", **{"from": "model"})]
    img = torch.zeros(1, 3, 8, 12)
    texts, imgs = [text], [img]
    m.forward_inference_block_causal(plan, texts, imgs, max_length_vision=16, image_size=[16, 16], cfg_scale=1.0)
    assert texts == [] and imgs == []                   # consumed front to back, like the reference
    cond, uncond, start, _ = gen[0]
    want = torch.cat([E(emb, tok.encode(text)).float(), E(emb, [VSTART, 34, 34]).float(), torch.full((6, D), 0.5),
                      E(emb, [VEND]).float()]).to(torch.bfloat16)
    assert uncond is None and torch.equal(cond, want)
    with pytest.raises(ValueError):
        m.forward_inference_block_causal([plan[0], plan[2]], [text], [], max_length_vision=64, image_size=[16, 16])
    with pytest.raises(NotImplementedError):            # anything generated after an image
        m.forward_inference_block_causal([plan[0], plan[2], dict(type="text", **{"from": "model"})], [text], [],
                                         max_length_vision=16, image_size=[16, 16])


def test_plan_text_decoding_cache_and_reset():
    # turn 1 ends with <|im_end|> after 3 tokens -> context cleared, cache kept; turn 2 is cut off by max_length_text
    # -> context NOT cleared; turn 3 therefore re-feeds turn 2's context + its own (the reference's literal behaviour)
    m, emb, llm, gen = make_stub([5, 6, IM_END, 7, 8, 9, 1, 2, 3])
    plan = [dict(type="text", **{"from": "user"}), dict(type="text", **{"from": "model"}),
            dict(type="text", **{"from": "user"}), dict(type="text", **{"from": "model"}),
            dict(type="text", **{"from": "user"}), dict(type="text", **{"from": "model"})]
    out = m.forward_inference_block_causal(plan, ["abcd", "xy", "z"], [], max_length_text=3, do_sample=False)
    assert out["generated_text"] == ["t5 t6", "t7 t8 t9", "t1 t2 t3"]     # <|im_end|> skipped as a special token
    assert m.last_text_ids.tolist() == [1, 2, 3]
    # forwards: ctx(4) + 2 single-token steps (the end token is never fed) | ctx(2) + 2 steps | ctx(2 + 1) + 2 steps
    assert llm.calls == [4, 1, 1, 2, 1, 1, 3, 1, 1]
    with pytest.raises(NotImplementedError):            # image generation on top of a non-empty conditional cache
        m2, *_ = make_stub([5, IM_END])
        m2.forward_inference_block_causal([plan[0], plan[1], dict(type="image", **{"from": "model"})], ["ab"], [],
                                          max_length_text=4, max_length_vision=16, image_size=[16, 16], do_sample=False)
    with pytest.raises(ValueError):
        m.forward_inference_block_causal([dict(type="audio", **{"from": "user"})], [], [])


def test_forward_dispatch():
    m, *_ = make_stub([IM_END])
    out = m.forward([dict(type="text", **{"from": "user"}), dict(type="text", **{"from": "model"})], ["hi"], [],
                    do_sample=False)
    assert out == {"generated_text": [""], "generated_image": []}
    m.training = True
    with pytest.raises(NotImplementedError):
        m.forward()


def test_cache_capacity_bound_holds_for_random_chat_plans():
    """the persistent conditional cache is allocated once, up front (``_interleaved_capacity``): the stub decoder asserts on
    every appended token that it still fits, over random multi-turn plans incl. cut-off turns (context re-fed literally)"""
    import random
    rnd = random.Random(0)
    for trial in range(40):
        n_turns = rnd.randint(1, 5)
        max_len = rnd.randint(1, 6)
        plan, texts, script = [], [], []
        for _ in range(n_turns):
            for _ in range(rnd.randint(1, 2)):                  # one or two user items before every model turn
                if rnd.random() < 0.3:
                    plan.append(dict(type="image", **{"from": "user"}))
                else:
                    plan.append(dict(type="text", **{"from": "user"}))
                    texts.append("x" * rnd.randint(1, 9))
            plan.append(dict(type="text", **{"from": "model"}))
            ends_at = rnd.randint(1, max_len + 2)               # beyond max_len: the turn is cut off
            script += [IM_END if i + 1 == ends_at else 1 + i for i in range(min(max_len, ends_at))]
        imgs = [torch.zeros(1, 3, 4 * rnd.randint(1, 3), 4 * rnd.randint(1, 3)) for _ in plan if _["type"] == "image"]
        m, emb, llm, gen = make_stub(script)
        out = m.forward_inference_block_causal(plan, texts, imgs, max_length_text=max_len, image_size=[8, 8], cfg_scale=1.0,
                                               do_sample=False)
        assert len(out["generated_text"]) == n_turns and texts == [] and imgs == []
