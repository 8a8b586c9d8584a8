"""The ImageNet class-conditional generator on the GPU (bitdance_b200/imagenet.py; SURVEY.md section 8 rows a16 / f1)
against the CPU oracle (oracle/imagenet.py, autocast-bf16 policy) and against what the UNMODIFIED ``BitDance.sample``
returned on a B200 under CUDA autocast (tests/golden/reference_gpu_pins.npz)."""
import pytest
import torch

pytestmark = pytest.mark.gpu

CFG = dict(dim=128, n_layer=2, n_head=2, diff_layers=2, diff_dim=128, diff_adanln_layers=1, latent_dim=32, down_size=16,
           patch_size=1, resolution=64, cls_token_num=4, num_classes=10, parallel_num=4, parallel_mode="patch", time_shift=1.0)


def make(cfg, seed=4, head_engines=None):
    from bitdance_b200.imagenet import ImageNetEngine, imagenet_spec
    from bitdance_b200.synth import synth_state_dict
    sd = synth_state_dict(imagenet_spec(cfg), seed=seed, std=0.08)
    return sd, ImageNetEngine(sd, cfg, ae=None, head_engines=head_engines)


def draw_noise(cfg, n_cls, S, cfg_scale, seed=1):
    """per AR position [S+1, rows, pn, lat]: rows = all sequences while the linear ramp is at 1 (position 0), else n_cls"""
    g = torch.Generator().manual_seed(seed)
    hw = (cfg["resolution"] // cfg["down_size"]) ** 2
    steps = hw // cfg["parallel_num"]
    out = []
    for i in range(steps):
        guided = cfg_scale > 1.0 and (1.0 + (cfg_scale - 1.0) * i / steps) > 1.0
        rows = n_cls if (guided or cfg_scale <= 1.0) else 2 * n_cls
        out.append(torch.randn(S + 1, rows, cfg["parallel_num"], cfg["latent_dim"], generator=g))
    return out


# head_engines: None = the default (16 persistent head engines side by side, 9 SMs and one 128-row tile each), 0 = the
# multi-kernel path; 11 sequences x 16 tokens x 2 CFG groups = 3 tiles in flight at once, the last one ragged
@pytest.mark.parametrize("cfg_scale,cls_num,pn,head_engines,n_img",
                         [(3.0, 4, 4, None, 3), (1.0, 1, 16, None, 3), (2.5, 9, 16, None, 3), (2.5, 9, 16, 0, 3),
                          (3.0, 4, 16, None, 11)])
def test_imagenet_sample_vs_oracle(cfg_scale, cls_num, pn, head_engines, n_img):
    from oracle import imagenet as oi
    cfg = dict(CFG, cls_token_num=cls_num, parallel_num=pn)
    sd, eng = make(cfg, head_engines=head_engines)
    assert (len(eng._side) > 1) == (head_engines is None)
    S = 4
    class_ids = torch.tensor([3, 7, 1, 0, 9, 2, 5, 4, 8, 6, 3][:n_img])
    noise = draw_noise(cfg, len(class_ids), S, cfg_scale)
    tokens, packed = eng.sample_tokens(class_ids, S, cfg_scale, noise=[n.cuda() for n in noise])
    torch.cuda.synchronize()
    tr = []
    with torch.no_grad():
        tok_ref, grid_ref = oi.sample(sd, cfg, class_ids, S, cfg_scale, [list(n) for n in noise], rnd=oi.oh.bf16, trace=tr)
    t = tokens.cpu()
    a0 = (t[:, :pn] == tok_ref[:, :pn]).float().mean().item()
    a_all = (t == tok_ref).float().mean().item()
    print(f"ImageNet sample cfg={cfg_scale} cls={cls_num} pn={pn} engines={len(eng._side)} images={n_img}: "
          f"first-block token agreement {a0:.4f}, all blocks {a_all:.4f}")
    # free-running agreement decays with the AR position for a random-init (chaotic) model; the decoder is checked
    # teacher-forced at every position below, and the same figure against the REAL reference is the last test of this file
    assert a0 > 0.95 and a_all > 0.65
    grid = eng.tokens_to_grid(tokens).cpu()
    assert grid.shape == grid_ref.shape
    # the grid layout is the oracle's for the engine's own tokens
    assert torch.equal(grid, oi.unpatchify_raster(t, int(pn ** 0.5), (eng.h, eng.w)))
    bits = ((packed.cpu()[..., 0].long().unsqueeze(-1) >> torch.arange(32)) & 1).bool()
    assert torch.equal(bits, t > 0)


def test_imagenet_decoder_hidden_vs_oracle():
    """The class-conditional decoder alone (2-D pair RoPE, static KV, block-causal first step, SwiGLU connector) teacher-forced
    with the ORACLE's own sampled tokens: the hidden states that condition the head agree to bf16 level at EVERY AR
    position (3 layers, 9 cls tokens, so the causal prefix, the first block and 3 cached blocks are all exercised)."""
    from oracle import imagenet as oi
    cfg = dict(CFG, cls_token_num=9, parallel_num=4, n_layer=3)
    sd, eng = make(cfg, seed=6)
    S, cfg_scale = 2, 3.0
    class_ids = torch.tensor([2, 5])
    noise = draw_noise(cfg, 2, S, cfg_scale)
    tr = []
    with torch.no_grad():
        oi.sample(sd, cfg, class_ids, S, cfg_scale, [list(n) for n in noise], rnd=oi.oh.bf16, trace=tr)
    pn, cls, dim, lat = cfg["parallel_num"], cfg["cls_token_num"], cfg["dim"], cfg["latent_dim"]
    dev = eng.device
    cond = torch.cat([class_ids, torch.full_like(class_ids, cfg["num_classes"])]).to(dev)
    R = 4
    cache = eng._cache(R)
    c = eng.cls_embedding[cond].view(R, cls, dim)
    eng._forward(c[:, :cls - 1].contiguous(), cache, causal=True)
    x0 = torch.cat([c[:, cls - 1:], eng.query_token.expand(R, -1, -1)], dim=1).contiguous()
    z = eng._forward(x0, cache, causal=False, out_add=eng.pos_for_diff[:pn].contiguous())
    rel = lambda a, b: ((a - b).abs().max() / (b.abs().max() + 1e-6)).item()
    errs = [rel(z.cpu(), tr[0]["z"])]
    for i in range(1, eng.h * eng.w // pn):
        last = tr[i - 1]["last"].to(dev, torch.bfloat16).contiguous()          # [R, pn, lat], all rows as the oracle fed them
        x = eng._proj_in(last.view(R * pn, lat)).view(R, pn, dim)
        z = eng._forward(x, cache, causal=False, out_add=eng.pos_for_diff[i * pn:(i + 1) * pn].contiguous())
        errs.append(rel(z.cpu(), tr[i]["z"]))
    print("ImageNet decoder, teacher-forced, rel err per AR position:", [round(e, 4) for e in errs])
    assert max(errs) < 3e-2
    assert cache.seq_lens.tolist() == [cls - 1 + eng.h * eng.w] * R


def test_imagenet_api_mirror_and_reference_on_gpu():
    """The drop-in module (``src.model_parallel``: get_model_args / create_model / load_state_dict(strict) / sample) and,
    when the shipped reference is present, the UNMODIFIED reference model on this GPU under CUDA autocast with the same
    weights and noise: first-block token agreement."""
    import os
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, os.path.join(root, "imagenet_gen"))
    for k in [k for k in sys.modules if k == "src" or k.startswith("src.")]:
        del sys.modules[k]
    from src.model_parallel import create_model, get_model_args
    from bitdance_b200.imagenet import MODELS
    args = get_model_args().parse_args(["--model", "BitDance-B", "--image-size", "256", "--latent-dim", "32",
                                        "--parallel-num", "16", "--cls-token-num", "64"])
    assert MODELS["BitDance-B"]["dim"] == 768
    # a small instance through the same class (BitDance-B itself + the 460 M-parameter VAE is exercised by bench runs)
    from bitdance_b200.imagenet_gen.src.model_parallel import BitDance
    from bitdance_b200.synth import synth_state_dict
    small = dict(dim=128, n_layer=2, n_head=2, diff_layers=2, diff_dim=128, diff_adanln_layers=1, latent_dim=32, down_size=16,
                 patch_size=1, resolution=64, diff_batch_mul=1, cls_token_num=4, num_classes=10, parallel_num=4,
                 parallel_mode="patch")
    model = BitDance(**small)
    spec = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    sd = synth_state_dict(spec, seed=9, std=0.05)
    model.load_state_dict(sd, strict=True)
    model = model.to("cuda")
    torch.manual_seed(3)
    img = model.sample(torch.tensor([1, 2]).cuda(), sample_steps=3, cfg_scale=2.0)
    assert img.shape == (2, 3, 64, 64) and torch.isfinite(img.float()).all()
    torch.manual_seed(3)
    img2 = model.sample(torch.tensor([1, 2]).cuda(), sample_steps=3, cfg_scale=2.0)
    assert torch.equal(img, img2)
    with pytest.raises(NotImplementedError):
        model(img, torch.tensor([1, 2]).cuda())
    assert create_model is not None and args.parallel_num == 16


def test_imagenet_vs_unmodified_reference_on_gpu():
    """Against the UNMODIFIED ``BitDance.sample`` run on a B200 under CUDA autocast with the same weights (the seeded
    synth_state_dict below): its token grid and the noise it drew are stored in tests/golden/reference_gpu_pins.npz
    (tests/golden/make_reference_gpu_pins.py), and the noise is replayed in the engine."""
    import os
    import numpy as np
    from bitdance_b200.imagenet import ImageNetEngine, imagenet_spec
    from bitdance_b200.synth import synth_state_dict
    golden = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_gpu_pins.npz"))
    cfg = dict(CFG)
    sd = synth_state_dict(imagenet_spec(cfg), seed=4, std=0.08)
    eng = ImageNetEngine(sd, cfg, ae=None)
    S, cfg_scale = 4, 3.0
    class_ids = torch.tensor([3, 7, 1]).cuda()
    flat, rec, o = torch.from_numpy(golden["imagenet_noise"]), [], 0
    for shape in golden["imagenet_noise_shapes"]:
        n = int(np.prod(shape))
        rec.append(flat[o:o + n].view(*(int(d) for d in shape)).cuda())
        o += n
    steps = eng.h * eng.w // eng.pn
    assert len(rec) == steps * (S + 1)
    noise = [torch.stack(rec[i * (S + 1):(i + 1) * (S + 1)]).float().contiguous() for i in range(steps)]
    tokens, _ = eng.sample_tokens(class_ids, S, cfg_scale, noise=noise)
    grid = eng.tokens_to_grid(tokens)
    ref_tok = torch.from_numpy(golden["imagenet_grid"]).float().to(grid.device)
    a_all = (grid == ref_tok).float().mean().item()
    # first block = the first p x p patch of the grid
    p = eng.ps
    a0 = (grid[:, :, :p, :p] == ref_tok[:, :, :p, :p]).float().mean().item()
    print(f"ImageNet vs the unmodified reference on a B200 (CUDA autocast): first-block token agreement {a0:.4f}, "
          f"whole grid {a_all:.4f}")
    assert a0 > 0.95 and a_all > 0.65
