"""CPU-side checks of the ImageNet class-conditional path (SURVEY.md section 8 rows a16 / f1): host tables and the API mirror.
The arithmetic on the GPU is covered by tests/test_imagenet_gpu.py; the oracle itself is pinned against the reference in
tests/test_oracle_vs_reference.py::test_imagenet_sample_vs_reference."""
import pytest
import torch

CFGS = [dict(dim=128, n_layer=2, n_head=2, diff_layers=2, diff_dim=128, diff_adanln_layers=1, latent_dim=32, down_size=16,
             patch_size=1, resolution=64, cls_token_num=4, num_classes=10, parallel_num=4, parallel_mode="patch"),
        dict(dim=768, n_layer=1, n_head=12, diff_layers=1, diff_dim=768, diff_adanln_layers=1, latent_dim=32, down_size=16,
             patch_size=1, resolution=256, cls_token_num=64, num_classes=1000, parallel_num=16, parallel_mode="patch"),
        dict(dim=128, n_layer=1, n_head=2, diff_layers=1, diff_dim=128, diff_adanln_layers=1, latent_dim=16, down_size=16,
             patch_size=1, resolution=128, cls_token_num=1, num_classes=5, parallel_num=4, parallel_mode="standard")]


@pytest.mark.parametrize("cfg", CFGS)
def test_rope_tables_equal_the_oracle_buffers(cfg):
    """rope_tables_2d (what the pair-RoPE kernel indexes by absolute position) == the reference's registered freqs_cis
    buffer as restated by the oracle (precompute_freqs_cis_2d + patch-raster reorder + dropped last block)."""
    from bitdance_b200.imagenet import ffn_hidden, rope_tables_2d
    from oracle import imagenet as oi
    cos, sin, h, w = rope_tables_2d(cfg)
    fc, mask, h2, w2 = oi.make_buffers(cfg)
    assert (h, w) == (h2, w2) and cos.shape == fc.shape[:2]
    assert torch.equal(cos, fc[..., 0]) and torch.equal(sin, fc[..., 1])
    assert cos.shape[0] == h * w + cfg["cls_token_num"] - 1
    assert ffn_hidden(768) == 2048 and ffn_hidden(1024) == 2816 and ffn_hidden(1280) == 3584


def test_two_pass_first_step_equals_the_block_causal_mask():
    """The engine runs AR position 0 as (cls - 1 leading tokens, causal) + (first block, bidirectional over itself and the
    past); that is exactly the reference's additive block-causal mask restricted to the first cls + pn - 1 tokens."""
    from oracle import imagenet as oi
    for cls, pn in [(4, 4), (64, 16), (1, 4), (9, 16)]:
        n0 = cls + pn - 1
        m = oi.block_causal_mask(cls - 1 + 4 * pn, cls - 1, pn)[:n0, :n0]
        visible = m == 0
        want = torch.zeros(n0, n0, dtype=torch.bool)
        for i in range(cls - 1):
            want[i, :i + 1] = True                 # causal prefix
        want[cls - 1:, :] = True                   # the block sees the whole prefix and itself
        assert torch.equal(visible, want), (cls, pn)


def test_api_mirror_state_dict_equals_the_reference():
    """imagenet_spec / the BitDance mirror hold exactly the reference module's parameters (names and shapes) for the
    small test model (the reference's, as stored in tests/golden/reference_pins.npz by tests/golden/make_reference_pins.py)."""
    import json
    import os
    import numpy as np
    from bitdance_b200.imagenet_gen.src.model_parallel import BitDance
    kw = dict(dim=128, n_layer=2, n_head=2, diff_layers=2, diff_dim=128, diff_adanln_layers=1, latent_dim=32, down_size=16,
              patch_size=1, resolution=64, diff_batch_mul=1, cls_token_num=4, num_classes=10, parallel_num=4,
              parallel_mode="patch")
    golden = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_pins.npz"))
    a = {k: tuple(v) for k, v in json.loads(str(golden["imagenet_small_spec"])).items()}
    b = {k: tuple(v.shape) for k, v in BitDance(**kw).state_dict().items()}
    assert a == b
