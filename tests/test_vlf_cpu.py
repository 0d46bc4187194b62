"""CPU: the streaming evaluation of BiMultiHeadAttention (two attention calls, no S x N_t score tensor; used above
`stream_threshold_bytes`, i.e. for phrase prompts at scale) against the literal op sequence of the reference
(ape/layers/fuse_helper.py:67-166) as restated in the same module, and against the reference module itself."""
import pytest
import torch

from ape_b200.layers.vision_language_fusion import BiAttentionBlock


@pytest.mark.parametrize("S,N", [(300, 7), (1000, 64), (64, 200)])
def test_streaming_equals_literal(S, N):
    torch.manual_seed(0)
    blk = BiAttentionBlock(256, 128, 512, 8, init_values=1 / 6, stable_softmax_2d=True).eval()
    with torch.no_grad():
        for p in blk.parameters():
            if p.dim() == 1:
                p.add_(torch.randn_like(p) * 0.05)
        v, l = torch.randn(2, S, 256), torch.randn(2, N, 128)
        blk.attn.stream_threshold_bytes = 1 << 60
        v0, l0 = blk(v, l)
        blk.attn.stream_threshold_bytes = 0
        v1, l1 = blk(v, l)
    torch.testing.assert_close(v1, v0, rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(l1, l0, rtol=1e-5, atol=1e-5)


def test_streaming_is_skipped_when_the_clamps_could_bind():
    torch.manual_seed(1)
    blk = BiAttentionBlock(256, 128, 512, 8, init_values=1 / 6, stable_softmax_2d=True).eval()
    with torch.no_grad():
        blk.attn.l_proj.weight.mul_(1e5)  # scores far beyond +-5e4: the literal path (with its clamps) must be taken
        v, l = torch.randn(1, 50, 256), torch.randn(1, 5, 128)
        blk.attn.stream_threshold_bytes = 1 << 60
        v0, l0 = blk(v, l)
        blk.attn.stream_threshold_bytes = 0
        v1, l1 = blk(v, l)
    assert torch.equal(v1, v0) and torch.equal(l1, l0)


def reference_case():
    """The block with the synthetic weights (ape_b200/synthetic.py), seeded inputs and the seeded sample of vision rows whose
    reference outputs tests/golden/vlf_reference.npz holds (with every language row)."""
    from ape_b200 import synthetic

    mine = BiAttentionBlock(256, 128, 512, 8, init_values=1 / 6, stable_softmax_2d=True).eval()
    synthetic.fill_state_dict(mine)
    g = torch.Generator().manual_seed(2)
    v, l = torch.randn(2, 400, 256, generator=g), torch.randn(2, 9, 128, generator=g)
    rows = torch.randperm(400, generator=g)[:32].sort()[0]
    return mine, v, l, rows


def test_literal_path_equals_reference_module():
    """The restated literal path against the reference's own BiAttentionBlock (recorded by tests/golden/gen_reference_golden.py)."""
    from conftest import load_golden

    gold = load_golden("vlf_reference.npz")
    mine, v, l, rows = reference_case()
    rv, rl = gold["v_rows"], gold["l"]
    with torch.no_grad():
        mine.attn.stream_threshold_bytes = 1 << 60
        mv, ml = mine(v, l)
        mine.attn.stream_threshold_bytes = 0
        sv, sl = mine(v, l)
    torch.testing.assert_close(mv[:, rows], rv, rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(ml, rl, rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(sv[:, rows], rv, rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(sl, rl, rtol=1e-5, atol=1e-5)
