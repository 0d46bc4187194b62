"""GPU parity tests for ms_deform_attn_forward through the C-ABI (ape_b200 -> libape_b200.so),
against (1) the C oracle, (2) golden vectors generated from the reference, (3) the reference's
own CUDA kernel compiled for sm_100a (recorded outputs), plus size-independent properties at the
full APE-L_D shapes."""
import glob
import os

import pytest
import torch

from conftest import GOLDEN, load_golden
from oracle import msda as O

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
L5_1024 = [(256, 256), (128, 128), (64, 64), (32, 32), (16, 16)]
L4 = [(128, 128), (64, 64), (32, 32), (16, 16)]


@pytest.fixture(scope="module")
def ape():
    import ape_b200

    return ape_b200


def run(ape, value, ss, st, loc, attn, variant=-1):
    return ape.ops.ms_deform_attn_forward(value, ss, st, loc, attn, 64, variant=variant)


def to_dev(ts, dtype=None):
    out = []
    for t in ts:
        t = t.to(DEV)
        if dtype is not None and t.is_floating_point():
            t = t.to(dtype)
        out.append(t)
    return out


GOLD = sorted(os.path.basename(p) for p in glob.glob(os.path.join(GOLDEN, "msda_*.npz")) if "module" not in p)


@pytest.mark.parametrize("case", GOLD)
def test_golden_vectors_from_reference(ape, case):
    g = load_golden(case)
    v, ss, st, loc, attn = to_dev([g["value"], g["shapes"], g["starts"], g["loc"], g["attn"]])
    out = torch.ops.ape.ms_deform_attn_forward(v, ss, st, loc, attn, 64)
    # tolerance stated by north_star: 1e-3 rel; fp32 reassociation gives ~1e-6 here
    torch.testing.assert_close(out.cpu(), g["out"], rtol=1e-5, atol=5e-6)


@pytest.mark.parametrize("variant", [-1, 1, 2, 8, 1 | (1 << 8), 1 | (2 << 8), 8 | (2 << 8), 0x1000])
@pytest.mark.parametrize("border", [False, True])
def test_fp32_vs_c_oracle_all_variants(ape, variant, border):
    ins = O.make_inputs(2, 333, 8, 32, [(40, 56), (20, 28), (10, 14), (5, 7), (3, 4)], 4, seed=11, border=border)
    want = O.msda_c(*ins)
    got = run(ape, *to_dev(ins), variant=variant)
    torch.testing.assert_close(got.cpu(), want, rtol=1e-4, atol=2e-5)


@pytest.mark.parametrize("dtype,atol", [(torch.float16, 2e-3), (torch.bfloat16, 1.5e-2)])
def test_half_precisions_vs_oracle_on_rounded_inputs(ape, dtype, atol):
    ins = O.make_inputs(2, 257, 8, 32, [(33, 47), (17, 24), (9, 12), (5, 6)], 4, seed=12, border=True)
    dins = to_dev(ins, dtype)
    # oracle sees exactly the rounded inputs; remaining error = output rounding (fp32 accumulation inside)
    want = O.msda_c(*[t.cpu() for t in dins])
    got = run(ape, *dins)
    assert got.dtype == dtype
    torch.testing.assert_close(got.float().cpu(), want, rtol=1e-2, atol=atol)


@pytest.mark.parametrize("D,H,P,shapes", [
    (8, 4, 2, [(7, 9)]),                 # fp32 lanes-per-row 2
    (16, 4, 8, [(9, 7), (5, 4)]),        # lanes-per-row 4, P=8
    (64, 2, 4, [(12, 12), (6, 6)]),      # lanes-per-row 16
    (128, 1, 1, [(5, 5)]),               # lanes-per-row 32, single point
    (24, 3, 3, [(6, 5), (3, 3)]),        # not a power of two -> scalar kernel, H not a power of two
    (4, 2, 4, [(4, 4)]),                 # one 16-byte lane per row
])
def test_other_head_dims_and_points(ape, D, H, P, shapes):
    ins = O.make_inputs(3, 41, H, D, shapes, P, seed=13, border=True)
    want = O.msda_c(*ins)
    got = run(ape, *to_dev(ins))
    torch.testing.assert_close(got.cpu(), want, rtol=1e-4, atol=2e-5)


def test_empty_and_degenerate_inputs(ape):
    ins = O.make_inputs(1, 5, 8, 32, [(4, 4)], 4, seed=1)
    v, ss, st, loc, attn = to_dev(ins)
    # no queries
    out = run(ape, v, ss, st, loc[:, :0].contiguous(), attn[:, :0].contiguous())
    assert out.shape == (1, 0, 256)
    # every sample out of range -> exact zeros (output is fully written, no pre-zeroing needed)
    out = run(ape, v, ss, st, loc * 0 + 3.0, attn)
    assert out.abs().max().item() == 0
    out = run(ape, v, ss, st, loc * 0 - 1.0, attn)
    assert out.abs().max().item() == 0
    # NaN locations fail the in-range test (all comparisons false) -> skipped, like the reference
    out = run(ape, v, ss, st, loc * float("nan"), attn)
    assert out.abs().max().item() == 0
    # non-contiguous input is rejected like the reference's AT_ASSERTM
    with pytest.raises(RuntimeError, match="contiguous"):
        run(ape, v.transpose(1, 2), ss, st, loc, attn)


def test_exact_corner_and_edge_locations(ape):
    # texel centres: loc = (i+0.5)/size must return the texel itself
    H_, W_ = 5, 7
    v = torch.arange(H_ * W_ * 8, dtype=torch.float32).view(1, H_ * W_, 1, 8)
    ss = torch.tensor([[H_, W_]])
    st = torch.tensor([0])
    ys, xs = torch.meshgrid(torch.arange(H_), torch.arange(W_), indexing="ij")
    loc = torch.stack([(xs + 0.5) / W_, (ys + 0.5) / H_], -1).view(1, H_ * W_, 1, 1, 1, 2).float()
    attn = torch.ones(1, H_ * W_, 1, 1, 1)
    got = run(ape, *to_dev([v, ss, st, loc, attn]))
    torch.testing.assert_close(got.cpu().view(H_ * W_, 8), v.view(H_ * W_, 8), rtol=0, atol=1e-4)


def ref_kernel_cases():
    """(name, device inputs, sampled query indices) of the comparisons with the reference's own CUDA kernel, whose outputs at
    those queries tests/golden/gen_msda_ref_kernel_golden.py recorded in ref_kernel_msda.npz."""
    S = sum(h * w for h, w in L5_1024)
    dec = O.make_inputs(2, 900, 8, 32, L5_1024, 4, seed=3, border=True)
    g = torch.Generator().manual_seed(4)
    dec_idx = torch.randperm(900, generator=g)[:32].sort()[0]
    enc_idx = torch.randperm(S, generator=g)[:64].sort()[0]
    return [("decoder_f32", to_dev(dec, torch.float32), dec_idx), ("decoder_f16", to_dev(dec, torch.float16), dec_idx),
            ("encoder_f32", to_dev(O.make_inputs(1, S, 8, 32, L5_1024, 4, seed=3, border=True)), enc_idx)]


@pytest.fixture(scope="module")
def ref_kernel():
    gold = load_golden("ref_kernel_msda.npz")
    return {name: (ins, idx.to(DEV), gold[name].to(DEV)) for name, ins, idx in ref_kernel_cases()}


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_against_reference_cuda_kernel_decoder_shape(ape, ref_kernel, dtype):
    ins, idx, ref = ref_kernel["decoder_f32" if dtype == torch.float32 else "decoder_f16"]
    got = run(ape, *ins)[:, idx]
    assert ref.dtype == dtype
    if dtype == torch.float32:
        torch.testing.assert_close(got, ref, rtol=1e-5, atol=5e-6)
    else:
        # the reference accumulates in half (…cuh:270); we accumulate in fp32
        torch.testing.assert_close(got.float(), ref.float(), rtol=2e-2, atol=2e-2)


def test_against_reference_cuda_kernel_encoder_shape_full_size(ape, ref_kernel):
    """BASELINE.json config 2 shape: Q = S = 87 296, 5 levels (too slow for the CPU oracle; the
    reference's own kernel is the checker, at a seeded sample of queries)."""
    ins, idx, ref = ref_kernel["encoder_f32"]
    for variant in (-1, 1, 8):
        got = run(ape, *ins, variant=variant)[:, idx]
        torch.testing.assert_close(got, ref, rtol=1e-5, atol=5e-6)


def test_full_size_properties(ape):
    """Size-independent properties at the full encoder shape: linearity in value, linearity in the
    attention weights, batch independence, and a CPU-oracle spot check on a random query subset."""
    S = sum(h * w for h, w in L5_1024)
    v, ss, st, loc, attn = to_dev(O.make_inputs(2, S, 8, 32, L5_1024, 4, seed=21, border=True))
    base = run(ape, v, ss, st, loc, attn)
    v2 = torch.randn_like(v)
    lin = run(ape, v * 0.5 + v2, ss, st, loc, attn)
    torch.testing.assert_close(lin, base * 0.5 + run(ape, v2, ss, st, loc, attn), rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(run(ape, v, ss, st, loc, attn * 2), base * 2, rtol=1e-5, atol=1e-5)
    swapped = run(ape, v.flip(0).contiguous(), ss, st, loc.flip(0).contiguous(), attn.flip(0).contiguous())
    assert torch.equal(swapped.flip(0), base)
    idx = torch.randperm(S, generator=torch.Generator().manual_seed(0))[:512].to(DEV)
    want = O.msda_c(v.cpu(), ss.cpu(), st.cpu(), loc[:, idx].cpu(), attn[:, idx].cpu())
    torch.testing.assert_close(base[:, idx].cpu(), want, rtol=1e-4, atol=2e-5)


def test_cuda_graph_capture(ape):
    ins = to_dev(O.make_inputs(1, 900, 8, 32, L4, 4, seed=5))
    eager = run(ape, *ins)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        run(ape, *ins)
        s.synchronize()
        with torch.cuda.graph(g, stream=s):
            out = run(ape, *ins)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager)


@pytest.mark.parametrize("tag", ["ref2", "ref4"])
@pytest.mark.parametrize("dtype", [torch.float32])
def test_module_forward_matches_reference_module_golden(ape, tag, dtype):
    """Whole MultiScaleDeformableAttention.forward (multi_scale_deform_attn.py:215-358) recorded from
    the reference module (pytorch_attn=True) vs ape_b200's module (fused kernel)."""
    from ape_b200.layers import MultiScaleDeformableAttention

    g = load_golden(f"msda_module_{tag}.npz")
    L = g["shapes"].shape[0]
    m = MultiScaleDeformableAttention(embed_dim=64, num_heads=4, num_levels=L, num_points=4, dropout=0.0,
                                      batch_first=True).eval()
    sd = {k[3:]: v for k, v in g.items() if k.startswith("sd.")}
    missing, unexpected = m.load_state_dict(sd, strict=True)
    assert not missing and not unexpected  # same parameter names as the reference module
    m = m.to(DEV)
    torch.backends.cuda.matmul.allow_tf32 = False
    with torch.no_grad():
        out = m(g["query"].to(DEV), value=g["value"].to(DEV), identity=g["query"].to(DEV),
                query_pos=g["query_pos"].to(DEV), key_padding_mask=g["mask"].to(DEV),
                reference_points=g["ref"].to(DEV), spatial_shapes=g["shapes"].to(DEV),
                level_start_index=g["starts"].to(DEV))
    torch.testing.assert_close(out.cpu(), g["out"], rtol=1e-3, atol=1e-4)


def test_fused_entry_equals_unfused_composition(ape):
    """ape_msda_fused_fwd == softmax + location arithmetic (torch) + ape_msda_fwd."""
    B, Q, H, D, P = 2, 500, 8, 32, 4
    shapes = [(30, 40), (15, 20), (8, 10), (4, 5), (2, 3)]
    L = len(shapes)
    g = torch.Generator().manual_seed(9)
    ss = torch.tensor(shapes)
    st = O.level_start_index(ss)
    S = int((ss[:, 0] * ss[:, 1]).sum())
    value = torch.randn(B, S, H, D, generator=g).to(DEV)
    offs = (torch.randn(B, Q, H * L * P * 2, generator=g) * 3).to(DEV)
    logits = torch.randn(B, Q, H * L * P, generator=g).to(DEV)
    for ref_dim in (2, 4):
        ref = torch.rand(B, Q, L, ref_dim, generator=g).to(DEV)
        o6 = offs.view(B, Q, H, L, P, 2)
        attn = logits.view(B, Q, H, L * P).softmax(-1).view(B, Q, H, L, P)
        if ref_dim == 2:
            norm = torch.stack([ss[:, 1], ss[:, 0]], -1).to(DEV)
            loc = ref[:, :, None, :, None, :] + o6 / norm[None, None, None, :, None, :]
        else:
            loc = ref[:, :, None, :, None, :2] + o6 / P * ref[:, :, None, :, None, 2:] * 0.5
        want = run(ape, value, ss.to(DEV), st.to(DEV), loc.contiguous(), attn.contiguous())
        # offsets/logits as column slices of one wider buffer (how the module calls it)
        qo = torch.cat([offs, logits], -1)
        got = ape.ops.ms_deform_attn_fused_forward(value, ss.to(DEV), st.to(DEV), qo[..., :H * L * P * 2],
                                                   qo[..., H * L * P * 2:], ref, P)
        torch.testing.assert_close(got, want, rtol=1e-4, atol=2e-5)


def _encoder_like_case(shapes, B, H, D, P, dtype, seed, off_scale):
    """Queries = pixels; reference points = pixel centres (get_reference_points, deformable_transformer_vl.py:371-400);
    offsets of a few pixels, as the sampling_offsets bias grid produces (multi_scale_deform_attn.py:195-207)."""
    L = len(shapes)
    g = torch.Generator().manual_seed(seed)
    ss = torch.tensor(shapes)
    st = O.level_start_index(ss)
    S = int((ss[:, 0] * ss[:, 1]).sum())
    value = torch.randn(B, S, H, D, generator=g).to(DEV, dtype)
    offs = torch.randn(B, S, H * L * P * 2, generator=g) * off_scale
    qo = torch.cat([offs, torch.randn(B, S, H * L * P, generator=g)], -1).to(DEV, dtype)
    pts = []
    for (h, w) in shapes:
        ys, xs = torch.meshgrid((torch.arange(h) + 0.5) / h, (torch.arange(w) + 0.5) / w, indexing="ij")
        pts.append(torch.stack([xs.reshape(-1), ys.reshape(-1)], -1))
    ref = torch.cat(pts, 0)[None, :, None, :].expand(B, S, L, 2).contiguous().to(DEV)
    return value, ss, st, qo, ref


def _pair_run(ape, value, ss, st, shapes, qo, n_off, ref, P, H, mask=None, hpc=0, tile_w=None, head_major=None):
    B, S = value.shape[:2]
    v2 = ape.ops.msda_pair_values(value.view(B, S, -1), H, token_mask=mask)
    return ape.ops.ms_deform_attn_pair_fused_forward(v2, ss.to(DEV), st.to(DEV), shapes, qo[..., :n_off], qo[..., n_off:], ref, P,
                                                     heads_per_cta=hpc, tile_w=tile_w, head_major=head_major)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("shapes", [[(40, 56), (20, 28), (10, 14), (5, 7), (3, 4)], [(16, 16), (8, 8)], [(33, 17)],
                                    [(32, 48), (16, 24), (8, 12), (4, 6), (2, 3)], [(64, 32), (32, 16), (16, 8), (8, 4)],
                                    [(7, 2), (1, 2)]])
def test_pair_kernel_equals_generic_fused(ape, dtype, shapes):
    """ape_msda_pair_fused_fwd (pair layout, 16-bit corner blend per level, fp32 across levels) against ape_msda_fused_fwd
    (fp32 blend) on encoder-like calls: same sampling semantics incl. every border case; the difference is the 16-bit
    rounding of the per-level partial sums (bounded below by the rounding of the 16-bit output itself)."""
    B, H, D, P = 2, 8, 32, 4
    n_off = H * len(shapes) * P * 2
    tol = {torch.float16: 4e-3, torch.bfloat16: 3e-2}[dtype]
    assert ape.ops.msda_pair_supported(shapes, H, D, P, dtype)
    for seed, off_scale in ((17, 3.0), (18, 8.0), (19, 0.5), (20, 40.0)):  # (20: most samples out of range / on borders)
        value, ss, st, qo, ref = _encoder_like_case(shapes, B, H, D, P, dtype, seed, off_scale)
        a = ape.ops.ms_deform_attn_fused_forward(value, ss.to(DEV), st.to(DEV), qo[..., :n_off], qo[..., n_off:], ref, P)
        # CTA mappings: auto (8-wide pixel tiles), all heads per CTA, consecutive queries, 16 / 32 / 4-wide tiles, head-major order
        for hpc, tw, hm in ((0, None, None), (8, None, None), (0, 0, 0), (0, 16, 1), (0, 32, 0), (0, 4, 1), (2, 8, 1)):
            b = _pair_run(ape, value, ss, st, shapes, qo, n_off, ref, P, H, hpc=hpc, tile_w=tw, head_major=hm)
            torch.testing.assert_close(b.float(), a.float(), rtol=tol, atol=tol)
    # arbitrary (non pixel-centre) reference points and boxes, fp32 offsets / logits, a token mask
    g = torch.Generator().manual_seed(23)
    S = value.shape[1]
    mask = (torch.rand(B, S, generator=g) < 0.2).to(DEV)
    for ref_dim in (2, 4):
        r = torch.rand(B, S, len(shapes), ref_dim, generator=g).to(DEV)
        vm = value.masked_fill(mask[:, :, None, None], 0.0)
        a = ape.ops.ms_deform_attn_fused_forward(vm, ss.to(DEV), st.to(DEV), qo[..., :n_off], qo[..., n_off:], r, P)
        b = _pair_run(ape, value, ss, st, shapes, qo, n_off, r, P, H, mask=mask)
        torch.testing.assert_close(b.float(), a.float(), rtol=tol, atol=tol)
        qf = qo.float()
        c = _pair_run(ape, value, ss, st, shapes, qf, n_off, r, P, H, mask=mask)
        torch.testing.assert_close(c.float(), a.float(), rtol=tol, atol=tol)


def test_pair_kernel_propagates_no_nan_from_out_of_range_locations(ape):
    """NaN / Inf sampling offsets are out of range in the reference (weight exactly 0): they must not poison the sum."""
    shapes = [(16, 16), (8, 8)]
    B, H, D, P = 1, 8, 32, 4
    n_off = H * len(shapes) * P * 2
    value, ss, st, qo, ref = _encoder_like_case(shapes, B, H, D, P, torch.float16, 3, 2.0)
    qo = qo.clone()
    qo[0, ::7, 0] = float("nan")
    qo[0, ::5, 3] = float("inf")
    a = ape.ops.ms_deform_attn_fused_forward(value, ss.to(DEV), st.to(DEV), qo[..., :n_off], qo[..., n_off:], ref, P)
    b = _pair_run(ape, value, ss, st, shapes, qo, n_off, ref, P, H)
    assert torch.isfinite(b).all() and torch.isfinite(a).all()
    torch.testing.assert_close(b.float(), a.float(), rtol=4e-3, atol=4e-3)


def test_pair_kernel_full_size_vs_oracle(ape):
    """APE-L_D 1024^2 encoder shape (S = 87 296), fp16: pair kernel vs the C oracle (double accumulation) on a random subset
    of queries; prints the error of both the fp32-blend kernel and the pair kernel."""
    shapes = [(256, 256), (128, 128), (64, 64), (32, 32), (16, 16)]
    B, H, D, P, L = 1, 8, 32, 4, 5
    value, ss, st, qo, ref = _encoder_like_case(shapes, B, H, D, P, torch.float16, 5, 2.5)
    n_off = H * L * P * 2
    got = _pair_run(ape, value, ss, st, shapes, qo, n_off, ref, P, H)
    gen = ape.ops.ms_deform_attn_fused_forward(value, ss.to(DEV), st.to(DEV), qo[..., :n_off], qo[..., n_off:], ref, P)
    S = value.shape[1]
    idx = torch.randperm(S, generator=torch.Generator().manual_seed(1))[:3000].sort()[0].to(DEV)
    o6 = qo[0, idx, :n_off].float().view(1, -1, H, L, P, 2)
    attn = qo[0, idx, n_off:].float().view(1, -1, H, L * P).softmax(-1).view(1, -1, H, L, P)
    norm = torch.stack([ss[:, 1], ss[:, 0]], -1).to(DEV).float()
    loc = ref[:, idx][:, :, None, :, None, :] + o6 / norm[None, None, None, :, None, :]
    want = O.msda_c(value.float().cpu(), ss, st, loc.cpu().contiguous(), attn.cpu().contiguous())
    e_pair = (got[0, idx].float().cpu() - want[0]).abs()
    e_gen = (gen[0, idx].float().cpu() - want[0]).abs()
    rms = want.pow(2).mean().sqrt().item()
    print(f"\nfull-size fp16 MSDA vs C oracle (rms {rms:.3f}): fp32-blend kernel max {e_gen.max():.2e} mean {e_gen.mean():.2e}; "
          f"pair kernel max {e_pair.max():.2e} mean {e_pair.mean():.2e}")
    torch.testing.assert_close(got[0, idx].float().cpu(), want[0], rtol=3e-3, atol=3e-3)
