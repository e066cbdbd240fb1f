"""NaViT (reference na_vit.py): oracle and host-side mirror against outputs of the reference (CPU)."""
import pytest
import torch

from conftest import load_golden, reference_init
from oracle import navit_oracle as NO
from oracle import vit_oracle as O
from vit_pytorch_b200.na_vit import NaViT, group_images_by_max_seq_len


@pytest.fixture(scope="module")
def g():
    return load_golden("navit_tiny")


def test_oracle_per_image_equals_reference_packed(g):
    """The unpacked, mask-free per-image restatement reproduces the reference's packed + masked forward."""
    sd = O.upcast(g["state_dict"])
    imgs = [im.float() for im in g["images"]]
    out = NO.navit_forward(sd, g["kwargs"], [[imgs[i] for i in r] for r in g["rows"]])
    assert out.shape == g["logits_fp32"].shape
    assert torch.allclose(out, g["logits_fp32"], rtol=1e-4, atol=2e-5), (out - g["logits_fp32"]).abs().max()
    # packing is irrelevant to the result: the reference's own greedy re-grouping gives the same logits
    assert torch.allclose(out, g["logits_grouped_fp32"], rtol=1e-4, atol=2e-5)


def test_grouping_matches_reference_rule(g):
    imgs = g["images"]
    ours = group_images_by_max_seq_len(imgs, 8, max_seq_len=g["group_max_seq_len"])
    orc = NO.group_images_by_max_seq_len(imgs, 8, max_seq_len=g["group_max_seq_len"])
    sizes = lambda groups: [[tuple(im.shape[-2:]) for im in grp] for grp in groups]
    assert sizes(ours) == sizes(orc)
    toks = [[(im.shape[-2] // 8) * (im.shape[-1] // 8) for im in grp] for grp in ours]
    assert all(sum(t) <= 80 for t in toks) and sum(len(t) for t in toks) == len(imgs)
    with pytest.raises(AssertionError, match="exceeds maximum sequence length"):
        group_images_by_max_seq_len([torch.zeros(3, 64, 64)], 8, max_seq_len=10)


def test_module_state_dict_and_forward(g):
    m = NaViT(**g["kwargs"]).eval()
    assert list(m.state_dict().keys()) == list(g["state_dict"].keys())
    m.load_state_dict(g["state_dict"])
    m = m.float()
    imgs = [im.float() for im in g["images"]]
    with torch.inference_mode():
        packed = m([[imgs[i] for i in r] for r in g["rows"]])
        grouped = m(imgs, group_images=True, group_max_seq_len=g["group_max_seq_len"])
        single_row = m(imgs[:3])                                   # List[Tensor] = one row
    assert torch.allclose(packed, g["logits_fp32"], rtol=1e-4, atol=2e-5)
    assert torch.allclose(grouped, g["logits_grouped_fp32"], rtol=1e-4, atol=2e-5)
    assert torch.allclose(single_row, g["logits_fp32"][:3], rtol=1e-4, atol=2e-5)
    assert m.fused_reason() is not None                            # no input given: stated, not hidden
    assert m.fused_reason(imgs) == "input is not on a CUDA device"   # fp32 CPU call -> the PyTorch graph


def test_patch_order_is_channel_major():
    img = torch.arange(3 * 4 * 6, dtype=torch.float32).reshape(3, 4, 6)
    p = NO.patchify_cpp(img, 2)
    # token (h=1, w=2), element (c=2, p1=1, p2=0)
    assert p[1 * 3 + 2, (2 * 2 + 1) * 2 + 0] == img[2, 1 * 2 + 1, 2 * 2 + 0]


def test_same_seed_init_and_live_reference():
    """Seeded reference NaViT (reference_surface.pt): bit-identical parameters from the same seed, and the drop-in
    and the oracle reproduce the reference's packed forward of three images."""
    surface = load_golden("reference_surface")
    b = reference_init("navit", NaViT).eval()
    imgs, want = surface["navit"]["images"], surface["navit"]["logits"]
    with torch.inference_mode():
        got = b([imgs[:2], imgs[2:]])
    assert torch.allclose(got, want, rtol=1e-5, atol=1e-6)
    kwargs = surface["init"]["navit"]["kwargs"]
    assert torch.allclose(NO.navit_forward(O.upcast(b.state_dict()), kwargs, [imgs[:2], imgs[2:]]), want,
                          rtol=1e-4, atol=1e-5)


def test_varlen_index_arrays_host_logic():
    """_lib.VarlenIndex: one packed buffer holds cu_seqlens / query-tile prefix / patch-row prefix / dims / addresses."""
    from vit_pytorch_b200 import _lib
    p = 16
    sizes = [(48, 32), (16, 16), (512, 512), (64, 80), (2064, 16)]
    imgs = [torch.zeros(3, h, w, dtype=torch.bfloat16) for h, w in sizes]
    ix = _lib.VarlenIndex(imgs, p, "cpu")
    lens = [(h // p) * (w // p) for h, w in sizes]
    assert ix.S == len(sizes) and ix.T == sum(lens) and ix.lengths == lens
    assert ix.cu.dtype == torch.int32 and ix.cu.tolist() == [0] + torch.tensor(lens).cumsum(0).tolist()
    tiles = [(n + 127) // 128 for n in lens]
    assert ix.tile_prefix.tolist() == [0] + torch.tensor(tiles).cumsum(0).tolist() and ix.total_tiles == sum(tiles)
    rows = [h // p for h, _ in sizes]
    assert ix.row_prefix.tolist() == [0] + torch.tensor(rows).cumsum(0).tolist() and ix.total_rows == sum(rows)
    assert ix.dims.tolist() == [v for hw in sizes for v in hw] and ix.max_w == 512
    assert ix.img_ptrs.dtype == torch.int64 and ix.img_ptrs.tolist() == [im.data_ptr() for im in imgs]
    assert ix.cu.data_ptr() % 4 == 0 and ix.img_ptrs.data_ptr() % 8 == 0


def test_navit_lnfold_prepared_tensors_reproduce_layernorm_linear():
    """Host side of the LN-fold (na_vit.py:_prepared): with W_g = W * gamma (bf16), s = rowsum(W_g) and the row
    statistics of the bf16 token copy,  rstd * (xb W_g^T - mu * s) + t  equals  Linear(LayerNorm(x))  of the reference
    modules (Attention.norm -> to_q / to_kv and FeedForward[0] -> [1], na_vit.py:142-146,105-113)."""
    torch.manual_seed(0)
    m = NaViT(image_size=64, patch_size=8, num_classes=5, dim=64, depth=2, heads=2, mlp_dim=128).eval()
    with torch.no_grad():
        for p in m.parameters():                      # non-trivial gammas
            if p.ndim == 1:
                p.add_(0.3 * torch.randn_like(p))
    t = m._prepared()
    x = torch.randn(37, 64) * 2 + 0.5
    xb = x.bfloat16().float()
    mu = xb.mean(1, keepdim=True)
    rstd = torch.rsqrt((xb * xb).mean(1, keepdim=True) - mu * mu + 1e-5)
    for i, (attn, ff) in enumerate(m.transformer.layers):
        with torch.no_grad():
            xn = attn.norm(xb)
            want_qkv = torch.cat([attn.to_q(xn), attn.to_kv(xn)], dim=-1)
            want_h = ff[1](ff[0](xb))
        got_qkv = rstd * (xb @ t[f"{i}.a.qkvg"].float().t() - mu * t[f"{i}.a.qkvs"]) + t[f"{i}.a.qkvt"]
        got_h = rstd * (xb @ t[f"{i}.f.w1g"].float().t() - mu * t[f"{i}.f.w1s"]) + t[f"{i}.f.b1"]
        assert torch.allclose(got_qkv, want_qkv, rtol=2e-2, atol=2e-2), (got_qkv - want_qkv).abs().max()
        assert torch.allclose(got_h, want_h, rtol=2e-2, atol=2e-2), (got_h - want_h).abs().max()
        assert t[f"{i}.a.gqk"].numel() == 2 * 2 * 64 and t[f"{i}.a.qkvt"].abs().max() == 0


def test_oracle_and_dropin_at_config5_geometry_equal_the_reference_golden():
    """BASELINE.json configs[4] geometry (dim 1024, depth 6, heads 16, mlp 4096; images of 1 ... 1024 tokens): the
    per-image oracle and the drop-in's own PyTorch graph, on weights rebuilt from the seeds, reproduce the fp32
    logits the UNMODIFIED reference produced (tests/golden/navit_config5.pt, made by make_golden.py)."""
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    from navit_c5_spec import NAVIT_C5, navit_config5_images, navit_config5_model
    g = load_golden("navit_config5")
    assert g["spec"] == NAVIT_C5
    m = navit_config5_model(NaViT)
    imgs = [im.float() for im in navit_config5_images()]
    ref = g["logits_fp32"]
    got = NO.navit_forward(O.upcast(m.state_dict()), NAVIT_C5["kwargs"], [imgs])
    assert got.shape == ref.shape == (len(imgs), 1000)
    assert (got - ref).abs().max().item() < 2e-4, (got - ref).abs().max().item()
    with torch.inference_mode():
        own = m(imgs[:4] + imgs[8:])          # drop-in graph on a subset (the 1024- and 1-token images included)
    assert (own - torch.cat([ref[:4], ref[8:]])).abs().max().item() < 2e-4
