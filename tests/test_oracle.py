"""The oracle (oracle/vit_oracle.py) against outputs of the reference: committed golden fixtures, and the reference's
logits on seeded models (tests/golden/reference_surface.pt)."""
import pytest
import torch

from conftest import load_golden, reference_init, state_digest
from oracle import vit_oracle as O

SURFACE = load_golden("reference_surface")


def test_oracle_matches_golden(golden):
    sd = O.upcast(golden["state_dict"])
    out = O.forward(golden["kind"], sd, golden["kwargs"], golden["input"].float())
    ref = golden["logits_fp32"]
    assert out.shape == ref.shape
    # fp32 vs fp32 of the same algorithm: only summation-order noise
    assert torch.allclose(out, ref, rtol=1e-5, atol=5e-6), (out - ref).abs().max()


def test_oracle_fp64_bounds_fp32_noise(golden):
    sd = O.upcast(golden["state_dict"], torch.float64)
    out = O.forward(golden["kind"], sd, golden["kwargs"], golden["input"].double())
    assert (out.float() - golden["logits_fp32"]).abs().max() < 2e-5


def test_oracle_tokens_match_golden():
    g = load_golden("vit_tiny_cls")
    sd = O.upcast(g["state_dict"])
    x = O.patch_embed(sd, g["input"].float()[:1], 4, 4)
    x = torch.cat([sd["cls_token"][None], x], 1) + sd["pos_embedding"][: x.shape[1] + 1]
    tok = O.transformer(sd, x, g["kwargs"]["depth"], g["kwargs"]["heads"], "vit")
    assert torch.allclose(tok, g["tokens_fp32"], rtol=1e-5, atol=1e-5)


def test_patchify_index_formula():
    img = torch.arange(2 * 3 * 8 * 12, dtype=torch.float32).reshape(2, 3, 8, 12)
    p = O.patchify(img, 4, 2)
    gw = 12 // 2
    for (b, h, w, p1, p2, c) in [(0, 0, 0, 0, 0, 0), (1, 1, 5, 3, 1, 2), (0, 1, 2, 2, 0, 1)]:
        assert p[b, h * gw + w, (p1 * 2 + p2) * 3 + c] == img[b, c, h * 4 + p1, w * 2 + p2]


def test_sincos_table_properties():
    pe = O.posemb_sincos_2d(3, 5, 16)
    assert pe.shape == (15, 16) and pe.dtype == torch.float32
    # token 0 is (y=0, x=0): sin = 0, cos = 1
    assert torch.equal(pe[0], torch.tensor([0.] * 4 + [1.] * 4 + [0.] * 4 + [1.] * 4))
    # token index = y*w + x: token 7 -> y=1, x=2, omega_0 = 1
    assert torch.allclose(pe[7, 0], torch.sin(torch.tensor(2.0))) and torch.allclose(pe[7, 8], torch.sin(torch.tensor(1.0)))


def test_gelu_and_softmax_against_torch():
    x = torch.linspace(-6, 6, 1001)
    assert torch.allclose(O.gelu_erf(x), torch.nn.functional.gelu(x), atol=1e-6)
    s = torch.randn(4, 7, 9)
    assert torch.allclose(O.softmax_last(s), s.softmax(-1), atol=1e-6)


def test_flops_formula_matches_baseline_md():
    f = O.flops_per_image(image_size=224, patch_size=16, dim=768, depth=12, heads=12, mlp_dim=3072, num_classes=1000)
    assert abs(f / 1e9 - 35.128) < 5e-3
    f = O.flops_per_image(image_size=224, patch_size=16, dim=1024, depth=24, heads=16, mlp_dim=4096, num_classes=1000)
    assert abs(f / 1e9 - 123.109) < 5e-3
    f = O.flops_per_image(image_size=224, patch_size=16, dim=768, depth=12, heads=12, mlp_dim=3072, num_classes=1000,
                          cls_tokens=0)
    assert abs(f / 1e9 - 34.943) < 5e-3


@pytest.mark.parametrize("kind,seed", [("vit", 11), ("simple", 12), ("vit", 13)])
def test_oracle_matches_live_reference(kind, seed):
    """Seeded reference models on a seeded input (reference_surface.pt): the drop-in's constructor rebuilds the
    reference's parameters bit for bit, the oracle on them gives the reference's logits."""
    from vit_pytorch_b200 import SimpleViT, ViT
    name = f"{kind}_{seed}"
    model = reference_init(name, ViT if kind == "vit" else SimpleViT)
    img = torch.randn(3, 3, 64, 64)
    want = SURFACE["oracle"][name]
    assert state_digest({"img": img})["img"] == want["input"]
    got = O.forward(kind, O.upcast(model.state_dict()), SURFACE["init"][name]["kwargs"], img)
    assert torch.allclose(got, want["logits"], rtol=1e-5, atol=5e-6)


def test_oracle_matches_live_reference_vit_b16():
    from vit_pytorch_b200 import ViT
    model = reference_init("vit_b16", ViT)
    torch.manual_seed(1)
    img = torch.randn(1, 3, 224, 224)
    want = SURFACE["oracle"]["vit_b16"]
    assert state_digest({"img": img})["img"] == want["input"]
    got = O.vit_forward(O.upcast(model.state_dict()), SURFACE["init"]["vit_b16"]["kwargs"], img)
    assert torch.allclose(got, want["logits"], rtol=1e-4, atol=2e-5), (got - want["logits"]).abs().max()
