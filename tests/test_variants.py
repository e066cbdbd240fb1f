"""Host-side drop-in contract of the SURVEY.md 8(f3) SimpleViT-family variants and of attention without output
projection: same state_dict layout, same fp32 values as the UNMODIFIED reference (goldens made by
tests/golden/make_golden.py round2), same constructor keywords, bit-identical init under one seed.  CPU only."""
import inspect

import pytest
import torch

from conftest import load_golden, reference_init
from golden_weights import dropin_class

SURFACE = load_golden("reference_surface")

VARIANTS = ["simplevit_registers", "simplevit_qknorm", "simplevit_patchdrop", "simplevit_flash",
            "simplevit_1d", "simplevit_3d", "simplevit_3d_pf1"]
ALL = ["vit_tiny_noproj"] + VARIANTS


@pytest.fixture(params=ALL)
def g(request):
    return load_golden(request.param)


def test_state_dict_layout_equals_reference(g):
    m = dropin_class(g["kind"])(**g["kwargs"])
    ours, ref = m.state_dict(), g["state_dict"]
    assert list(ours.keys()) == list(ref.keys())
    for k in ref:
        assert ours[k].shape == ref[k].shape, k


def test_eager_forward_equals_reference_golden(g):
    m = dropin_class(g["kind"])(**g["kwargs"]).eval()
    m.load_state_dict(g["state_dict"])
    m = m.float()
    with torch.inference_mode():
        out = m(g["input"].float())
    assert out.shape == g["logits_fp32"].shape
    assert torch.allclose(out, g["logits_fp32"], rtol=1e-5, atol=5e-6), (out - g["logits_fp32"]).abs().max()
    assert m.fused_reason(g["input"].float()) is not None          # CPU fp32 call: PyTorch graph, reason stated


@pytest.mark.parametrize("name", VARIANTS)
def test_constructor_keywords_and_same_seed_init_equal_the_reference(name):
    g = load_golden(name)
    our_cls = dropin_class(g["kind"])
    ps_our = [(p, v.default) for p, v in inspect.signature(our_cls.__init__).parameters.items() if p != "self"]
    assert ps_our == SURFACE["signatures"][g["kind"]]
    assert SURFACE["init"][name]["kwargs"] == g["kwargs"]
    reference_init(name, our_cls)                # parameters drawn under seed 123: bit-identical to the reference's


def test_patch_dropout_is_training_only():
    from vit_pytorch_b200.simple_vit_with_patch_dropout import PatchDropout, SimpleViT
    pd = PatchDropout(0.5)
    x = torch.randn(2, 16, 8)
    pd.eval()
    assert pd(x) is x
    pd.train()
    assert pd(x).shape == (2, 8, 8)
    m = SimpleViT(image_size=32, patch_size=8, num_classes=3, dim=32, depth=1, heads=1, mlp_dim=32).train()
    assert m.fused_reason(torch.randn(1, 3, 32, 32)) == "patch dropout is active (training)"
    assert m(torch.randn(2, 3, 32, 32)).shape == (2, 3)


def test_qk_norm_head_is_a_layernorm_like_the_reference():
    from vit_pytorch_b200.simple_vit_with_qk_norm import SimpleViT
    m = SimpleViT(image_size=32, patch_size=8, num_classes=5, dim=32, depth=1, heads=1, mlp_dim=32).eval()
    assert isinstance(m.linear_head, torch.nn.LayerNorm)
    assert m(torch.randn(2, 3, 32, 32)).shape == (2, 32)           # features, not logits (reference quirk)


def test_refresh_fused_weights_invalidates_prepared_copies():
    """Writes through `.data` do not bump parameter versions (ADVICE r1): the explicit epoch does."""
    from vit_pytorch_b200 import ViT, engine
    m = ViT(image_size=32, patch_size=8, num_classes=3, dim=64, depth=1, heads=1, mlp_dim=64)
    ps = list(m.parameters())
    k0 = engine._version_key(ps)
    ps[0].data.mul_(2.0)
    assert engine._version_key(ps) == k0                            # the blind spot
    m.refresh_fused_weights()
    assert engine._version_key(ps) != k0
    k1 = engine._version_key(ps)
    m.load_state_dict(m.state_dict())
    assert engine._version_key(ps) != k1                            # load_state_dict refreshes on its own


# ---------------------------------------------------------------------------------------------------------------------
# nested-tensor NaViT front-end (SURVEY.md 8(f2), reference na_vit_nested_tensor.py)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["navit_nested_tiny", "navit_nested_noqknorm"])
def test_navit_nested_dropin_equals_reference_golden(name):
    from vit_pytorch_b200.na_vit_nested_tensor import NaViT
    g = load_golden(name)
    m = NaViT(**g["kwargs"]).eval()
    assert list(m.state_dict().keys()) == list(g["state_dict"].keys())
    m.load_state_dict(g["state_dict"])
    m = m.float()
    imgs = [im.float() for im in g["images"]]
    with torch.inference_mode():
        out = m(imgs)
    assert out.shape == g["logits_fp32"].shape
    assert torch.allclose(out, g["logits_fp32"], rtol=1e-4, atol=2e-5), (out - g["logits_fp32"]).abs().max()
    assert m.fused_reason(imgs) == "input is not on a CUDA device"


def test_navit_nested_same_seed_init_and_signature_equal_the_reference():
    from vit_pytorch_b200.na_vit_nested_tensor import NaViT
    po = [(p, v.default) for p, v in inspect.signature(NaViT.__init__).parameters.items() if p != "self"]
    assert po == SURFACE["signatures"]["na_vit_nested_tensor"]
    reference_init("navit_nested", NaViT)        # parameters drawn under seed 5: bit-identical to the reference's
