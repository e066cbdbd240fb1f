"""Host-side drop-in contract of vit_pytorch_b200.ViT / SimpleViT (SURVEY.md 8b): constructor signature, state_dict
layout, attribute surface, eager-graph values against the reference goldens, dispatch rules.  CPU only."""
import inspect

import pytest
import torch
from torch import nn

from conftest import load_golden, reference_init, state_digest
from vit_pytorch_b200 import SimpleViT, ViT
from vit_pytorch_b200 import simple_vit as sv_mod
from vit_pytorch_b200 import vit as vit_mod

SURFACE = load_golden("reference_surface")


def _build(g):
    cls = ViT if g["kind"] == "vit" else SimpleViT
    m = cls(**g["kwargs"]).eval()
    m.load_state_dict(g["state_dict"])      # strict: key set and shapes must equal the reference's
    return m


def test_state_dict_layout_equals_reference(golden):
    cls = ViT if golden["kind"] == "vit" else SimpleViT
    m = cls(**golden["kwargs"])
    ours, ref = m.state_dict(), golden["state_dict"]
    assert list(ours.keys()) == list(ref.keys())          # same names AND same registration order
    for k in ref:
        assert ours[k].shape == ref[k].shape, k


def test_eager_forward_equals_reference_golden(golden):
    m = _build(golden).float()
    with torch.inference_mode():
        out = m(golden["input"].float())
    assert torch.allclose(out, golden["logits_fp32"], rtol=1e-5, atol=5e-6)


def test_constructor_signatures():
    sig = inspect.signature(ViT.__init__)
    names = [p for p in sig.parameters if p != "self"]
    assert names == ["image_size", "patch_size", "num_classes", "dim", "depth", "heads", "mlp_dim", "pool", "channels",
                     "dim_head", "dropout", "emb_dropout"]
    assert all(sig.parameters[n].kind is inspect.Parameter.KEYWORD_ONLY for n in names)
    assert sig.parameters["pool"].default == "cls" and sig.parameters["dim_head"].default == 64
    sig = inspect.signature(SimpleViT.__init__)
    names = [p for p in sig.parameters if p != "self"]
    assert names == ["image_size", "patch_size", "num_classes", "dim", "depth", "heads", "mlp_dim", "channels",
                     "dim_head"]


def test_assertion_messages():
    with pytest.raises(AssertionError, match="Image dimensions must be divisible by the patch size."):
        ViT(image_size=30, patch_size=4, num_classes=2, dim=8, depth=1, heads=1, mlp_dim=8)
    with pytest.raises(AssertionError, match="pool type must be either cls"):
        ViT(image_size=32, patch_size=4, num_classes=2, dim=8, depth=1, heads=1, mlp_dim=8, pool="max")
    with pytest.raises(AssertionError, match="multiple of 4"):
        SimpleViT(image_size=32, patch_size=4, num_classes=2, dim=6, depth=1, heads=1, mlp_dim=8)


def test_attribute_surface():
    v = ViT(image_size=32, patch_size=(8, 4), num_classes=5, dim=64, depth=2, heads=2, mlp_dim=96, dim_head=16)
    assert v.patch_size == (8, 4) and v.pool == "cls"
    assert isinstance(v.to_latent, nn.Identity) and isinstance(v.dropout, nn.Dropout)
    assert isinstance(v.to_patch_embedding[1], nn.LayerNorm) and isinstance(v.to_patch_embedding[2], nn.Linear)
    assert v.to_patch_embedding[2].weight.shape == (64, 3 * 8 * 4)
    assert v.cls_token.shape == (1, 64) and v.pos_embedding.shape == (4 * 8 + 1, 64)
    attn, ff = v.transformer.layers[1]
    assert isinstance(attn, vit_mod.Attention) and isinstance(attn.attend, nn.Softmax)
    assert attn.heads == 2 and attn.scale == 16 ** -0.5
    assert isinstance(attn.to_out, nn.Sequential) and isinstance(ff.net, nn.Sequential) and len(ff.net) == 6
    # to_patch_embedding[0] alone is the patchify op (MAE uses it separately, reference mae.py:28-31)
    img = torch.randn(2, 3, 32, 32)
    assert v.to_patch_embedding[0](img).shape == (2, 32, 96)
    s = SimpleViT(image_size=32, patch_size=8, num_classes=5, dim=64, depth=1, heads=2, mlp_dim=96, dim_head=16)
    assert "pos_embedding" not in s.state_dict() and s.pos_embedding.shape == (16, 64)
    assert isinstance(s.transformer.layers[0][0].to_out, nn.Linear) and s.transformer.layers[0][0].to_out.bias is None
    assert len(s.transformer.layers[0][1].net) == 4 and hasattr(s, "linear_head")


def test_edge_cases_shapes():
    # pool='mean' -> no cls token; num_classes=0 -> tokens; heads=1 & dim_head=dim -> Identity projection
    v = ViT(image_size=32, patch_size=8, num_classes=0, dim=32, depth=1, heads=1, mlp_dim=48, dim_head=32,
            pool="mean").eval()
    assert v.cls_token.shape == (0, 32) and v.mlp_head is None
    assert isinstance(v.transformer.layers[0][0].to_out, nn.Identity)
    assert v(torch.randn(2, 3, 32, 32)).shape == (2, 16, 32)
    # smaller, non-square input than image_size (reference README.md:1720-1745)
    v = ViT(image_size=64, patch_size=16, num_classes=7, dim=32, depth=1, heads=2, mlp_dim=48, dim_head=16).eval()
    assert v(torch.randn(2, 3, 64, 32)).shape == (2, 7)
    # the reference's own shape test (tests/test_vit.py:4-20), in train mode with dropout
    v = ViT(image_size=256, patch_size=32, num_classes=1000, dim=64, depth=2, heads=4, mlp_dim=96, dropout=0.1,
            emb_dropout=0.1)
    assert v(torch.randn(1, 3, 256, 256)).shape == (1, 1000)


def test_transformer_callable_on_arbitrary_tokens():
    v = ViT(image_size=32, patch_size=8, num_classes=3, dim=32, depth=2, heads=2, mlp_dim=48, dim_head=16).eval()
    assert v.transformer(torch.randn(2, 5, 32)).shape == (2, 5, 32)     # MAE-style subset of tokens


def test_dispatch_reasons_on_cpu():
    v = ViT(image_size=32, patch_size=8, num_classes=3, dim=128, depth=1, heads=2, mlp_dim=128).eval()
    img = torch.randn(1, 3, 32, 32)
    assert v.fused_reason(img) == "input is not on a CUDA device"
    assert v.transformer.fused_reason(torch.randn(1, 4, 128)) == "input is not on a CUDA device"
    s = SimpleViT(image_size=32, patch_size=8, num_classes=3, dim=128, depth=1, heads=2, mlp_dim=128).eval()
    assert s.fused_reason(img) is not None


def test_hooks_force_the_observable_graph():
    from vit_pytorch_b200.engine import hooks_inside
    v = ViT(image_size=32, patch_size=8, num_classes=3, dim=32, depth=1, heads=2, mlp_dim=48, dim_head=16).eval()
    assert not hooks_inside(v, skip=(v.to_latent,))
    v.to_latent.register_forward_hook(lambda m, i, o: None)       # Dino-style hook on to_latent is allowed
    assert not hooks_inside(v, skip=(v.to_latent,))
    seen = []
    h = v.transformer.layers[0][0].attend.register_forward_hook(lambda m, i, o: seen.append(o.shape))
    assert hooks_inside(v, skip=(v.to_latent,)) and hooks_inside(v.transformer)
    v(torch.randn(2, 3, 32, 32))
    assert seen == [torch.Size([2, 2, 17, 17])]                    # Recorder-style attention maps (B,H,N,N)
    h.remove()


@pytest.mark.parametrize("kind", ["vit", "simple"])
def test_same_seed_gives_bit_identical_init(kind):
    # reference_init checks every parameter against the digest of the reference constructor under the same seed
    b = reference_init(kind, ViT if kind == "vit" else SimpleViT)
    if kind == "simple":
        assert state_digest({"pos_embedding": b.pos_embedding}) == SURFACE["init"]["simple"]["buffers"]


def test_reference_wrappers_accept_the_dropin():
    """Extractor (reference extractor.py:46-59) hooks `vit.transformer` and returns the logits with the transformer
    output: on a drop-in with the reference's seeded weights both equal what the reference's Extractor returned on the
    reference's own ViT."""
    v = reference_init("vit_hooks", ViT).eval()
    g = SURFACE["hooks"]
    seen = []
    v.transformer.register_forward_hook(lambda m, i, o: seen.append(o))
    with torch.no_grad():
        logits = v(g["img"])
    assert torch.allclose(logits, g["logits"], rtol=1e-5, atol=1e-6)
    assert len(seen) == 1 and torch.allclose(seen[0], g["embeddings"], rtol=1e-5, atol=1e-5)


def test_reference_mae_wrapper_runs_on_the_dropin():
    """MAE (reference mae.py:26-31,46-55,60,74) reads `pos_embedding`, `to_patch_embedding[0]`, `[1:]`, `[2].weight`,
    `pool` and calls `encoder.transformer(tokens)` on the unmasked quarter of the tokens: every value it reads or gets
    back equals the reference ViT's (stored from a run of the reference), and gradients reach the encoder through that
    call.  (pool='mean': with the 2-D `pos_embedding` of vit.py:107 the wrapper's `[:, 1:n+1]` slice for pool='cls'
    -- and SimMIM's, simmim.py:45 -- fails on the reference's own ViT too, so there is nothing to match.)"""
    ours = reference_init("vit_mae", ViT).eval()
    g = SURFACE["mae"]
    assert ours.pool == "mean" and ours.pos_embedding.shape[-2:] == (16, 64)
    assert ours.to_patch_embedding[2].weight.shape[-1] == g["pixel_values_per_patch"]
    with torch.no_grad():
        patches = ours.to_patch_embedding[0](g["img"])
        tokens = nn.Sequential(*ours.to_patch_embedding[1:])(patches) + ours.pos_embedding
        encoded = ours.transformer(tokens[torch.arange(3)[:, None], g["keep"]])
    assert torch.equal(patches, g["patches"])
    assert torch.allclose(tokens, g["tokens"], rtol=1e-5, atol=1e-6)
    assert torch.allclose(encoded, g["encoded"], rtol=1e-5, atol=1e-5), (encoded - g["encoded"]).abs().max()
    ours.transformer(tokens[:, :4].detach()).sum().backward()     # and it trains through that call
    assert ours.transformer.layers[0][0].to_qkv.weight.grad is not None


def test_reference_distill_wrapper_accepts_the_dropin_as_teacher():
    """DistillWrapper (reference distill.py:139-141) calls `teacher(img)` under no_grad: the drop-in with the
    reference's seeded weights returns the reference ViT's logits for that call."""
    teacher = reference_init("distill", ViT).eval()
    g = SURFACE["distill"]
    with torch.no_grad():
        logits = teacher(g["img"].float())
    assert not logits.requires_grad
    assert torch.allclose(logits, g["logits_fp32"], rtol=1e-5, atol=1e-6)


def test_recorder_and_extractor_twins():
    """vit_pytorch_b200.recorder / .extractor mirror reference recorder.py:10-59 / extractor.py:18-92."""
    from vit_pytorch_b200.extractor import Extractor
    from vit_pytorch_b200.recorder import Recorder
    torch.manual_seed(0)
    v = ViT(image_size=32, patch_size=8, num_classes=3, dim=32, depth=2, heads=2, mlp_dim=48, dim_head=16).eval()
    img = torch.randn(2, 3, 32, 32)
    with torch.no_grad():
        plain = v(img)
        rec = Recorder(v)
        pred, attns = rec(img)
        assert attns.shape == (2, 2, 2, 17, 17) and torch.allclose(attns.sum(-1), torch.ones(2, 2, 2, 17), atol=1e-5)
        assert torch.equal(pred, plain)
        assert rec.eject() is v and not any(l[0].attend._forward_hooks for l in v.transformer.layers)
        ext = Extractor(v)
        pred, emb = ext(img)
        assert torch.equal(pred, plain) and emb.shape == (2, 17, 32)
        assert ext(img, return_embeddings_only=True).shape == (2, 17, 32)
        first = Extractor(v, layer=v.transformer.layers[0][1], layer_save_input=True)
        _, inp = first(img)
        assert isinstance(inp, tuple) and inp[0].shape == (2, 17, 32)
    # the reference's Recorder on the reference's ViT with the same seeded weights and input
    assert state_digest(v.state_dict()) == SURFACE["init"]["vit_hooks"]["digest"]
    with torch.no_grad():
        _, attns = Recorder(v)(SURFACE["hooks"]["img"])
    assert torch.allclose(SURFACE["hooks"]["attns"], attns, atol=1e-6)


def test_reference_accept_video_wrapper_runs_on_the_dropin():
    """AcceptVideoWrapper (reference accept_video_wrapper.py:70-76,108) reads `image_net.patch_size` and feeds the
    frames of a clip through `image_net.forward` as one batch: the drop-in with the reference's seeded weights gives
    the patch size and the per-frame outputs of the reference's own ViT."""
    ours = reference_init("vit_video", ViT).eval()
    g = SURFACE["video"]
    assert ours.patch_size == g["patch_size"] == (8, 8)
    with torch.no_grad():
        frames = ours(g["video"].permute(0, 2, 1, 3, 4).reshape(8, 3, 32, 32))
    assert torch.allclose(frames, g["frames"], rtol=1e-5, atol=1e-6)
