"""-m gpu: the fused forward of the drop-in modules against (a) the committed reference goldens, (b) the oracle at
ViT-B/16 size, (c) size-independent properties at BASELINE.json's full batch."""
import pytest
import torch

from conftest import load_golden
from oracle import vit_oracle as O
from vit_pytorch_b200 import SimpleViT, ViT, _lib

pytestmark = pytest.mark.gpu
DEV = "cuda"

# north_star tolerance for bf16: rtol=1e-2 / atol=1e-3 against the reference forward
RTOL, ATOL = 1e-2, 1e-3


def fused_model(g):
    cls = ViT if g["kind"] == "vit" else SimpleViT
    m = cls(**g["kwargs"]).eval()
    m.load_state_dict(g["state_dict"])
    return m.to(DEV, torch.bfloat16)


def stats(got, ref):
    d = (got.float().cpu() - ref).abs()
    return d.max().item(), d.mean().item(), (d <= ATOL + RTOL * ref.abs()).float().mean().item()


def test_fused_path_is_selected_and_counts_launches(golden):
    m = fused_model(golden)
    img = golden["input"].to(DEV)
    _lib.reset_launch_count()
    with torch.inference_mode():
        assert m.fused_reason(img) is None
        m(img)
    torch.cuda.synchronize()
    depth = golden["kwargs"]["depth"]
    assert _lib.launch_count() >= 3 + 5 * depth + 1        # 7 per layer with LayerNorm kernels, 5 when folded


def test_config1_simplevit_tiny_allclose():
    """BASELINE.json configs[0]: strict allclose against the reference's fp32 logits."""
    g = load_golden("simplevit_tiny")
    m = fused_model(g)
    with torch.inference_mode():
        out = m(g["input"].to(DEV))
    assert out.dtype == torch.bfloat16 and out.shape == g["logits_fp32"].shape
    assert torch.allclose(out.float().cpu(), g["logits_fp32"], rtol=RTOL, atol=ATOL), stats(out, g["logits_fp32"])


def test_goldens_no_worse_than_reference_bf16(golden):
    """Every golden case, error measured against the reference's fp32 logits: at least as many outputs inside
    rtol=1e-2/atol=1e-3 as the reference's OWN bf16 forward achieves on the same inputs (capped at 99 %), and a
    maximum error not above 1.25x the reference-bf16 maximum."""
    m = fused_model(golden)
    with torch.inference_mode():
        out = m(golden["input"].to(DEV))
    ref = golden["logits_fp32"]
    mx, mean, frac = stats(out, ref)
    ref_d = (golden["logits_ref_bf16"] - ref).abs()
    ref_mx = ref_d.max().item()
    ref_frac = (ref_d <= ATOL + RTOL * ref.abs()).float().mean().item()
    print(f"{golden['name']}: ours max {mx:.5f} mean {mean:.5f} within {frac:.4f} | reference-bf16 max {ref_mx:.5f} "
          f"within {ref_frac:.4f}")
    assert frac >= min(0.99, ref_frac), (mx, mean, frac, ref_frac)
    assert mx <= max(1.25 * ref_mx, 2 * ATOL), (mx, ref_mx)


@pytest.mark.parametrize("mode", ["fold", "exact"])
def test_both_layernorm_modes_against_golden(mode, monkeypatch):
    """LN folded into the GEMM epilogues (default) and the literal LayerNorm-kernel schedule both meet the bar."""
    monkeypatch.setenv("B200VIT_LN_MODE", mode)
    for name in ("simplevit_tiny", "vit_tiny_cls"):
        g = load_golden(name)
        m = fused_model(g)
        with torch.inference_mode():
            out = m(g["input"].to(DEV))
        ref = g["logits_fp32"]
        mx, mean, frac = stats(out, ref)
        ref_d = (g["logits_ref_bf16"] - ref).abs()
        print(f"{name} [{mode}]: max {mx:.5f} mean {mean:.5f} within {frac:.4f}")
        assert mx <= max(1.25 * ref_d.max().item(), 2 * ATOL)


def test_transformer_on_arbitrary_tokens_fused():
    """Transformer called directly on a token subset (MAE / SimMIM usage, reference mae.py:74)."""
    g = load_golden("vit_tiny_cls")
    m = fused_model(g)
    sd = O.upcast(g["state_dict"])
    torch.manual_seed(5)
    tok = torch.randn(3, 23, 192).bfloat16()
    with torch.inference_mode():
        assert m.transformer.fused_reason(tok.to(DEV)) is None
        out = m.transformer(tok.to(DEV))
    ref = O.transformer(sd, tok.float(), 2, 3, "vit")
    assert stats(out, ref)[2] > 0.98


def test_fused_equals_own_eager_graph_closely():
    g = load_golden("vit_tiny_cls")
    m = fused_model(g)
    img = g["input"].to(DEV)
    with torch.inference_mode():
        a = m.forward_fused(img).float()
        b = m.forward_eager(img).float()
    assert (a - b).abs().max() < 3e-2       # eager bf16 graph is the noisier of the two


@pytest.mark.parametrize("kind", ["vit", "simple"])
def test_vit_b16_against_oracle(kind):
    """BASELINE.json configs[1] geometry at B=2 (the oracle finishes in seconds): error vs the fp32 oracle must be
    below the reference's own bf16 noise floor measured in BASELINE.md section 6 (max 0.0211 / 64.6 % within tol for
    ViT-B/16; 0.0046 / 92.8 % for SimpleViT-B/16)."""
    kwargs = dict(image_size=224, patch_size=16, num_classes=1000, dim=768, depth=12, heads=12, mlp_dim=3072)
    torch.manual_seed(0)
    m = (ViT if kind == "vit" else SimpleViT)(**kwargs).eval().bfloat16()
    torch.manual_seed(1)
    img = torch.randn(2, 3, 224, 224).bfloat16()
    ref = O.forward(kind, O.upcast(m.state_dict()), kwargs, img.float())
    m = m.to(DEV)
    with torch.inference_mode():
        out = m(img.to(DEV))
    mx, mean, frac = stats(out, ref)
    from vit_pytorch_b200.engine import ln_mode
    print(f"{kind}-B/16 [{ln_mode()}] vs fp32 oracle: max {mx:.5f} mean {mean:.5f} within_tol {frac:.4f}")
    assert mx < 0.0211 and frac > (0.90 if kind == "vit" else 0.928), (mx, mean, frac)


@pytest.mark.parametrize("name,kwargs,floor_max,floor_frac", [
    # BASELINE.json configs[2] / configs[3] geometry (dim_head = reference default 64); the floors are the reference's
    # own bf16 forward against its fp32 forward, BASELINE.md section 6
    ("ViT-L/16", dict(image_size=224, patch_size=16, num_classes=1000, dim=1024, depth=24, heads=16, mlp_dim=4096),
     0.0249, 0.525),
    ("ViT-H/14", dict(image_size=224, patch_size=14, num_classes=1000, dim=1280, depth=32, heads=16, mlp_dim=5120),
     0.0257, 0.478),
    # the canonical ViT-H/14 head width: dim_head = 80 (SURVEY.md 8d config 4 "run with dim_head=64 and 80")
    ("ViT-H/14 dim_head 80", dict(image_size=224, patch_size=14, num_classes=1000, dim=1280, depth=32, heads=16,
                                  mlp_dim=5120, dim_head=80), 0.0298, 0.478),
])
def test_large_configs_against_oracle(name, kwargs, floor_max, floor_frac):
    torch.manual_seed(0)
    m = ViT(**kwargs).eval().bfloat16()
    torch.manual_seed(1)
    img = torch.randn(2, 3, 224, 224).bfloat16()
    ref = O.vit_forward(O.upcast(m.state_dict()), kwargs, img.float())
    m = m.to(DEV)
    with torch.inference_mode():
        assert m.fused_reason(img.to(DEV)) is None
        out = m(img.to(DEV))
    mx, mean, frac = stats(out, ref)
    print(f"{name} vs fp32 oracle: max {mx:.5f} mean {mean:.5f} within_tol {frac:.4f} "
          f"(reference-bf16 floor: max {floor_max}, within {floor_frac})")
    assert mx < floor_max and frac > floor_frac, (mx, mean, frac)


def test_long_sequence_uses_key_block_attention():
    """384x384 input (N = 577 > 512): the encoder switches to the key-block (varlen) attention kernel."""
    kwargs = dict(image_size=384, patch_size=16, num_classes=10, dim=256, depth=2, heads=4, mlp_dim=512)
    torch.manual_seed(0)
    m = ViT(**kwargs).eval().bfloat16()
    torch.manual_seed(1)
    img = torch.randn(2, 3, 384, 384).bfloat16()
    ref = O.vit_forward(O.upcast(m.state_dict()), kwargs, img.float())
    m = m.to(DEV)
    with torch.inference_mode():
        assert m.fused_reason(img.to(DEV)) is None
        out = m(img.to(DEV))
    mx, mean, frac = stats(out, ref)
    print(f"ViT 384^2 (N=577) vs fp32 oracle: max {mx:.5f} mean {mean:.5f} within_tol {frac:.4f}")
    assert mx < 2e-2 and frac > 0.85


@pytest.mark.parametrize("mode", ["exact", "fold"])
def test_full_batch_properties_b512(mode, monkeypatch):
    monkeypatch.setenv("B200VIT_LN_MODE", mode)
    _full_batch_properties_b512()


def _full_batch_properties_b512():
    """BASELINE.json configs[1] at its full batch (512): properties that need no oracle run --
    (1) batch-permutation equivariance, bit exact (every image is computed independently of its batch slot);
    (2) batch-size invariance: image i gives the same logits in a batch of 512 and in a batch of 2;
    (3) outputs finite."""
    kwargs = dict(image_size=224, patch_size=16, num_classes=1000, dim=768, depth=12, heads=12, mlp_dim=3072)
    torch.manual_seed(0)
    m = ViT(**kwargs).eval().to(DEV, torch.bfloat16)
    torch.manual_seed(1)
    img = torch.randn(512, 3, 224, 224, device=DEV).bfloat16()
    with torch.inference_mode():
        out = m(img)
        perm = torch.randperm(512, device=DEV)
        out_p = m(img[perm])
        out_2 = m(img[:2].contiguous())
    assert out.shape == (512, 1000) and torch.isfinite(out.float()).all()
    assert torch.equal(out[perm], out_p)
    assert torch.equal(out[:2], out_2)


def test_missing_library_raises_on_eligible_input(monkeypatch, tmp_path):
    g = load_golden("simplevit_tiny")
    m = fused_model(g)
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", tmp_path / "missing.so")
    with pytest.raises(_lib.B200VitError):
        with torch.inference_mode():
            m(g["input"].to(DEV))


def test_cuda_graph_replay_is_bit_identical():
    """vit_pytorch_b200.graph.GraphedForward: every library launch lands in the capture stream; replays on new inputs
    reproduce the call-by-call fused forward bit for bit."""
    from vit_pytorch_b200.graph import GraphedForward
    torch.manual_seed(0)
    m = ViT(image_size=64, patch_size=16, num_classes=10, dim=128, depth=2, heads=2, mlp_dim=256).eval()
    m = m.to(DEV, torch.bfloat16)
    a = torch.randn(4, 3, 64, 64, device=DEV).bfloat16()
    b = torch.randn(4, 3, 64, 64, device=DEV).bfloat16()
    with torch.inference_mode():
        ya, yb = m(a).clone(), m(b).clone()
        g = GraphedForward(m, a)
        assert torch.equal(g(b), yb)
        assert torch.equal(g(a), ya)
    with pytest.raises(ValueError):
        g(a[:2])


@pytest.mark.parametrize("kind", ["vit_cls", "vit_mean", "simple"])
def test_extractor_hook_keeps_the_fused_path(kind):
    """Extractor (reference extractor.py:50-59) hooks `vit.transformer`: the fused forward routes the tokens through
    that module call, so the hook sees the encoder output while every block still runs in the sm_100a kernels."""
    from vit_pytorch_b200.extractor import Extractor
    torch.manual_seed(0)
    kw = dict(image_size=64, patch_size=8, num_classes=10, dim=128, depth=2, heads=2, mlp_dim=256)
    m = (SimpleViT(**kw) if kind == "simple" else ViT(pool="mean" if kind == "vit_mean" else "cls", **kw)).eval()
    m = m.to(DEV, torch.bfloat16)
    img = torch.randn(3, 3, 64, 64, device=DEV).bfloat16()
    with torch.inference_mode():
        plain = m(img)
        ext = Extractor(m)
        assert m.fused_reason(img) is None
        _lib.reset_launch_count()
        pred, emb = ext(img)
        assert _lib.launch_count() >= 3 + 5 * 2
        n = 64 + (1 if kind == "vit_cls" else 0)         # pool="mean" has no cls token (vit.py:105-106)
        assert emb.shape == (3, n, 128) and emb.dtype == torch.bfloat16
        assert (pred.float() - plain.float()).abs().max() < 2e-2          # tokens passed through bf16 once
        ext.eject()
        ref_emb = {}
        h = m.transformer.register_forward_hook(lambda _m, _i, o: ref_emb.setdefault("o", o))
        m.float().forward_eager(img.float())
        h.remove()
    assert (emb.float() - ref_emb["o"]).abs().max() < 6e-2 and (emb.float() - ref_emb["o"]).abs().mean() < 6e-3


def test_hook_inside_the_transformer_still_forces_the_pytorch_graph():
    from vit_pytorch_b200.recorder import Recorder
    torch.manual_seed(0)
    m = ViT(image_size=32, patch_size=8, num_classes=4, dim=128, depth=2, heads=2, mlp_dim=256).eval()
    m = m.to(DEV, torch.bfloat16)
    img = torch.randn(2, 3, 32, 32, device=DEV).bfloat16()
    rec = Recorder(m)
    with torch.inference_mode():
        _lib.reset_launch_count()
        pred, attns = rec(img)
        assert _lib.launch_count() == 0 and "hooks" in m.fused_reason(img)
        assert attns.shape == (2, 2, 2, 17, 17)
        rec.eject()
        assert m.fused_reason(img) is None
        assert (m(img).float() - pred.float()).abs().max() < 3e-2


@pytest.mark.parametrize("case", ["vit_golden", "qk_norm", "long_sequence", "dh80"])
def test_one_call_encoder_equals_the_per_kernel_host_loop(case, monkeypatch):
    """b200vit_encoder_blocks (all layers in one C-ABI call, the default) launches exactly the kernels the Python loop
    launches, with the same arguments: bit-identical logits and the same launch count."""
    torch.manual_seed(0)
    if case == "vit_golden":
        g = load_golden("vit_tiny_cls")
        m = fused_model(g)
        x = g["input"].to(DEV)
    elif case == "qk_norm":
        from vit_pytorch_b200.simple_vit_with_qk_norm import SimpleViT as QK
        m = QK(image_size=64, patch_size=8, num_classes=7, dim=128, depth=2, heads=2, mlp_dim=256).eval()
        m = m.to(DEV, torch.bfloat16)
        x = torch.randn(3, 3, 64, 64, device=DEV).bfloat16()
    elif case == "long_sequence":
        m = ViT(image_size=224, patch_size=8, num_classes=5, dim=128, depth=2, heads=2, mlp_dim=256).eval()
        m = m.to(DEV, torch.bfloat16)                     # N = 785 > 512: key-block attention inside the C loop
        x = torch.randn(2, 3, 224, 224, device=DEV).bfloat16()
    else:
        m = ViT(image_size=56, patch_size=14, num_classes=5, dim=160, depth=2, heads=2, dim_head=80, mlp_dim=320).eval()
        m = m.to(DEV, torch.bfloat16)
        x = torch.randn(4, 3, 56, 56, device=DEV).bfloat16()
    outs, counts = {}, {}
    for loop in ("c", "python"):
        monkeypatch.setenv("B200VIT_HOST_LOOP", loop)
        _lib.reset_launch_count()
        with torch.inference_mode():
            assert m.fused_reason(x) is None, m.fused_reason(x)
            outs[loop] = m(x).clone()
        torch.cuda.synchronize()
        counts[loop] = _lib.launch_count()
    assert torch.equal(outs["c"], outs["python"])
    assert counts["c"] == counts["python"] > 0


@pytest.mark.parametrize("mode", ["fold", "exact"])
def test_trained_like_statistics_stay_below_the_bf16_floor(mode, monkeypatch):
    """Random-init weights are benign; trained ViTs are not: a few residual channels carry massive activations, the
    residual stream has a common offset (row mean several sigma away from zero -- the case where normalising an
    already bf16-rounded row, as the LN-fold path AND the reference's bf16 module do, loses digits), LayerNorm gains
    are spread out and attention is peaky.  Expectation: the module's own fp32 PyTorch graph (equal to the reference,
    tests/test_dropin.py); pass criterion: no worse than the same graph in bf16 (= the reference's bf16 forward)."""
    monkeypatch.setenv("B200VIT_LN_MODE", mode)
    torch.manual_seed(0)
    kw = dict(image_size=224, patch_size=16, num_classes=100, dim=384, depth=6, heads=6, mlp_dim=1536)
    m = ViT(**kw).eval()
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        for name, p in m.named_parameters():
            if p.dim() == 1 and name.endswith("weight"):                        # LayerNorm gains: 0.4 .. 2.5
                p.copy_(torch.exp(0.45 * torch.randn(p.shape, generator=g)))
            elif p.dim() == 1 and "norm" in name and name.endswith("bias"):
                p.copy_(0.3 * torch.randn(p.shape, generator=g))
        for i, (attn, ff) in enumerate(m.transformer.layers):
            attn.to_qkv.weight[: 2 * 384] *= 2.5                                 # q, k: peaky softmax
            fc2 = ff.net[4] if hasattr(ff, "net") else None
            if i < 2:
                for c in (7, 100, 250):                                          # massive-activation channels
                    fc2.weight[c] *= 20.0
                    fc2.bias[c] += 8.0
                fc2.bias += 1.5                                                  # common offset of the whole stream
        for p in m.parameters():
            p.copy_(p.bfloat16().float())
    img = torch.randn(4, 3, 224, 224, generator=g).bfloat16()
    m = m.to(DEV)
    with torch.inference_mode():
        ref = m.forward_eager(img.to(DEV).float()).float().cpu()
        # how hostile the stream is: row mean / row std of the residual stream entering the last layer
        x = m.to_patch_embedding(img.to(DEV).float())
        x = torch.cat((m.cls_token.unsqueeze(0).expand(4, -1, -1), x), dim=1) + m.pos_embedding[:197]
        for attn, ff in list(m.transformer.layers)[:-1]:
            x = attn(x) + x
            x = ff(x) + x
        ratio = (x.mean(-1).abs() / x.std(-1)).mean().item()
        peak = x.abs().max().item()
        mb = m.bfloat16()
        floor = mb.forward_eager(img.to(DEV)).float().cpu()
        assert mb.fused_reason(img.to(DEV)) is None
        out = mb(img.to(DEV)).float().cpu()
    d, f = (out - ref).abs(), (floor - ref).abs()
    print(f"trained-like [{mode}]: |row mean| / row std {ratio:.2f}, max |x| {peak:.0f}, logits |max| {ref.abs().max():.2f}; "
          f"fused max {d.max():.4f} mean {d.mean():.5f}; bf16 graph max {f.max():.4f} mean {f.mean():.5f}")
    assert torch.isfinite(out).all()
    assert d.mean() <= f.mean() * 1.05 + 1e-4 and d.max() <= f.max() * 1.5 + 1e-3


def test_reference_distill_wrapper_runs_its_teacher_on_the_fused_path():
    """DistillWrapper (reference distill.py:139-141) calls `teacher(img)` under no_grad: with the drop-in as the
    teacher (cuda, bf16, frozen) that call is the fused sm_100a forward, and it returns the reference's teacher logits
    (fp32, stored) no less accurately than the reference's own bf16 teacher does."""
    from conftest import reference_init
    teacher = reference_init("distill_gpu", ViT).eval().to(DEV, torch.bfloat16)
    for p in teacher.parameters():
        p.requires_grad_(False)
    g = load_golden("reference_surface")["distill_gpu"]
    img = g["img"].to(DEV)
    _lib.reset_launch_count()
    with torch.no_grad():
        logits = teacher(img)
    assert _lib.launch_count() >= 3 + 5 * 2                      # the teacher forward ran in the library's kernels
    ref = g["logits_fp32"]
    d, f = (logits.float().cpu() - ref).abs(), (g["logits_ref_bf16"] - ref).abs()
    print(f"distill teacher: fused max {d.max():.5f} mean {d.mean():.5f}; reference-bf16 max {f.max():.5f} "
          f"mean {f.mean():.5f}")
    assert torch.isfinite(logits).all() and d.max() <= f.max() * 1.5 + 1e-3
