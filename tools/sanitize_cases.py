"""Small invocations of every kernel of libb200vit.so, for compute-sanitizer (tools/sanitize.sh).  Shapes are tiny but
cover: both GEMM kernels in every epilogue mode (incl. the 4-warp long-K epilogue and the head-norm epilogue), the
pipelined / round-1 / varlen attention kernels, the row kernels through three golden models, and a NaViT batch."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vit_pytorch_b200 import NaViT, SimpleViT, ViT, _lib  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
from golden_weights import load  # noqa: E402
which = set(sys.argv[1:]) or {"gemm", "attention", "models", "navit"}
torch.manual_seed(0)
dev = "cuda"
L = _lib.lib()

if "gemm" in which:
    for force, M, N, K in ((1, 200, 264, 128), (2, 512, 512, 128), (2, 300, 256, 2048)):
        L.b200vit_debug_set(4, force)
        a = torch.randn(M, K, device=dev).bfloat16(); w = torch.randn(N, K, device=dev).bfloat16()
        b = torch.randn(N, device=dev); x = torch.randn(M, N, device=dev)
        ob = torch.zeros(M, N, device=dev, dtype=torch.bfloat16)
        _lib.gemm(a, w, out_bf16=ob, bias=b, gelu=True)
        _lib.gemm(a, w, out_f32=x, bias=b, resid=x)
        if N % 64 == 0:
            st = torch.zeros(M, _lib.stats_parts(N), 2, device=dev)
            _lib.gemm(a, w, out_f32=x, out_bf16=ob, bias=b, resid=x, stats_out=st)
            sums = torch.zeros(M, 1, 2, device=dev); xb = torch.zeros(M, K, device=dev, dtype=torch.bfloat16)
            _lib.rowstats_cast(a.float(), xb, sums)
            _lib.gemm(xb, w, out_bf16=ob, bias=b, ln_sums=sums, col_s=w.float().sum(1).contiguous())
            _lib.gemm_headnorm(a, w, out_bf16=ob, head_gamma=torch.ones(128, device=dev), norm_heads=2)
    L.b200vit_debug_set(4, 0)
    print("gemm cases done")

if "attention" in which:
    for mode, (B, N, H) in ((2, (3, 197, 2)), (2, (160, 64, 2)), (1, (2, 197, 2)), (0, (1, 300, 1)), (0, (2, 50, 3))):
        L.b200vit_debug_set(1, mode)
        qkv = torch.randn(B * N, 3 * H * 64, device=dev).bfloat16()
        o = torch.zeros(B * N, H * 64, device=dev, dtype=torch.bfloat16)
        _lib.attention(qkv, o, B, N, H, 64, 0.125)
    L.b200vit_debug_set(1, 0)
    for dh, (B, N, H) in ((64, (3, 257, 2)), (80, (2, 258, 2)), (64, (150, 257, 2)), (80, (2, 197, 3))):
        # key tail (N = 257..260: 256-key score tile + the last keys from shared memory), both head widths
        qkv = torch.randn(B * N, 3 * H * dh, device=dev).bfloat16()
        o = torch.zeros(B * N, H * dh, device=dev, dtype=torch.bfloat16)
        _lib.attention(qkv, o, B, N, H, dh, dh ** -0.5)
    for mode in (0, 1, 2):
        L.b200vit_debug_set(11, mode)
        lengths = [197, 1, 130, 300, 64]
        T = sum(lengths)
        qkv = torch.randn(T, 3 * 2 * 64, device=dev).bfloat16()
        # keys growing along the sequence: the one-pass kernel (mode 0) moves its reference max and rescales O in TMEM
        qkv[:, 128:256] = (qkv[:, 128:256].float() * (1 + torch.arange(T, device=dev)[:, None] / 8.0)).bfloat16()
        qkv[:, :128] = (qkv[:, :128].float() * 4).bfloat16()
        o = torch.zeros(T, 2 * 64, device=dev, dtype=torch.bfloat16)
        cu, tp, tiles = _lib.varlen_index(lengths, dev)
        _lib.attention_varlen(qkv, o, cu, tp, tiles, 2, 64, 0.125)
    L.b200vit_debug_set(11, 0)
    print("attention cases done")

if "models" in which:
    for name in ("simplevit_tiny", "vit_tiny_cls", "vit_tiny_mean_nonsquare"):
        g = load(os.path.join(ROOT, "tests", "golden", name + ".pt"))
        m = (ViT if g["kind"] == "vit" else SimpleViT)(**g["kwargs"]).eval()
        m.load_state_dict(g["state_dict"])
        m = m.to(dev, torch.bfloat16)
        with torch.inference_mode():
            out = m(g["input"].to(dev))
        print(name, "max err", (out.float().cpu() - g["logits_fp32"]).abs().max().item())
    # 16x16x3 patches (patchify_ln16c3), N = 197 -> pipelined attention, CTA-pair GEMMs
    m = ViT(image_size=224, patch_size=16, num_classes=16, dim=256, depth=1, heads=4, mlp_dim=512).eval().to(dev, torch.bfloat16)
    with torch.inference_mode():
        out = m(torch.randn(6, 3, 224, 224, device=dev).bfloat16())
    print("vit 224/16 finite", bool(torch.isfinite(out.float()).all()))

if "navit" in which:
    g = torch.load(os.path.join(ROOT, "tests", "golden", "navit_tiny.pt"), weights_only=False)
    m = NaViT(**g["kwargs"]).eval()
    m.load_state_dict(g["state_dict"])
    m = m.to(dev, torch.bfloat16)
    with torch.inference_mode():
        out = m([im.to(dev) for im in g["images"]])
    print("navit_tiny max err", (out.float().cpu() - g["logits_fp32"]).abs().max().item())
    m = NaViT(image_size=256, patch_size=16, num_classes=10, dim=256, depth=1, heads=4, mlp_dim=512).eval().to(dev, torch.bfloat16)
    imgs = [torch.randn(3, h, w, device=dev).bfloat16() for h, w in ((256, 256), (16, 16), (64, 240), (128, 144))]
    with torch.inference_mode():
        out = m(imgs)
    print("navit 16x16 patches finite", bool(torch.isfinite(out.float()).all()))

torch.cuda.synchronize()
print("SANITIZE_CASES_DONE")
