"""Generate golden fixtures from the UNMODIFIED reference (lucidrains/vit-pytorch at /root/reference).

Run in the build container only (the GPU box has no /root/reference):

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py

For each case: build the reference model under torch.manual_seed(seed), round its parameters to bf16-representable
values (so the same numbers can be fed to the bf16 CUDA path), run the reference forward in fp32 on CPU on a
bf16-representable input, and additionally run the reference's own bf16 forward (its noise floor).  Saved per case
(tests/golden/<name>.pt): kind, ctor kwargs, seed and the sha256 digest of the bf16 state_dict (golden_weights.py
rebuilds the weights from the seed), input (bf16), logits_fp32, logits_ref_bf16, tokens_fp32 (transformer output for
the first sample) and the library versions.
"""
from __future__ import annotations

import os
import sys

import torch

REF = os.environ.get("VIT_REFERENCE", "/root/reference")
sys.path.insert(0, REF)
sys.dont_write_bytecode = True

from vit_pytorch import ViT, SimpleViT  # noqa: E402  (the reference)

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

from golden_weights import golden_model, state_digest  # noqa: E402  (tests/golden/)

CASES = {
    # BASELINE.json configs[0]: SimpleViT tiny (num_classes / mlp_dim chosen in SURVEY.md 8d)
    "simplevit_tiny": dict(kind="simple", seed=0, batch=4, img=(32, 32),
                           kwargs=dict(image_size=32, patch_size=4, num_classes=10, dim=192, depth=2, heads=3,
                                       mlp_dim=768)),
    # ViT, cls pooling, with biases everywhere, same tiny geometry
    "vit_tiny_cls": dict(kind="vit", seed=1, batch=3, img=(32, 32),
                         kwargs=dict(image_size=32, patch_size=4, num_classes=10, dim=192, depth=2, heads=3,
                                     mlp_dim=768)),
    # ViT, mean pooling, tuple sizes, smaller non-square input than image_size (README.md:1720-1766), N = 8 tokens
    "vit_tiny_mean_nonsquare": dict(kind="vit", seed=2, batch=2, img=(32, 16),
                                    kwargs=dict(image_size=(32, 32), patch_size=(8, 4), num_classes=24, dim=128,
                                                depth=3, heads=2, mlp_dim=256, pool="mean")),
    # ViT without head: returns tokens (vit.py:132-133)
    "vit_tiny_tokens": dict(kind="vit", seed=3, batch=2, img=(32, 32),
                            kwargs=dict(image_size=32, patch_size=8, num_classes=0, dim=128, depth=1, heads=2,
                                        mlp_dim=256)),
}

# Round 2: attention without output projection (vit.py:34,46-49) and the SURVEY.md 8(f3) SimpleViT-family variants.
# `kind` = module name inside the reference package for the variants.
CASES2 = {
    "vit_tiny_noproj": dict(kind="vit", seed=4, batch=3, img=(32, 32),
                            kwargs=dict(image_size=32, patch_size=8, num_classes=7, dim=64, depth=2, heads=1,
                                        dim_head=64, mlp_dim=128)),
    "simplevit_registers": dict(kind="simple_vit_with_register_tokens", seed=6, batch=3, img=(32, 32),
                                kwargs=dict(image_size=32, patch_size=4, num_classes=10, dim=128, depth=2, heads=2,
                                            mlp_dim=256, num_register_tokens=4)),
    "simplevit_qknorm": dict(kind="simple_vit_with_qk_norm", seed=7, batch=3, img=(32, 32),
                             kwargs=dict(image_size=32, patch_size=4, num_classes=10, dim=128, depth=2, heads=2,
                                         mlp_dim=256)),
    "simplevit_patchdrop": dict(kind="simple_vit_with_patch_dropout", seed=8, batch=3, img=(32, 48),
                                kwargs=dict(image_size=64, patch_size=8, num_classes=10, dim=128, depth=2, heads=2,
                                            mlp_dim=256, patch_dropout=0.5)),
    "simplevit_flash": dict(kind="simple_flash_attn_vit", seed=9, batch=3, img=(48, 32),
                            kwargs=dict(image_size=64, patch_size=8, num_classes=10, dim=128, depth=2, heads=2,
                                        mlp_dim=256, use_flash=True)),
}


# Round 2, later: the 1-D / 3-D front-ends of SURVEY.md 8(f3) (series and video inputs; `img` = the non-channel dims)
CASES3 = {
    "simplevit_1d": dict(kind="simple_vit_1d", seed=12, batch=3, img=(256,),
                         kwargs=dict(seq_len=256, patch_size=16, num_classes=10, dim=128, depth=2, heads=2,
                                     mlp_dim=256)),
    "simplevit_3d": dict(kind="simple_vit_3d", seed=13, batch=2, img=(4, 32, 24),
                         kwargs=dict(image_size=(32, 24), image_patch_size=8, frames=4, frame_patch_size=2,
                                     num_classes=10, dim=128, depth=2, heads=2, mlp_dim=256)),
    "simplevit_3d_pf1": dict(kind="simple_vit_3d", seed=14, batch=2, img=(3, 32, 48),
                             kwargs=dict(image_size=(32, 48), image_patch_size=16, frames=3, frame_patch_size=1,
                                         num_classes=10, dim=192, depth=2, heads=3, mlp_dim=384)),
}


def reference_class(kind: str):
    """kind -> class of the UNMODIFIED reference."""
    import importlib
    if kind in ("vit", "simple"):
        return ViT if kind == "vit" else SimpleViT
    return importlib.import_module("vit_pytorch." + kind).SimpleViT


def make(name: str, spec: dict) -> None:
    cls = reference_class(spec["kind"])
    model = golden_model(cls, spec["kwargs"], spec["seed"])
    torch.manual_seed(100 + spec["seed"])
    img = torch.randn(spec["batch"], 3, *spec["img"]).bfloat16()
    with torch.inference_mode():
        logits = model(img.float())
        tokens = None
        if spec["kind"] == "vit":
            x = model.to_patch_embedding(img.float()[:1])
            x = torch.cat((model.cls_token[None], x), dim=1)
            x = x + model.pos_embedding[: x.shape[1]]
            tokens = model.transformer(x)
        model_bf16 = cls(**spec["kwargs"]).eval()
        model_bf16.load_state_dict(model.state_dict())
        model_bf16 = model_bf16.bfloat16()
        logits_bf16 = model_bf16(img)
    blob = {
        "name": name,
        "kind": spec["kind"],
        "kwargs": spec["kwargs"],
        "seed": spec["seed"],
        "state_digest": state_digest({k: v.bfloat16() for k, v in model.state_dict().items()}),
        "input": img,
        "logits_fp32": logits.clone(),
        "logits_ref_bf16": logits_bf16.float().clone(),
        "tokens_fp32": None if tokens is None else tokens.clone(),
        "versions": {"torch": str(torch.__version__), "reference": "vit-pytorch 1.23.6 @ /root/reference"},
    }
    path = os.path.join(HERE, name + ".pt")
    torch.save(blob, path)
    print(f"{name}: logits {tuple(logits.shape)} |max| {logits.abs().max():.4f}; "
          f"ref-bf16 max err {(logits_bf16.float() - logits).abs().max():.5f}; {os.path.getsize(path) / 1e6:.2f} MB")


def make_navit() -> None:
    """NaViT (reference na_vit.py): 7 images of 5 different resolutions, given as two pre-packed rows AND re-packed by
    the reference's own greedy grouping; fp32 logits of both calls are stored."""
    from vit_pytorch.na_vit import NaViT
    kwargs = dict(image_size=64, patch_size=8, num_classes=11, dim=128, depth=2, heads=2, mlp_dim=192, dim_head=64)
    torch.manual_seed(5)
    model = NaViT(**kwargs).eval()
    g = torch.Generator().manual_seed(1005)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if n.endswith("gamma"):
                p.add_(0.1 * torch.randn(p.shape, generator=g))
            p.copy_(p.bfloat16().float())
    torch.manual_seed(105)
    sizes = [(64, 64), (32, 48), (16, 16), (64, 32), (24, 40), (8, 64), (48, 48)]
    imgs = [torch.randn(3, h, w).bfloat16() for h, w in sizes]
    rows = [[0, 1, 2], [3, 4, 5, 6]]
    with torch.inference_mode():
        packed = model([[imgs[i].float() for i in r] for r in rows])
        grouped = model([im.float() for im in imgs], group_images=True, group_max_seq_len=80)
    blob = {"name": "navit_tiny", "kind": "navit", "kwargs": kwargs,
            "state_dict": {k: v.bfloat16() for k, v in model.state_dict().items()},
            "images": imgs, "rows": rows, "group_max_seq_len": 80,
            "logits_fp32": packed.clone(), "logits_grouped_fp32": grouped.clone(),
            "versions": {"torch": str(torch.__version__), "reference": "vit-pytorch 1.23.6 @ /root/reference"}}
    path = os.path.join(HERE, "navit_tiny.pt")
    torch.save(blob, path)
    print(f"navit_tiny: logits {tuple(packed.shape)} |max| {packed.abs().max():.4f}; packed vs grouped "
          f"{(packed - grouped).abs().max():.2e}; {os.path.getsize(path) / 1e6:.2f} MB")


from navit_c5_spec import NAVIT_C5, navit_config5_images, navit_config5_model  # noqa: E402  (tests/golden/)


def make_navit_config5() -> None:
    from vit_pytorch.na_vit import NaViT
    model = navit_config5_model(NaViT)
    imgs = navit_config5_images()
    with torch.inference_mode():
        fp32 = model([im.float() for im in imgs], group_images=True, group_max_seq_len=4096)
        bf16 = model.bfloat16()([im for im in imgs], group_images=True, group_max_seq_len=4096)
    d = (bf16.float() - fp32).abs()
    floor = {"max": d.max().item(), "mean": d.mean().item(),
             "frac_within_tol": (d <= 1e-3 + 1e-2 * fp32.abs()).float().mean().item()}
    blob = {"name": "navit_config5", "kind": "navit", "spec": NAVIT_C5, "logits_fp32": fp32.clone(),
            "logits_ref_bf16": bf16.clone(), "ref_bf16_floor": floor,
            "versions": {"torch": str(torch.__version__), "reference": "vit-pytorch 1.23.6 @ /root/reference"}}
    path = os.path.join(HERE, "navit_config5.pt")
    torch.save(blob, path)
    print(f"navit_config5: logits {tuple(fp32.shape)} |max| {fp32.abs().max():.4f}; reference-bf16 floor {floor}; "
          f"{os.path.getsize(path) / 1e6:.2f} MB")


def make_navit_nested() -> None:
    """Nested-tensor NaViT (reference na_vit_nested_tensor.py): 6 images of 5 resolutions, with and without the q / k
    LayerNorm.  The reference runs its jagged-batch forward (torch.nested + SDPA) on CPU."""
    from vit_pytorch.na_vit_nested_tensor import NaViT
    for name, qk in (("navit_nested_tiny", True), ("navit_nested_noqknorm", False)):
        kwargs = dict(image_size=64, patch_size=8, num_classes=11, dim=128, depth=2, heads=2, mlp_dim=192, dim_head=64,
                      qk_rmsnorm=qk)
        torch.manual_seed(11)
        model = NaViT(**kwargs).eval()
        g = torch.Generator().manual_seed(1011)
        with torch.no_grad():
            for n, p in model.named_parameters():
                if p.dim() == 1 and n.endswith("weight"):               # every LayerNorm scale (incl. the per-head ones)
                    p.add_(0.1 * torch.randn(p.shape, generator=g))
                elif p.dim() == 1 and n.endswith("bias"):
                    p.add_(0.05 * torch.randn(p.shape, generator=g))
                p.copy_(p.bfloat16().float())
        torch.manual_seed(111)
        sizes = [(64, 64), (32, 48), (8, 8), (64, 16), (24, 40), (48, 48)]
        imgs = [torch.randn(3, h, w).bfloat16() for h, w in sizes]
        with torch.inference_mode():
            fp32 = model([im.float() for im in imgs])
            bf16 = model.bfloat16()([im for im in imgs])
        blob = {"name": name, "kind": "navit_nested", "kwargs": kwargs,
                "state_dict": {k: v.bfloat16() for k, v in model.state_dict().items()}, "images": imgs,
                "logits_fp32": fp32.clone(), "logits_ref_bf16": bf16.float().clone(),
                "versions": {"torch": str(torch.__version__), "reference": "vit-pytorch 1.23.6 @ /root/reference"}}
        path = os.path.join(HERE, name + ".pt")
        torch.save(blob, path)
        print(f"{name}: logits {tuple(fp32.shape)} |max| {fp32.abs().max():.4f}; ref-bf16 max err "
              f"{(bf16.float() - fp32).abs().max():.5f}; {os.path.getsize(path) / 1e6:.2f} MB")


def _signature(cls) -> list:
    import inspect
    return [(n, p.default) for n, p in inspect.signature(cls.__init__).parameters.items() if n != "self"]


def make_reference_surface() -> None:
    """reference_surface.pt: what the tests used to ask the reference package itself -- constructor signatures, the
    parameters its constructors draw under a seed (sha256 per tensor, golden_weights.state_digest), its fp32
    outputs on seeded models, and the values its wrappers (Extractor, Recorder, MAE, DistillWrapper,
    AcceptVideoWrapper) read from or compute with a ViT."""
    import importlib
    from vit_pytorch.na_vit import NaViT as RefNaViT
    from vit_pytorch.na_vit_nested_tensor import NaViT as RefNestedNaViT
    from vit_pytorch.recorder import Recorder
    from vit_pytorch.extractor import Extractor
    blob = {"init": {}, "signatures": {}, "oracle": {}}

    def init(name, cls, seed, kwargs, buffers=()):
        torch.manual_seed(seed)
        m = cls(**kwargs)
        blob["init"][name] = {"seed": seed, "kwargs": kwargs, "digest": state_digest(m.state_dict()),
                              "buffers": state_digest({b: getattr(m, b) for b in buffers})}
        return m

    small = dict(image_size=32, patch_size=8, num_classes=5, dim=64, depth=2, heads=2, mlp_dim=96, dim_head=32)
    init("vit", ViT, 123, small)
    init("simple", SimpleViT, 123, small, buffers=("pos_embedding",))
    for name, spec in {**CASES2, **CASES3}.items():
        if spec["kind"] != "vit":
            init(name, reference_class(spec["kind"]), 123, spec["kwargs"])
            blob["signatures"][spec["kind"]] = _signature(reference_class(spec["kind"]))
    init("navit_nested", RefNestedNaViT, 5,
         dict(image_size=32, patch_size=8, num_classes=5, dim=64, depth=1, heads=1, mlp_dim=64))
    blob["signatures"]["na_vit_nested_tensor"] = _signature(RefNestedNaViT)

    # tests/test_oracle.py: seeded reference models and inputs, fp32 logits
    live = {"vit_11": ("vit", 11), "simple_12": ("simple", 12), "vit_13": ("vit", 13)}
    for name, (kind, seed) in live.items():
        kwargs = dict(image_size=64, patch_size=16, num_classes=17, dim=128, depth=2, heads=2, mlp_dim=192)
        if seed == 13:
            kwargs["pool"] = "mean"
        model = init(name, ViT if kind == "vit" else SimpleViT, seed, kwargs).eval()
        img = torch.randn(3, 3, 64, 64)
        with torch.inference_mode():
            blob["oracle"][name] = {"kind": kind, "input": state_digest({"img": img})["img"], "logits": model(img)}
    vit_b16 = dict(image_size=224, patch_size=16, num_classes=1000, dim=768, depth=12, heads=12, mlp_dim=3072)
    model = init("vit_b16", ViT, 0, vit_b16).eval()
    torch.manual_seed(1)
    img = torch.randn(1, 3, 224, 224)
    with torch.inference_mode():
        blob["oracle"]["vit_b16"] = {"kind": "vit", "input": state_digest({"img": img})["img"], "logits": model(img)}

    # tests/test_navit.py: packed NaViT forward on three images
    kwargs = dict(image_size=32, patch_size=8, num_classes=5, dim=64, depth=1, heads=2, mlp_dim=96, dim_head=32)
    model = init("navit", RefNaViT, 9, kwargs).eval()
    imgs = [torch.randn(3, 32, 16), torch.randn(3, 8, 8), torch.randn(3, 24, 32)]
    with torch.inference_mode():
        blob["navit"] = {"images": imgs, "logits": model([imgs[:2], imgs[2:]])}

    # Extractor / Recorder (tests/test_dropin.py): embeddings and attention maps of a seeded ViT
    kwargs = dict(image_size=32, patch_size=8, num_classes=3, dim=32, depth=2, heads=2, mlp_dim=48, dim_head=16)
    v = init("vit_hooks", ViT, 0, kwargs).eval()
    img = torch.randn(2, 3, 32, 32)
    with torch.no_grad():
        logits, emb = Extractor(v)(img)
        _, attns = Recorder(v)(img)
    blob["hooks"] = {"img": img, "logits": logits, "embeddings": emb, "attns": attns}

    # MAE: the encoder members it reads and the encoder call on the unmasked quarter of the tokens
    kwargs = dict(image_size=32, patch_size=8, num_classes=5, dim=64, depth=2, heads=2, mlp_dim=96, pool="mean")
    enc = init("vit_mae", ViT, 0, kwargs).eval()
    img = torch.randn(3, 3, 32, 32)
    with torch.no_grad():
        patches = enc.to_patch_embedding[0](img)
        tokens = torch.nn.Sequential(*enc.to_patch_embedding[1:])(patches) + enc.pos_embedding
        torch.manual_seed(2)
        keep = torch.rand(3, patches.shape[1]).argsort(dim=-1)[:, int(0.75 * patches.shape[1]):]
        encoded = enc.transformer(tokens[torch.arange(3)[:, None], keep])
    blob["mae"] = {"img": img, "patches": patches, "tokens": tokens, "keep": keep, "encoded": encoded,
                   "pixel_values_per_patch": enc.to_patch_embedding[2].weight.shape[-1]}

    # AcceptVideoWrapper: `patch_size`, and the frames of a clip through forward() as one batch
    kwargs = dict(image_size=32, patch_size=8, num_classes=7, dim=32, depth=1, heads=2, mlp_dim=48, dim_head=16)
    net = init("vit_video", ViT, 0, kwargs).eval()
    torch.manual_seed(3)
    video = torch.randn(2, 3, 4, 32, 32)
    Wrapper = importlib.import_module("vit_pytorch.accept_video_wrapper").AcceptVideoWrapper
    with torch.no_grad():
        frames = net(video.permute(0, 2, 1, 3, 4).reshape(8, 3, 32, 32))
        wrapped = Wrapper(net, add_time_pos_emb=False)(video)
    assert torch.allclose(wrapped, frames.reshape(2, 4, 7))
    blob["video"] = {"video": video, "patch_size": Wrapper(net).patch_size, "frames": frames}

    # DistillWrapper calls teacher(img) under no_grad: fp32 and the reference's own bf16 teacher logits
    for name, kwargs, shape in (("distill", dict(image_size=32, patch_size=8, num_classes=5, dim=64, depth=1,
                                                 heads=2, mlp_dim=96), (2, 3, 32, 32)),
                                ("distill_gpu", dict(image_size=64, patch_size=8, num_classes=10, dim=128, depth=2,
                                                     heads=2, mlp_dim=256), (4, 3, 64, 64))):
        teacher = init(name, ViT, 0, kwargs).eval()
        torch.manual_seed(4)
        img = torch.randn(shape).bfloat16()
        with torch.no_grad():
            blob[name] = {"img": img, "logits_fp32": teacher(img.float()),
                          "logits_ref_bf16": teacher.bfloat16()(img).float()}

    blob["versions"] = {"torch": str(torch.__version__), "reference": "vit-pytorch 1.23.6"}
    path = os.path.join(HERE, "reference_surface.pt")
    torch.save(blob, path)
    print(f"reference_surface: {len(blob['init'])} seeded constructors, {len(blob['signatures'])} signatures; "
          f"{os.path.getsize(path) / 1e6:.2f} MB")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "surface":
        make_reference_surface()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "navit_nested":
        make_navit_nested()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "navit_config5":
        make_navit_config5()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "frontends":
        for n, s in CASES3.items():
            make(n, s)
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "round2":
        for n, s in CASES2.items():
            make(n, s)
        sys.exit(0)
    for n, s in {**CASES, **CASES2, **CASES3}.items():
        make(n, s)
    make_navit()
    make_navit_config5()
    make_navit_nested()
    make_reference_surface()
