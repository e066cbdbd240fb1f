"""How the weights of a make_golden.py case are drawn, shared by make_golden.py (which draws them with the reference's
classes) and by the tests and smoke() (which draw them with the drop-in's).  The drop-in's constructors consume the
RNG exactly like the reference's (tests/test_dropin.py, tests/test_variants.py), so a fixture stores the seed and a
sha256 digest of the bf16 state_dict instead of the weights themselves; load() rebuilds them and checks the digest."""
import hashlib
import importlib

import torch


def state_digest(sd) -> dict:
    """name -> (shape, sha256 of the raw bytes) of every tensor: equal digests mean bit-identical tensors."""
    out = {}
    for k, v in sd.items():
        t = v.detach().cpu().contiguous()
        if t.dtype == torch.bfloat16:
            t = t.view(torch.int16)
        out[k] = (tuple(v.shape), hashlib.sha256(t.numpy().tobytes()).hexdigest())
    return out


def golden_model(cls, kwargs: dict, seed: int):
    """`cls(**kwargs)` under torch.manual_seed(seed), with bf16-representable parameters and LayerNorm affine
    parameters / q-k norm scales perturbed from their init so that they are actually exercised."""
    torch.manual_seed(seed)
    model = cls(**kwargs).eval()
    g = torch.Generator().manual_seed(1000 + seed)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if p.dim() == 1 and ("norm" in n or n.split(".")[-2] in ("0", "1", "3")) and n.endswith("weight"):
                p.add_(0.1 * torch.randn(p.shape, generator=g))
            elif p.dim() == 1 and n.endswith("bias"):
                p.add_(0.05 * torch.randn(p.shape, generator=g))
            elif n.endswith("gamma"):                       # per-head q / k RMSNorm scales
                p.mul_(1.0 + 0.2 * torch.randn(p.shape, generator=g))
            p.copy_(p.bfloat16().float())
    return model


def dropin_class(kind: str):
    """Fixture `kind` -> the drop-in class (`kind` names the reference module for the SimpleViT variants)."""
    if kind in ("vit", "simple"):
        from vit_pytorch_b200 import SimpleViT, ViT
        return ViT if kind == "vit" else SimpleViT
    return importlib.import_module("vit_pytorch_b200." + kind).SimpleViT


def load(path: str) -> dict:
    """A fixture; when it stores its weights as seed + digest, `state_dict` is rebuilt with the drop-in's class and
    checked bit for bit against the digest of the reference's."""
    blob = torch.load(path, weights_only=False)
    if "state_digest" in blob:
        model = golden_model(dropin_class(blob["kind"]), blob["kwargs"], blob["seed"])
        sd = {k: v.bfloat16() for k, v in model.state_dict().items()}
        # same names in the same order, same shapes, same bits as the reference's
        assert list(state_digest(sd).items()) == list(blob["state_digest"].items()), \
            f"{path}: rebuilt weights differ from the reference's"
        blob["state_dict"] = sd
    return blob
