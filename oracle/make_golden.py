"""Pin the oracle against the REAL reference and write tests/golden/*.pt.

Runs only in the build container (needs /root/reference; never on the GPU box).  The
reference's own `RobotVisionFM` is imported from /root/reference/src through two shims
(SURVEY.md section 8c): an `omegaconf` stub and offline `from_pretrained` factories.  For
each case the oracle's deterministic weights are loaded into the reference module, the
reference forward / get_loss / backward are run in fp32 on CPU, the oracle restatement is
asserted equal, and a compact fixture (strided slices + norms + scalars) is saved.

    python oracle/make_golden.py [case ...]      # no argument = every case
"""
from __future__ import annotations

import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle import theia_oracle as O  # noqa: E402



def import_reference():
    """the reference's RobotVisionFM straight from /root/reference/src (shims: baseline/ref_shim.py)"""
    from baseline import ref_shim
    return ref_shim.import_reference(prefer_installed=False)


def sl(t: torch.Tensor) -> torch.Tensor:
    """strided sample that keeps fixtures small (tests/test_oracle.py and tests/test_teachers_gpu.py repeat it as
    _sl: the three must stay identical)"""
    f = t.detach().flatten()
    step = max(1, f.numel() // 4096)
    return f[::step][:4096].clone()


def summarize(t: torch.Tensor) -> dict:
    t = t.detach().double()
    return {"shape": tuple(t.shape), "sample": sl(t.float()), "l2": t.norm().item(), "mean": t.mean().item()}


CASES = [
    # name, backbone, teachers, B, do_resize
    ("tiny_dinov2_b2", "facebook/deit-tiny-patch16-224", "dinov2", 2, False),
    ("tiny_cdiv_b2_resize", "facebook/deit-tiny-patch16-224", "cdiv", 2, True),
    ("tiny_cddsv_b1", "facebook/deit-tiny-patch16-224", "cddsv", 1, False),
    ("tiny_dinov2_cls_b3", "facebook/deit-tiny-patch16-224", "dinov2+cls", 3, False),  # distill_cls (train_rvfm.py:239-246)
    ("tiny_nocls_dinov2_b2", "nocls-facebook/deit-tiny-patch16-224", "dinov2", 2, False),  # DeiTNoCLS (backbones.py:344)
    ("tiny_reg_dinov2_b2", "reg-facebook/deit-tiny-patch16-224", "dinov2", 2, False),      # DeiTReg (backbones.py:424)
    # the backbone / teacher set BASELINE.json's metric is quoted on (deit-base + cdiv)
    ("base_cdiv_b2", "facebook/deit-base-patch16-224", "cdiv", 2, False),
]


def main():
    RobotVisionFM = import_reference()
    os.makedirs(os.path.join(os.path.dirname(HERE), "tests", "golden"), exist_ok=True)
    torch.manual_seed(0)
    only = set(sys.argv[1:])
    for name, backbone, tset, B, do_resize in CASES:
        if only and name not in only:
            continue
        cfg = O.make_config(backbone, tset.replace("+cls", ""), distill_cls=tset.endswith("+cls"))
        P = O.init_params(cfg, seed=0)
        ref = RobotVisionFM(backbone=backbone, pretrained=False, translator="lconv",
                            target_feature_sizes=dict(cfg.teachers), translator_kwargs={"hidden_size_factor": 1.0})
        sd = ref.state_dict()
        assert set(sd.keys()) == set(P.keys()), (set(sd) ^ set(P))
        for k in sd:
            assert tuple(sd[k].shape) == tuple(P[k].shape), k
        ref.load_state_dict(P)
        ref.train()
        images, targets = O.synthetic_batch(cfg, B, seed=0)
        kw = {"do_resize": do_resize}
        # --- reference ---
        feat_ref = ref.forward_feature(images, **kw)
        pred_ref = ref(images, **kw)
        losses_ref = ref.get_loss(pred_ref, targets)
        ml = 0.9 * losses_ref["cos_loss"] + 0.1 * losses_ref["l1_loss"]
        ref.zero_grad()
        ml.backward()
        grads_ref = {k: (p.grad if p.grad is not None else torch.zeros_like(p)) for k, p in ref.named_parameters()}
        # --- oracle restatement must agree (fp32 CPU, same kernels => tight) ---
        feat_o = O.forward_feature(P, images, cfg, **kw)
        pred_o, losses_o, grads_o = O.distill_step(P, images, targets, cfg, **kw)
        torch.testing.assert_close(feat_o, feat_ref, rtol=1e-4, atol=1e-5)
        for t in pred_ref:
            torch.testing.assert_close(pred_o[t], pred_ref[t], rtol=1e-4, atol=1e-4)
        for k in ("mse_loss", "cos_loss", "l1_loss"):
            torch.testing.assert_close(losses_o[k].detach(), losses_ref[k].detach(), rtol=1e-5, atol=1e-7)
        worst, worst_k = 0.0, ""
        gmax = max(v.norm().item() for v in grads_ref.values())
        for k in grads_ref:
            num = (grads_o[k] - grads_ref[k]).norm().item()
            # key.bias has a mathematically-zero gradient (softmax shift invariance): floor the
            # denominator so fp noise there is not reported as a relative error
            den = grads_ref[k].norm().item() + 1e-6 * gmax
            if num / den > worst:
                worst, worst_k = num / den, k
        # fp32 summation-order noise: ~1.6e-3 in the 3.1M-element LN of the 64x64 heads; deit-base (K = 3072 / 6912
        # reductions, SDPA vs explicit softmax) reaches 5e-3 on its smallest-gradient tensor
        assert worst < (1e-2 if "base" in backbone else 5e-3), (worst, worst_k)
        print("   worst-agreeing gradient tensor:", worst_k, f"{worst:.2e}")
        fx = {
            "case": name, "backbone": backbone, "teachers": list(cfg.teachers), "B": B, "seed": 0,
            "kwargs": kw,
            "feature": summarize(feat_ref),
            "pred": {t: summarize(v) for t, v in pred_ref.items()},
            "losses": {k: float(losses_ref[k]) for k in ("mse_loss", "cos_loss", "l1_loss")},
            "losses_per_model": {k: dict(losses_ref[k]) for k in
                                 ("mse_losses_per_model", "cos_losses_per_model", "l1_losses_per_model")},
            "main_loss": float(ml),
            "grad_l2": {k: v.double().norm().item() for k, v in grads_ref.items()},
            "grad_sample": {k: sl(v) for k, v in grads_ref.items()
                            if k.endswith("cls_token") or "layer.0.attention.attention.query" in k
                            or "layer.11.output.dense" in k or "adapter.8" in k or "pad.1" in k
                            or "adapter.3.weight" in k or "layernorm.weight" in k},
            "versions": {"torch": torch.__version__},
        }
        out = os.path.join(os.path.dirname(HERE), "tests", "golden", name + ".pt")
        torch.save(fx, out)
        print(f"{name}: oracle==reference (worst grad rel {worst:.2e}); main_loss {float(ml):.6f} -> {out} "
              f"({os.path.getsize(out) / 1024:.0f} KiB)")

    if not only or "tiny_anysize" in only:
        anysize(RobotVisionFM)
    if not only or "teachers" in only:
        teachers()
    if only and "readme_zeros" not in only:
        return
    # README quick-start (BASELINE config #1): zeros image through deit-tiny forward_feature
    cfg = O.make_config("facebook/deit-tiny-patch16-224", "dinov2")
    P = O.init_params(cfg, seed=0)
    ref = RobotVisionFM(backbone="facebook/deit-tiny-patch16-224", pretrained=False, translator="lconv",
                        target_feature_sizes=dict(cfg.teachers), translator_kwargs={"hidden_size_factor": 1.0})
    ref.load_state_dict(P)
    ref.eval()
    z = torch.zeros((1, 224, 224, 3), dtype=torch.uint8)
    with torch.no_grad():
        f = ref.forward_feature(z)
    fo = O.forward_feature(P, z, cfg)
    torch.testing.assert_close(fo, f, rtol=1e-4, atol=1e-5)
    assert tuple(f.shape) == (1, 196, 192)
    torch.save({"case": "readme_zeros", "feature": summarize(f)},
               os.path.join(os.path.dirname(HERE), "tests", "golden", "readme_zeros.pt"))
    print("readme_zeros ok", tuple(f.shape))


ANYSIZE = [  # (H, W, do_resize): the processor resizes to 256 x 256 and / or centre-crops / zero-pads to 224 x 224
    (300, 240, True), (160, 200, True), (480, 640, True), (160, 200, False), (256, 320, False), (200, 300, False),
]


def anysize_images(H, W, B=2):
    return torch.randint(0, 256, (B, H, W, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(H * 1000 + W))


def anysize(RobotVisionFM):
    """images of other extents than 224 x 224 through the reference's forward_feature (CPU uint8 tensors: torchvision's
    fixed-point resize); the oracle must agree, the summaries become tests/golden/anysize_tiny.pt"""
    cfg = O.make_config("facebook/deit-tiny-patch16-224", "dinov2")
    P = O.init_params(cfg, seed=0)
    ref = RobotVisionFM(backbone="facebook/deit-tiny-patch16-224", pretrained=False, translator="lconv",
                        target_feature_sizes=dict(cfg.teachers), translator_kwargs={"hidden_size_factor": 1.0})
    ref.load_state_dict(P)
    ref.eval()
    out = []
    for H, W, do_resize in ANYSIZE:
        x = anysize_images(H, W)
        with torch.no_grad():
            f = ref.forward_feature(x, do_resize=do_resize, interpolate_pos_encoding=True)
            f2 = ref.forward_feature(x, do_resize=do_resize)
        assert torch.equal(f, f2) and tuple(f.shape) == (2, 196, 192)  # the flag is the identity on this path
        fo = O.forward_feature(P, x, cfg, do_resize=do_resize)
        torch.testing.assert_close(fo, f, rtol=1e-4, atol=1e-5)
        out.append({"H": H, "W": W, "do_resize": do_resize, "feature": summarize(f)})
        print(f"anysize {H}x{W} do_resize={do_resize}: oracle == reference, |f| = {float(f.abs().mean()):.4f}")
    path = os.path.join(os.path.dirname(HERE), "tests", "golden", "anysize_tiny.pt")
    torch.save({"case": "tiny_anysize", "cases": out}, path)
    print("->", path, f"({os.path.getsize(path) / 1024:.0f} KiB)")


def teachers():
    """the reference's teacher wrappers (get_dinov2_feature / get_clip_feature / get_vit_feature) on the seeded HF
    models and images of tests/test_teachers_gpu.py, fp32 on CPU; the summaries become tests/golden/teachers.pt"""
    from theia.foundation_models.vision_language_models.clip import get_clip_feature
    from theia.foundation_models.vision_models.dinov2 import get_dinov2_feature
    from theia.foundation_models.vision_models.vit import get_vit_feature
    from tests._teacher_util import CASES, _build, _images, _processors, _randomize
    fns = {"dinov2": get_dinov2_feature, "clip": get_clip_feature, "vit": get_vit_feature}
    out = []
    for kind, arch, B in CASES:
        hf = _randomize(_build(kind, arch), seed=1)
        want = fns[kind](hf, _processors()[kind], _images(B))
        out.append({"kind": kind, "arch": arch, "B": B, "outputs": [summarize(w) for w in want]})
        print(f"teacher {kind} {arch} B={B}: {[tuple(w.shape) for w in want]}")
    path = os.path.join(os.path.dirname(HERE), "tests", "golden", "teachers.pt")
    torch.save({"case": "teachers", "cases": out, "versions": {"torch": torch.__version__}}, path)
    print("->", path, f"({os.path.getsize(path) / 1024:.0f} KiB)")


if __name__ == "__main__":
    main()
