"""HF teacher architectures with seeded random weights + the processors of the real checkpoints (offline)."""
import math

import numpy as np
import torch
import torch.nn.functional as F


# (kind, (hidden, heads, layers, patch), batch) of tests/test_teachers_gpu.py and tests/golden/teachers.pt
CASES = [
    ("dinov2", (1024, 16, 24, 14), 3),  # facebook/dinov2-large: 257 tokens
    ("dinov2", (384, 6, 12, 14), 5),    # facebook/dinov2-small
    ("clip", (1024, 16, 24, 14), 2),    # openai/clip-vit-large-patch14: quick_gelu, pre_layrnorm, post_layernorm(cls)
    ("clip", (768, 12, 12, 16), 4),     # openai/clip-vit-base-patch16: 197 tokens (the student's attention kernel)
    ("vit", (768, 12, 12, 16), 3),      # google/vit-base-patch16-224-in21k
    ("vit", (1024, 16, 4, 14), 2),      # ViT-L/14 geometry, shortened
    ("vit", (1280, 16, 32, 14), 2),     # google/vit-huge-patch14-224-in21k (the reference's default): head dim 80
]


def _images(B):
    """B seeded uint8 HWC images, the first one constant (all zeros)"""
    rng = np.random.default_rng(3)
    images = [rng.integers(0, 256, (224, 224, 3), dtype=np.uint8) for _ in range(B)]
    images[0][:] = 0
    return images


def _randomize(model, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if "lambda1" in n:  # DINOv2 LayerScale
                p.copy_(0.3 + 0.7 * torch.rand(p.shape, generator=g))
            elif p.ndim == 1 and ("norm" in n or "layrnorm" in n) and n.endswith("weight"):
                p.copy_(1.0 + 0.2 * torch.randn(p.shape, generator=g))
            elif p.ndim == 1:
                p.copy_(0.1 * torch.randn(p.shape, generator=g))
            elif p.ndim == 2 and "position" not in n:
                gain = 1.5 if any(k in n for k in ("query", "key", "q_proj", "k_proj")) else 1.0
                p.copy_(torch.randn(p.shape, generator=g) * gain / math.sqrt(p.shape[1]))
            elif p.ndim == 4:
                p.copy_(torch.randn(p.shape, generator=g) / math.sqrt(p[0].numel()))
            else:  # class / position embeddings
                p.copy_(0.3 * torch.randn(p.shape, generator=g))
    return model.eval()


def _processors():
    from transformers import BitImageProcessor, CLIPImageProcessor, ViTImageProcessor
    return {
        # facebook/dinov2-large preprocessor_config.json: resize 256 (bicubic), centre crop 224, ImageNet mean / std
        "dinov2": BitImageProcessor(do_resize=True, size={"shortest_edge": 256}, resample=3, do_center_crop=True,
                                    crop_size={"height": 224, "width": 224}, do_rescale=True, do_normalize=True,
                                    image_mean=[0.485, 0.456, 0.406], image_std=[0.229, 0.224, 0.225], do_convert_rgb=True),
        "clip": CLIPImageProcessor(),
        "vit": ViTImageProcessor(),
    }


def _build(kind, arch):
    from transformers import CLIPVisionConfig, CLIPVisionModel, Dinov2Config, Dinov2Model, ViTConfig, ViTModel
    D, H, Ly, patch = arch
    if kind == "dinov2":
        return Dinov2Model(Dinov2Config(hidden_size=D, num_hidden_layers=Ly, num_attention_heads=H, image_size=518, patch_size=patch))
    if kind == "clip":
        return CLIPVisionModel(CLIPVisionConfig(hidden_size=D, num_hidden_layers=Ly, num_attention_heads=H, image_size=224,
                                                patch_size=patch, intermediate_size=4 * D))
    return ViTModel(ViTConfig(hidden_size=D, num_hidden_layers=Ly, num_attention_heads=H, image_size=224, patch_size=patch,
                              intermediate_size=4 * D))


def _replay(t, pixel_values):
    """plain fp32 torch restatement of theia_vit_forward's launch sequence (csrc/vit_infer.cu) over the CONVERTED
    buffers of a TeacherViT: what the kernels compute, minus bf16 activation rounding"""
    c, W = t.cfg, t._t
    B = pixel_values.shape[0]
    p, g = c["patch"], c["image"] // c["patch"]
    # theia_patchify_f32: row = token, column = ch*p*p + i*p + j, zero padding columns / non-patch rows
    pat = pixel_values.unfold(2, p, p).unfold(3, p, p).permute(0, 2, 3, 1, 4, 5).reshape(B, g * g, 3 * p * p)
    rows = torch.zeros(B, c["tokens"], c["patch_k"], device=pixel_values.device)
    rows[:, c["patch_off"]:c["patch_off"] + g * g, :3 * p * p] = pat
    x = rows @ W["w_patch"].float().t()
    if W["b_patch"] is not None:
        x = x + W["b_patch"]
    ispatch = torch.zeros(c["tokens"], dtype=torch.bool, device=pixel_values.device)
    ispatch[c["patch_off"]:c["patch_off"] + g * g] = True
    x = torch.where(ispatch[None, :, None], x + W["tok_table"], W["tok_table"].expand_as(x))  # THEIA_EPI_POSCLS
    D, H = c["hidden"], c["heads"]
    ln = lambda v, w, b: F.layer_norm(v, (D,), w, b, c["ln_eps"])
    if W["pre_ln_w"] is not None:
        x = ln(x, W["pre_ln_w"], W["pre_ln_b"])
    for ly in t._layers:
        qkv = ln(x, ly["ln1_w"], ly["ln1_b"]) @ ly["w_qkv"].float().t() + ly["b_qkv"]
        q, k, v = (qkv[..., i * D:(i + 1) * D].reshape(B, -1, H, D // H).transpose(1, 2) for i in range(3))
        a = (torch.softmax(q @ k.transpose(2, 3) * (D // H) ** -0.5, -1) @ v).transpose(1, 2).reshape(B, -1, D)
        x = x + a @ ly["w_o"].float().t() + ly["b_o"]
        h = ln(x, ly["ln2_w"], ly["ln2_b"]) @ ly["w_fc1"].float().t() + ly["b_fc1"]
        h = h * torch.sigmoid(1.702 * h) if c["act"] == 1 else F.gelu(h)
        x = x + h @ ly["w_fc2"].float().t() + ly["b_fc2"]
    if c["final_ln_mode"] == 1:
        x = ln(x, W["final_ln_w"], W["final_ln_b"])
        return x, x[:, 0]
    return x, ln(x[:, 0], W["final_ln_w"], W["final_ln_b"])
