"""The reference's OWN training loop (`theia/scripts/train/train_rvfm.py::train`, lines 38-208, imported unmodified
from oracle/_ref) driving `theia_b200.RobotVisionFM`: DDP wrap (train_rvfm.py:258), the reference's parameter
groups (optimizers/utils.py:8-35), torch AdamW, the reference's LR scheduler (lr_schedulers.py:41-77), train + eval
epochs, `freeze_translator()` at the configured step ratio (:149-151), gradient clipping (:126-130), checkpoint saves (:153-156, :203-206).

Stubbed (control plane, out of scope): hydra / webdataset / wandb.log, and the dataloader factory, which yields
synthetic batches in the dataloader's format (uint8 HWC images on the CPU, z-scored bf16 teacher embeddings).
The checkpoint the loop writes is then loaded STRICTLY into the reference's own model, whose fp32 forward must agree
with the CUDA path -- the module is a drop-in in both directions."""
import os
import sys
import types

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _NS(types.SimpleNamespace):
    """attribute access like an OmegaConf node"""


def _import_reference_train():
    from baseline import ref_shim
    if ref_shim.reference_path() is None:
        pytest.skip("oracle/_ref (pip-installed copy of the reference, made by build()) is not present")
    ref_shim.install_shims()
    path = ref_shim.reference_path()
    if path not in sys.path:
        sys.path.insert(0, path)

    def stub(name, **attrs):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.__dict__.update(attrs)
            sys.modules[name] = m
        return sys.modules[name]

    hy = stub("hydra", main=lambda **kw: (lambda f: f))
    hy.utils = stub("hydra.utils", instantiate=lambda *a, **k: None)
    stub("webdataset")
    import importlib
    return importlib.import_module("theia.scripts.train.train_rvfm")


def test_reference_train_loop_runs_on_the_cuda_module(tmp_path, monkeypatch):
    import torch.distributed as dist
    from torch.nn.parallel import DistributedDataParallel as DDP
    from oracle import theia_oracle as O
    from theia_b200 import RobotVisionFM

    T = _import_reference_train()
    from theia.lr_schedulers.lr_schedulers import get_constant_lrs_with_linear_warm_up
    from theia.optimizers.utils import param_groups_weight_decay
    import wandb
    monkeypatch.setattr(wandb, "log", lambda *a, **k: None)

    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29577")
    torch.cuda.set_device(0)
    created = not dist.is_initialized()
    if created:
        dist.init_process_group("nccl", rank=0, world_size=1)
    try:
        backbone, B = "facebook/deit-tiny-patch16-224", 4
        ocfg = O.make_config(backbone, "cdiv")
        names = list(ocfg.teachers)
        # ---- what ddp_main (train_rvfm.py:221-329) builds, with the CUDA module swapped in ----
        rvfm = RobotVisionFM(translator="lconv", translator_kwargs={"hidden_size_factor": 1.0},
                             target_feature_sizes=dict(ocfg.teachers), target_loss_weights=None,
                             backbone=backbone, pretrained=False)
        rvfm.load_state_dict(O.init_params(ocfg, seed=0))
        rvfm.to(0)
        rvfm_ddp = DDP(rvfm, device_ids=[0], find_unused_parameters=False)
        groups = param_groups_weight_decay(rvfm_ddp, 0.01)  # the reference's own grouping
        optimizer = torch.optim.AdamW(groups, lr=2e-3 * (B * 1) / (64 * 8), betas=(0.9, 0.999))
        steps_per_epoch, epochs = 4, 1
        lr_scheduler = get_constant_lrs_with_linear_warm_up(optimizer, warm_up_steps=1, warm_up_lr_start_factor=1e-2)

        g = torch.Generator().manual_seed(7)

        def batches():
            while True:
                b = {"image": torch.randint(0, 256, (B, 224, 224, 3), dtype=torch.uint8, generator=g)}
                for t, (c, h, w) in ocfg.teachers.items():
                    b[t] = {"embedding": torch.randn((B, h * w, c), generator=g).to(torch.bfloat16)}
                yield b

        monkeypatch.setattr(T, "get_frame_dataloader", lambda *a, **k: object())
        monkeypatch.setattr(T, "get_frame_iterator", lambda loaders: batches())
        cfg = _NS(seed=0,
                  training=_NS(epochs=epochs, batch_size=B, num_workers=0, random_target_models=-1, main_loss="cos_l1",
                               grad_clip=True, grad_clip_norm_warmup=1.0, grad_clip_norm=5.0,
                               freeze_translator=True, freeze_translator_start_steps_ratio=1.0),
                  dataset=_NS(shuffle=False, shuffle_buffer_size=1),
                  logging=_NS(save_ckpt_interval=2, run_identifier_prefix="t", model_path=str(tmp_path)))
        before = {k: v.detach().clone() for k, v in rvfm.state_dict().items()}
        T.train(rvfm_ddp, names, optimizer, lr_scheduler, None, None, cfg=cfg, device=0,
                train_epoch_steps=steps_per_epoch, eval_epoch_steps=2,
                total_train_steps=steps_per_epoch * epochs, warmup_steps=1)
        torch.cuda.synchronize()
        # checkpoints written by the loop (every 2 steps and at the end of the epoch)
        ckpts = sorted(os.listdir(tmp_path))
        assert ckpts == ["t_step00000002.pth", "t_step00000004.pth"], ckpts
        sd = torch.load(os.path.join(tmp_path, ckpts[-1]), map_location="cpu")
        assert set(sd) == set(before)
        moved = sum(int(not torch.equal(sd[k], before[k].cpu())) for k in sd)
        assert moved > 200 and all(torch.isfinite(v).all() for v in sd.values())
        # freeze_translator() fired at the configured step (here the last one: under the reference's DDP wrapper with
        # find_unused_parameters=False no training iteration may follow it -- a property of the reference's loop, not
        # of the module; FlatAdamW's handling of frozen parameters is tested in test_model_gpu.py)
        assert all(not p.requires_grad for p in rvfm.translator.parameters())
        assert all(p.requires_grad for n, p in rvfm.named_parameters() if n.startswith("backbone"))
        # the checkpoint drops into the REFERENCE model (strict) and its fp32 forward agrees with the CUDA path
        from baseline import ref_shim
        Ref = ref_shim.import_reference()
        ref = Ref(backbone=backbone, pretrained=False, translator="lconv", target_feature_sizes=dict(ocfg.teachers),
                  translator_kwargs={"hidden_size_factor": 1.0})
        ref.load_state_dict({k: v.clone() for k, v in sd.items()}, strict=True)
        ref.eval().to(0)
        images = next(batches())["image"]
        with torch.no_grad():
            pr = ref(images.to(0))
            rvfm.eval()
            po = rvfm(images)  # CPU images, as the eval loop passes them (train_rvfm.py:165)
        for t in names:
            err = ((po[t].double() - pr[t].double()).norm() / pr[t].double().norm()).item()
            assert err < 3e-2, (t, err)
    finally:
        if created:
            dist.destroy_process_group()
