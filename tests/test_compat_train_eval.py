"""train_nerf.py / eval_nerf.py on the compat/ overlay (north_star: "so train_nerf.py, eval_nerf.py and mesh_nerf.py run
unmodified"): the scripts' call sequence is replayed against the overlay's modules with an in-memory dataset of images
rendered from the lego checkpoint: Trainer.fit (training_step on the fused loss+backward, optimiser / scheduler steps,
validation with image logging, ModelCheckpoint, resume), then the eval_nerf.py loop (batchify -> model.query -> PSNR) on
the checkpoint it wrote."""
import math
import os
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

sys.path.insert(0, os.path.join(ROOT, "tools"))


# ------------------------------------------------------------------------------------------------ GPU replay
class ImageDataset(torch.utils.data.Dataset):
    """What the reference's BlenderDataset yields per item (src/data/datasets.py:215-233): a dict of per-image tensors; the
    training split holds `num_random_rays` random rays of the image, the others the whole image."""

    def __init__(self, eng, poses, images, size, focal, rays=None):
        self.items = []
        for pose, img in zip(poses, images):
            o, d = eng.ray_bundle(pose, size, size, focal)
            self.items.append(dict(ray_origins=o.cpu(), ray_directions=d.cpu(), ray_targets=img.cpu(), ray_bounds=torch.tensor([2.0, 6.0]),
                                   hwf=(size, size, focal)))
        self.rays = rays

    def __len__(self):
        return len(self.items)

    def __getitem__(self, idx):
        it = dict(self.items[idx])
        if self.rays is not None:
            sel = torch.randperm(it["ray_targets"].shape[0] * it["ray_targets"].shape[1])[:self.rays]
            it["ray_directions"] = it["ray_directions"].reshape(-1, 3)[sel]
            it["ray_targets"] = it["ray_targets"].reshape(-1, 3)[sel]
        it["size"] = 1
        return it


@pytest.mark.gpu
def test_overlay_trainer_fit_checkpoint_resume_and_eval_sequence(tmp_path):
    import make_synthetic_blender as M
    from conftest import load_npz
    from test_gpu_parity import LEGO_CFG
    import nerfmeshes_b200 as nm
    sys.path.insert(0, os.path.join(ROOT, "compat"))
    try:
        import models as ov
        import pytorch_lightning as pl
        from pytorch_lightning.callbacks import Callback, ModelCheckpoint
        from pytorch_lightning.loggers import TensorBoardLogger
        from nerf.nerf_helpers import batchify, mse2psnr
        size, focal = 32, 0.5 * 32 / math.tan(0.5 * M.ANGLE_X)
        teacher = nm.NeRFModel.from_npz(LEGO_CFG, load_npz("weights_lego_nerf.npz")).eval().cuda()
        teng = teacher._engine()
        poses = [nm.pose_spherical(a, -30.0, 4.0) for a in np.linspace(-180, 180, 10, endpoint=False)]
        images = [teng.render_image(p, size, size, focal, 2.0, 6.0, want=["rgb"])["rgb"].view(size, size, 3).clamp(0, 1) for p in poses]

        cfg = M.config(str(tmp_path), tiny=True, train_iters=36, rays=512, size=size)

        class Model(ov.NeRFModel):
            def load_dataset(self, dataset_type):                       # the data layer is the reference's; here: in-memory images
                kind = getattr(dataset_type, "value", dataset_type)
                sl = {"train": slice(0, 6), "val": slice(6, 8), "test": slice(8, 10)}[kind]
                return ImageDataset(teng, poses[sl], images[sl], size, focal, rays=512 if kind == "train" else None)

            def load_train_dataset(self):
                self.train_dataset = self.load_dataset("train")

            def load_val_dataset(self):
                self.val_dataset = self.load_dataset("val")
                self._clamp_val_samples()

        class Recorder(Callback):
            def __init__(self):
                self.train, self.val = [], []

            def on_train_batch_end(self, trainer, pl_module, batch, batch_idx, dataloader_idx):
                self.train.append(trainer.callback_metrics["train/loss"])

            def on_validation_epoch_end(self, trainer, pl_module):
                self.val.append(trainer.callback_metrics["validation/loss"])

        torch.manual_seed(0)
        model = Model(cfg)
        logger = TensorBoardLogger(str(tmp_path / "logs" / "synthetic-lego"), "default")
        ckpt_dir = os.path.join(logger.log_dir, "checkpoints")
        rec = Recorder()
        trainer = pl.Trainer(logger=logger, checkpoint_callback=ModelCheckpoint(filepath=ckpt_dir, save_top_k=3, save_last=True, monitor="val_loss",
                                                                               mode="min", prefix="model_"),
                             callbacks=[rec], gpus=1, num_sanity_val_steps=0, resume_from_checkpoint=None, precision=32)
        trainer.fit(model)
        assert trainer.global_step == 36 and len(rec.train) == 36 and len(rec.val) >= 2
        assert np.mean(rec.train[-6:]) < 0.85 * np.mean(rec.train[:6]), rec.train          # it learns
        assert all(math.isfinite(x) for x in rec.train + rec.val)
        last = os.path.join(ckpt_dir, "model_last.ckpt")
        assert os.path.exists(last) and os.path.exists(os.path.join(logger.log_dir, "hparams.yaml"))
        assert any(f.startswith("events.out.tfevents") for f in os.listdir(logger.log_dir))   # validation images / scalars were logged

        # resume: a new trainer picks up step / optimiser state and continues
        cfg2 = M.config(str(tmp_path), tiny=True, train_iters=48, rays=512, size=size)
        model2 = Model(cfg2)
        tr2 = pl.Trainer(logger=None, checkpoint_callback=None, callbacks=[], gpus=1, resume_from_checkpoint=last)
        tr2.fit(model2)
        assert tr2.global_step == 48

        # eval_nerf.py's loop (src/eval_nerf.py:50-105) on the checkpoint: load_from_checkpoint -> eval -> chunked query -> PSNR
        ev = Model.load_from_checkpoint(last).eval().to("cuda")
        test = ImageDataset(teng, poses[8:], images[8:], size, focal)
        psnrs = []
        with torch.no_grad():
            for item in torch.utils.data.DataLoader(test, batch_size=1):
                d, tgt = item["ray_directions"].view(-1, 3), item["ray_targets"].view(-1, 3)
                loss, n = 0.0, d.shape[0] / 512
                for (dd, tt) in batchify(d, tgt, batch_size=512, device="cuda", progress=False):
                    out = ev.query((item["ray_origins"].view(-1, 3).to("cuda"), dd, item["ray_bounds"].view(2)))
                    loss += torch.nn.functional.mse_loss(out.rgb_map, tt)
                psnrs.append(float(mse2psnr(loss / n)))
        assert all(math.isfinite(p) and p > 8.0 for p in psnrs), psnrs
    finally:
        sys.path.remove(os.path.join(ROOT, "compat"))
        for m in [k for k in sys.modules if k.split(".")[0] in ("models", "nerf", "pytorch_lightning", "skimage")]:
            del sys.modules[m]
