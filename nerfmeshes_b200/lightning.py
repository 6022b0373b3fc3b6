"""The PyTorch-Lightning side of the reference's models, for the fused path — what `train_nerf.py` needs from `models.NeRFModel`
/ `models.BuFFModel` beyond forward/query: the hooks a Lightning 0.9 Trainer calls
  src/models/model_base.py:40-187   setup, dataloaders, validation_epoch_end (with its Chamfer metric), configure_optimizers,
                                    check_early_stopping
  src/models/model_nerf.py:88-230   NeRFModel.training_step / validation_step
  src/models/model_buff.py:75-165   BuFFModel.training_step / validation_step
as a mixin over nerfmeshes_b200.models (compat/models exports the combined classes).  Differences from the reference, all on
the training step: forward + loss + backward of a chunk are ONE library call (nm_loss_backward, see train.training_step), so
the step returns a loss without an autograd graph and the parameters' .grad are already filled when it returns — the
overlay's Trainer (compat/pytorch_lightning) steps the optimiser without calling backward again.  The datasets are the
reference's own (`data.datasets`, imported lazily: the data layer is out of scope and stays the reference's code)."""
from __future__ import annotations

import torch

from .train import mse2psnr, training_step as fused_training_step


def _cast_to_image(t: torch.Tensor):
    """nerf.cast_to_image: (H,W,3) float -> (3,H,W) uint8 array (src/nerf/nerf_helpers.py:162-168)."""
    import numpy as np
    return np.moveaxis(t.detach().cpu().float().mul(255).byte().numpy(), [-1], [0])


def _ray_batch(d: dict):
    """DataBundle.deserialize(batch).to_ray_batch() (src/data/data_helpers.py:134-146) on the dict a DataLoader yields."""
    g = lambda k: d.get(k)
    o, dirs, tgt, bounds = g("ray_origins"), g("ray_directions"), g("ray_targets"), g("ray_bounds")
    out = dict(ray_origins=o.reshape(-1, 3), ray_directions=dirs.reshape(-1, 3), ray_bounds=bounds.reshape(2),
               ray_targets=None if tgt is None else tgt.reshape(-1, 3), hwf=g("hwf"))
    if out["hwf"] is not None:
        out["hwf"] = tuple(float(x) if i == 2 else int(x) for i, x in enumerate(out["hwf"]))
    return out


class LightningHooks:
    """Mixin: list it BEFORE the nerfmeshes_b200 model class."""
    trainer = None
    logger = None
    train_dataset = None
    val_dataset = None
    val_num_samples = -1

    @property
    def device(self):
        p = next(self.parameters())
        return p.device

    def loss(self, a, b):
        return torch.nn.functional.mse_loss(a, b)

    @staticmethod
    def criterion_psnr(mse):
        return mse2psnr(float(mse))

    # ------------------------------------------------------------------ model_base.py:40-57
    def setup(self, stage):
        self.load_train_dataset()
        self.load_val_dataset()
        steps_train = int(self.cfg.experiment.train_iters)
        self.trainer.min_steps = steps_train
        self.trainer.max_steps = steps_train
        epochs_train = steps_train // len(self.train_dataset)
        self.trainer.max_epochs = epochs_train
        self.trainer.min_epochs = epochs_train
        self.trainer.check_val_every_n_epoch = int(self.cfg.experiment.validate_every) // len(self.train_dataset)

    # ------------------------------------------------------------------ model_base.py:106-147
    def load_dataset(self, dataset_type):
        from data.datasets import BlenderDataset, ColmapDataset           # the reference's data layer (out of scope here)
        kind = self.cfg.dataset.type
        if kind == "blender":
            return BlenderDataset(self.cfg, type=dataset_type)
        if kind == "colmap":
            return ColmapDataset(self.cfg, type=dataset_type)
        raise NotImplementedError(kind)

    def load_train_dataset(self):
        from data.datasets import DatasetType
        self.train_dataset = self.load_dataset(DatasetType.TRAIN)

    def load_val_dataset(self):
        from data.datasets import DatasetType
        self.val_dataset = self.load_dataset(DatasetType.VALIDATION)
        self._clamp_val_samples()

    def _clamp_val_samples(self):
        self.val_num_samples = int(self.cfg.nerf.validation.get("num_samples", -1))
        if self.val_num_samples != -1:
            self.val_num_samples = max(min(len(self.val_dataset), self.val_num_samples), 1)

    def train_dataloader(self):
        return torch.utils.data.DataLoader(self.train_dataset, batch_size=1, shuffle=False,
                                           num_workers=int(self.cfg.dataset.get("num_workers", 0)), pin_memory=False)

    def val_dataloader(self):
        sampler = None
        if self.val_num_samples != -1:
            sampler = torch.utils.data.RandomSampler(self.val_dataset, replacement=True, num_samples=self.val_num_samples)
        return torch.utils.data.DataLoader(self.val_dataset, shuffle=False, batch_size=1, sampler=sampler,
                                           num_workers=int(self.cfg.dataset.get("num_workers", 0)), pin_memory=False)

    # ------------------------------------------------------------------ model_base.py:179-187
    def check_early_stopping(self, rgb):
        exp = self.cfg.experiment
        if exp.get("use_early_stopping", False) and self.global_step == exp.get("early_stopping_step", -1):
            rgb_sum = float(rgb.sum())
            if rgb_sum < 1e-12:
                print(f"Model is stuck in local minima, model collapsing to {rgb_sum}")
                print("Restart the training again, exiting now...")
                raise SystemExit(-1)

    def _lr(self):
        return self.trainer.optimizers[0].param_groups[0]["lr"] if self.trainer is not None and self.trainer.optimizers else 0.0

    # ------------------------------------------------------------------ model_nerf.py:88-151 / model_buff.py:75-117
    def training_step(self, ray_batch, batch_idx):
        b = _ray_batch(ray_batch)
        dev = self.device
        o, d, tgt = b["ray_origins"].to(dev), b["ray_directions"].to(dev), b["ray_targets"].to(dev)
        if o.shape[0] == 1 and not hasattr(self, "tree"):
            o = o.reshape(3)                      # one shared origin per image (BuFF keeps (1,3): src/nerf/tree.py:231)
        out = fused_training_step(self, (o, d, b["ray_bounds"].cpu()), tgt, global_step=self.global_step, allreduce=False)
        if self.cfg.experiment.get("use_early_stopping", False) and self.global_step == self.cfg.experiment.get("early_stopping_step", -1):
            with torch.no_grad():
                was = self.training
                self.eval()
                self.check_early_stopping(self.query((o, d[:4096], b["ray_bounds"].cpu())).rgb_map)
                self.train(was)
        log = {k: torch.tensor(v) for k, v in out["log"].items()}
        log["train/lr"] = torch.tensor(self._lr())
        return {"loss": torch.tensor(out["loss"]), "log": log}

    # ------------------------------------------------------------------ model_nerf.py:153-230 / model_buff.py:119-161
    @torch.no_grad()
    def validation_step(self, image_ray_batch, batch_idx):
        b = _ray_batch(image_ray_batch)
        dev = self.device
        o, d, tgt = b["ray_origins"].to(dev), b["ray_directions"].to(dev), b["ray_targets"].to(dev)
        bounds = b["ray_bounds"].cpu()
        chunk = int(self.cfg.nerf.validation.chunksize)
        count = tgt.shape[0] / chunk
        per_ray_o = o.shape[0] == d.shape[0] and o.shape[0] > 1
        two = len(self._nets()) > 1 and self._nets()[1] is not None
        is_buff = hasattr(self, "tree")
        coarse_loss = torch.zeros((), device=dev)
        fine_loss = torch.zeros((), device=dev)
        rgb_c, rgb_f = [], []
        for i in range(0, tgt.shape[0], chunk):
            sl = slice(i, i + chunk)
            oo = o[sl] if per_ray_o else (o.reshape(1, 3) if is_buff else o.reshape(3))
            res = self.forward((oo, d[sl], bounds))
            cb, fb = (res, None) if is_buff else res
            coarse_loss = coarse_loss + self.loss(cb.rgb_map, tgt[sl])
            rgb_c.append(cb.rgb_map)
            if two and fb is not None:
                fine_loss = fine_loss + self.loss(fb.rgb_map, tgt[sl])
                rgb_f.append(fb.rgb_map)
        coarse_loss = coarse_loss / count
        loss = coarse_loss
        hwf = b["hwf"]
        exp = getattr(self.logger, "experiment", None)

        def add_image(tag, rgb):
            if exp is not None and hwf is not None:
                exp.add_image(tag + str(batch_idx), _cast_to_image(rgb.view(hwf[0], hwf[1], 3)), self.global_step)
        add_image("validation/rgb_coarse/", torch.cat(rgb_c, 0))
        if is_buff:
            log = {"validation/loss": loss, "validation/psnr": torch.tensor(mse2psnr(float(loss)))}
        else:
            log = {"validation/coarse_loss": coarse_loss, "validation/coarse_psnr": torch.tensor(mse2psnr(float(coarse_loss)))}
            if two:
                add_image("validation/rgb_fine/", torch.cat(rgb_f, 0))
                fine_loss = fine_loss / count
                loss = loss + fine_loss
                log.update({"validation/fine_loss": fine_loss, "validation/fine_psnr": torch.tensor(mse2psnr(float(fine_loss)))})
            log["validation/loss"] = loss
        add_image("validation/img_target/", tgt)
        return {"val_loss": loss, "log": log}

    # ------------------------------------------------------------------ model_base.py:75-104
    # The mesh of the Chamfer metric is extracted at mesh_nerf.py's command-line defaults (its argparse, :204-283).
    CHAMFER_MESH_ARGS = dict(limit=1.2, res=128, iso_level=32.0)
    CHAMFER_TARGET_MISSING = "To compute the chamfer loss, a target mesh .obj must be provided in the dataset folder"

    def chamfer_target_mesh(self):
        """val_dataset.target_mesh if the dataset has one, else <dataset.basedir>/model.obj through load_obj + create_mesh
        (the loader the reference keeps commented out in SynthesizableDataset.__init__, src/data/datasets.py:88-103), else None.
        Without a basedir there is no target file (a bare "model.obj" would be looked up in the working directory).  The
        loaded mesh is kept on the module and read again only when the file's path, size or modification time changes:
        parsing a large OBJ in Python takes seconds, and the hook runs every validation epoch."""
        import os
        from .mesh import create_mesh
        from .metrics import load_obj
        target = getattr(self.val_dataset, "target_mesh", None)
        if target is not None:
            return target
        basedir = self.cfg.dataset.get("basedir", None) if "dataset" in self.cfg else None
        if not basedir:
            return None
        path = os.path.join(str(basedir), "model.obj")
        if not os.path.isfile(path):
            return None
        st = os.stat(path)
        key = (os.path.abspath(path), st.st_size, st.st_mtime_ns)
        cached = getattr(self, "_chamfer_target_cache", None)
        if cached is None or cached[0] != key:
            verts, faces = load_obj(path)
            cached = (key, create_mesh(torch.from_numpy(verts), torch.from_numpy(faces)))
            self._chamfer_target_cache = cached
        return cached[1]

    def validation_epoch_end(self, outputs):
        log_mean = {"log": {}}
        for k in outputs[0]["log"].keys():
            log_mean["log"][k] = torch.stack([torch.as_tensor(x["log"][k]).float().cpu() for x in outputs]).mean()
        log_mean["val_loss"] = torch.stack([torch.as_tensor(x["val_loss"]).float().cpu() for x in outputs]).mean()
        if self.cfg.experiment.get("chamfer_loss", False):
            from data.datasets import SynthesizableDataset           # the reference's data layer (out of scope here)
            if isinstance(self.val_dataset, SynthesizableDataset):
                log_mean["log"]["validation/chamfer_loss"] = self.chamfer_loss()
        return log_mean

    @torch.no_grad()
    def chamfer_loss(self):
        """The Chamfer metric of model_base.py:82-102: points sampled on the target mesh and on the mesh extracted from this
        model, both normalised by create_mesh, compared with chamfer_distance.  Two defects of the reference are fixed: it
        called extract_geometry(self.get_model(), device, None), which fails on args=None and on a FlexibleNeRFModel (it has
        no sample_points); here the mesh comes from this model at CHAMFER_MESH_ARGS.  And its target_mesh was never loaded;
        here it is (chamfer_target_mesh)."""
        from types import SimpleNamespace
        from .mesh import create_mesh, extract_geometry
        from .metrics import chamfer_distance, sample_points_from_meshes
        target = self.chamfer_target_mesh()
        assert target is not None, self.CHAMFER_TARGET_MISSING
        vertices, faces, _, _ = extract_geometry(self, self.device, SimpleNamespace(**self.CHAMFER_MESH_ARGS))
        input_mesh = create_mesh(vertices, faces)
        n = int(self.cfg.experiment.chamfer_sampling_size)
        target_samples = sample_points_from_meshes(target, n)
        input_samples = sample_points_from_meshes(input_mesh, n)
        loss, _ = chamfer_distance(target_samples, input_samples)
        return loss
