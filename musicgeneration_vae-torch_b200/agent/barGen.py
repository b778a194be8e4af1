"""Training / sampling entry point with the surface of the reference's agent/barGen.py: ``BarGen(config)`` with
``run() / train() / train_epoch() / make_batch() / save_checkpoint() / load_checkpoint()``.

What is kept: the pre-training generator step (agent/barGen.py:249-252,302-335: zero_grad, generator forward, Loss,
backward, Adam lr 2e-3), the per-epoch ReduceLROnPlateau(mode='min', factor=0.8, cooldown=6) on the mean loss
(:70-81,361-367), the checkpoint dictionary keys (:174-197, including the ``module.`` prefix nn.DataParallel adds),
the data layout (.npz items concatenated by make_batch, :134-141) and the sampling loop used for the per-epoch
samples (agent/barGen2.py:316-336 == maker_bar.py:32-44).
What is different on purpose: one process per GPU with NCCL gradient all-reduce instead of nn.DataParallel
(agent/barGen.py:96-105) -- launch with torchrun; no per-step ``.item()`` (the running loss stays on the device and
is read once per logging interval); scalars go to a JSONL file when tensorboardX is absent.
Also different: batches reach the device through ``GeneratorTrainer.prefetch`` (the next batch's H2D copy overlaps the
current step), optionally as bits (``config.packed_input`` / ``config.packed_data_path``, data/packed.py); reference
checkpoints load including the ``torch.optim.Adam`` state.
Out of scope (SURVEY.md section 2 rows 12/14): the GAN schedules and the convolutional BarDiscriminator (the
Linear-stack discriminators and graph/model_with_gan.Model exist); after ``pretraining_step_size`` epochs the
generator keeps training on the label-smoothed BCE (``Loss(..., is_pretraining=False)``)."""
import json
import logging
import os
import random
import shutil

import numpy as np
import torch
from torch.utils.data import DataLoader

from .. import parallel
from ..data.bar_dataset import NoteDataset, SyntheticBars
from ..data.packed import PackedBatch, PackedMemmapDataset, PackedNoteDataset, collate_packed
from ..graph.model import Model
from ..maker_bar import sample_songs
from ..metrics import AverageMeter
from ..trainer import GeneratorTrainer


class _Plateau:
    """torch.optim.lr_scheduler.ReduceLROnPlateau(mode='min', factor, patience=10, cooldown, threshold=1e-4 rel)."""

    def __init__(self, factor=0.8, patience=10, cooldown=6, threshold=1e-4):
        self.factor, self.patience, self.cooldown, self.threshold = factor, patience, cooldown, threshold
        self.best, self.bad, self.cool = float("inf"), 0, 0

    def step(self, metric, lr):
        if metric < self.best * (1 - self.threshold):
            self.best, self.bad = metric, 0
        else:
            self.bad += 1
        if self.cool > 0:
            self.cool -= 1
            self.bad = 0
        if self.bad > self.patience:
            self.cool, self.bad = self.cooldown, 0
            return lr * self.factor
        return lr


class _MemmapLoader:
    """re-iterable view of PackedMemmapDataset.batches for one rank (same order every epoch, like the reference's
    DataLoader(shuffle=False), agent/barGen.py:38-41)"""

    def __init__(self, dataset, batch_size, rank, world, pin):
        self.dataset, self.batch_size, self.rank, self.world, self.pin = dataset, batch_size, rank, world, pin

    def __iter__(self):
        return self.dataset.batches(self.batch_size, shuffle=False, rank=self.rank, world=self.world, pin=self.pin)


class BarGen(object):
    def __init__(self, config, dataset=None):
        self.config = config
        self.pretraining_step_size = config.pretraining_step_size
        self.batch_size = config.batch_size
        self.rank, self.world, self.local_rank = parallel.init_from_env()
        torch.cuda.set_device(self.local_rank)
        self.device = torch.device("cuda", self.local_rank)
        self.logger = self.set_logger()

        data_dir = os.path.join(config.root_path, config.data_path)
        if dataset is not None:
            self.dataset = dataset
        elif getattr(config, "packed_array_path", None) and os.path.isdir(os.path.join(config.root_path,
                                                                                       config.packed_array_path)):
            self.dataset = PackedMemmapDataset(os.path.join(config.root_path, config.packed_array_path))
        elif getattr(config, "packed_data_path", None) and os.path.isdir(os.path.join(config.root_path,
                                                                                      config.packed_data_path)):
            self.dataset = PackedNoteDataset(config.root_path, config)
        elif os.path.isdir(data_dir):
            self.dataset = NoteDataset(config.root_path, config)
        elif getattr(config, "synthetic", False):
            self.dataset = SyntheticBars(64, 4, self.batch_size)         # explicit opt-in only (config.synthetic)
        else:
            # the reference raises from os.listdir (data/bar_dataset.py:12); a mistyped path must not train on noise
            raise FileNotFoundError("no dataset directory %r (nor config.packed_array_path / packed_data_path); set "
                                    "config.synthetic = True to train on random bars" % data_dir)
        # DistributedSampler semantics of agent/barGen_horovod.py:49-50: every rank takes an equally long shard (padded by
        # wrapping around), so all ranks run the same number of optimiser steps / all-reduces per epoch
        self.indices = parallel.shard_indices(len(self.dataset), self.rank, self.world)
        if isinstance(self.dataset, PackedMemmapDataset):
            # flat memory-mapped bit arrays: whole batches gathered with three fancy-index reads in this process
            # (~0.5 M bars/s measured), no worker; batch_size counts BARS here (an .npz item holds several)
            self.dataloader = _MemmapLoader(self.dataset, self.batch_size, self.rank, self.world, config.pin_memory)
        else:
            self.dataloader = DataLoader(torch.utils.data.Subset(self.dataset, self.indices),
                                         batch_size=self.batch_size, shuffle=False, num_workers=1,
                                         pin_memory=config.pin_memory, collate_fn=self.make_batch)

        self.manual_seed = random.randint(1, 10000)
        torch.manual_seed(self.manual_seed)
        torch.cuda.manual_seed_all(self.manual_seed)
        random.seed(self.manual_seed)

        self.generator = Model(vae_head=getattr(config, "vae_head", False),
                               refiner=getattr(config, "refiner", False)).to(self.device)
        flat = self.generator.flatten_parameters()
        self.reducer = None
        if self.world > 1:
            self.reducer = parallel.GradReducer.for_model(self.generator, flat, getattr(config, "bucket_mb", 64))
        self.lr_gen1 = config.learning_rate
        self.opt_gen1 = GeneratorTrainer(self.generator, lr=self.lr_gen1, reducer=self.reducer,
                                         micro_bars=getattr(config, "micro_bars", 0))
        self.scheduler_gen1 = _Plateau(factor=0.8, cooldown=6)
        self.iteration = 0
        self.epoch = 0
        self.load_checkpoint(config.checkpoint_file)
        if self.reducer is not None:                      # rank 0's weights / optimiser state win (horovod :130-134)
            self.reducer.broadcast_parameters(0, trainer=self.opt_gen1)
            self.lr_gen1 = self.opt_gen1.lr
            self._sync_host_state()
        self.summary = None
        if self.rank == 0:
            os.makedirs(os.path.join(config.root_path, config.summary_dir), exist_ok=True)
            self.summary = open(os.path.join(config.root_path, config.summary_dir, "scalars.jsonl"), "a")
            print("Number of generator parameters: {}".format(sum(p.numel() for p in self.generator.parameters())))

    def _sync_host_state(self):
        """epoch counter and LR-scheduler state of rank 0 (the only rank that is guaranteed to have read a checkpoint)"""
        import torch.distributed as dist
        st = self.scheduler_gen1
        v = torch.tensor([float(self.epoch), st.best if st.best != float("inf") else -1.0, float(st.bad), float(st.cool)],
                         dtype=torch.float64, device=self.device)
        dist.broadcast(v, src=0)
        self.epoch = int(v[0].item())
        st.best = float("inf") if v[1].item() < 0 else float(v[1].item())
        st.bad, st.cool = int(v[2].item()), int(v[3].item())

    def set_logger(self):
        logger = logging.getLogger("barGen")
        logger.setLevel(logging.DEBUG)
        if self.rank == 0 and not logger.handlers:
            h = logging.FileHandler(filename="train_epoch.log")
            h.setFormatter(logging.Formatter("%(asctime)s - %(name)s - %(levelname)s - %(message)s"))
            logger.addHandler(h)
        return logger

    def make_batch(self, samples):
        cat = lambda k: np.concatenate([s[k] for s in samples], axis=0)
        if "note_bits" in samples[0]:          # items already stored as bits (PackedNoteDataset): byte-level concat
            return collate_packed(samples)
        if getattr(self.config, "packed_input", False):
            # bit-packed batch (data/packed.py): 4320 B per sample across PCIe instead of 138 KB, expanded on the device
            return PackedBatch.from_arrays(cat("note"), cat("pre_note"), cat("pre_phrase"), cat("position"))
        return (torch.tensor(cat("note"), dtype=torch.float), torch.tensor(cat("pre_note"), dtype=torch.float),
                torch.tensor(cat("pre_phrase"), dtype=torch.float), torch.tensor(cat("position"), dtype=torch.long))

    # ---- checkpoints (agent/barGen.py:151-197) -----------------------------------------------------------
    def _ckpt_dir(self):
        return os.path.join(self.config.root_path, self.config.checkpoint_dir)

    def load_checkpoint(self, file_name):
        filename = os.path.join(self._ckpt_dir(), file_name)
        try:
            ck = torch.load(filename, map_location=self.device, weights_only=False)
        except OSError:
            if self.rank == 0:
                print("No checkpoint exists from '{}'. Skipping...".format(self._ckpt_dir()))
            return
        sd = {(k[len("module."):] if k.startswith("module.") else k): v for k, v in ck["generator_state_dict"].items()}
        own = self.generator.state_dict()       # refiner.* only into Model(refiner=True) and only where shapes agree
        sd = {k: v for k, v in sd.items() if not k.startswith("refiner.") or (k in own and tuple(own[k].shape) == tuple(v.shape))}
        self.generator.load_state_dict(sd, strict=False)
        opt = ck.get("gen_optimizer1")
        if isinstance(opt, dict) and ("exp_avg" in opt or "param_groups" in opt):   # ours, or torch.optim.Adam's (reference)
            self.opt_gen1.load_state_dict(opt)
            self.lr_gen1 = self.opt_gen1.lr
        self.epoch = ck.get("epoch", 0)
        sch = ck.get("scheduler_gen1")                   # not in reference checkpoints (it never restores its schedulers)
        if isinstance(sch, dict):
            self.scheduler_gen1.best, self.scheduler_gen1.bad, self.scheduler_gen1.cool = sch["best"], sch["bad"], sch["cool"]

    def save_checkpoint(self, file_name, epoch):
        if self.rank != 0:
            return
        os.makedirs(self._ckpt_dir(), exist_ok=True)
        tmp_name = os.path.join(self._ckpt_dir(), "checkpoint_{}.pth.tar".format(epoch))
        gen_sd = {"module." + k: v.detach().clone() for k, v in self.generator.state_dict().items()}
        # gen_optimizer1/2 in torch.optim.Adam.state_dict() form, as the reference stores them (agent/barGen.py:176-177): a
        # reference-side torch.optim.Adam.load_state_dict accepts it.  This agent trains the generator alone, so the
        # discriminator entries of the reference's dictionary (:178-186) are not written -- its load_checkpoint indexes
        # them unconditionally and needs them added (agent/barGen_with_gan.py here writes all of them).
        opt_sd = self.opt_gen1.torch_state_dict()
        st = self.scheduler_gen1
        state = {"epoch": self.epoch, "generator_state_dict": gen_sd, "gen_optimizer1": opt_sd, "gen_optimizer2": opt_sd,
                 "lr_gen": self.lr_gen1, "scheduler_gen1": {"best": st.best, "bad": st.bad, "cool": st.cool}}
        torch.save(state, tmp_name)
        shutil.copyfile(tmp_name, os.path.join(self._ckpt_dir(), file_name))

    # ---- training ---------------------------------------------------------------------------------------
    def run(self):
        try:
            self.train()
        except KeyboardInterrupt:
            print("You have entered CTRL+C.. Wait to finalize")

    def train(self):
        for _ in range(self.config.epoch):
            self.epoch += 1
            self.train_epoch()
            if self.epoch > self.pretraining_step_size + 50:
                self.save_checkpoint(self.config.checkpoint_file, self.epoch)

    def train_epoch(self):
        self.generator.train()
        self.opt_gen1.is_pretraining = self.epoch <= self.pretraining_step_size
        avg_gen_loss = AverageMeter()
        dev_sum, n = torch.zeros((), device=self.device), 0
        # fp32 4-tuples or PackedBatch from the loader; the next batch's H2D copy overlaps the current step
        for batch in self.opt_gen1.prefetch(self.dataloader):
            self.iteration += 1
            dev_sum += self.opt_gen1.step_batch(batch)                                  # stays on the device
            n += 1
        tot = torch.stack((dev_sum.double(), torch.tensor(float(n), dtype=torch.float64, device=self.device)))
        if self.world > 1:
            # every rank feeds the plateau scheduler the SAME epoch mean: with per-shard means the ranks cross the
            # threshold / patience in different epochs, their learning rates diverge and the replicas drift apart
            torch.distributed.all_reduce(tot)
        tot = tot.tolist()                                                              # one D2H read per epoch
        if tot[1] > 0:
            avg_gen_loss.update(tot[0] / tot[1], int(tot[1]))
        self.lr_gen1 = self.opt_gen1.lr = self.scheduler_gen1.step(avg_gen_loss.val, self.opt_gen1.lr)
        if self.summary is not None:
            tag = "pre_train/Generator_loss" if self.opt_gen1.is_pretraining else "train/Generator_loss"
            self.summary.write(json.dumps({"tag": tag, "value": avg_gen_loss.val, "iteration": self.iteration,
                                           "epoch": self.epoch, "lr": self.lr_gen1}) + "\n")
            self.summary.flush()
            self.logger.debug("pre_train lr: {}".format(self.lr_gen1))
        return avg_gen_loss.val

    def generate(self, music_length=2, songs=1, seed=0, sampler="threshold", temperature=1.0, primer=None,
                 latent_prior=None):
        """per-epoch sample generation of agent/barGen2.py:316-336 (same loop as maker_bar.py); ``latent_prior``
        (prior.LatentPrior fitted to this generator's encoder) draws the latents instead of N(0, I)"""
        g = torch.Generator(device=self.device).manual_seed(seed)
        if latent_prior is not None:
            lat = latent_prior.sample(music_length * 4, songs, g)
        else:
            lat = torch.randn(music_length * 4, songs, 1152, device=self.device, generator=g)
        return sample_songs(self.generator, lat, music_length, sampler=sampler, temperature=temperature,
                            seed=g.initial_seed(), primer=primer)
