"""Adversarial trainer (reference: agent/barGen_with_gan.py -- BASELINE config 4): generator (graph/model_with_gan.Model) +
convolutional BarDiscriminator + BarFeatureDiscriminator + the two latent (z) discriminators, with the reference's three
per-iteration schedules:

  train_pretrain (:351-379)  BCE reconstruction step of the generator (epochs <= pretraining_step_size)
  train_wae      (:381-460)  every other iteration a z-discriminator step (generator frozen, one extra generator forward),
                             then a generator step: BCE with label smoothing + three adversarial terms on z / pre_z / pf
  train_gan      (:462-537)  every other iteration a bar / feature-discriminator step on (pre_note | note) vs (pre_note |
                             generated), then a generator step FROM NOISE (``Model(noise, ..., False)``) against both

and the phase flipping of ``train_epoch`` (:297-305: 50 WAE epochs, then 100 GAN epochs, alternating).  Label conventions
are the reference's (real -> fake_target, generated -> valid_target in the discriminator steps).

``config.gan_schedule = "horovod"`` selects the per-iteration schedule of agent/barGen_horovod.py instead (:312-324):
EVERY iteration a ``train_discriminator`` step of all four discriminators on one frozen-generator forward (:380-432), then a
generator step -- ``train_wae_only`` (:510-553: the generator half of train_wae) or, in the GAN phase, ``train_add_gan``
(:555-607: BCE x 1.1 + the three z terms + 0.8 x the two from-noise adversarial terms, two generator forwards, ONE backward
through both) -- with its 40 / 160-epoch phase lengths (:336-341).

B200 mapping: every module's parameters live in one flat fp32 bucket (engine.FlatParams) -> one fused Adam launch per
optimiser; one process per GPU, gradients of whichever module trained are all-reduced over NCCL before its Adam step
(``GradReducer(overlap=False)`` for the generator: its encoder runs up to three backward passes per step here, so the
per-segment overlap of the pre-training step does not apply).  BatchNorm statistics of the BarDiscriminator are per rank, as
in the reference (no SyncBN, SURVEY.md section 8e).  Checkpoints carry all ten reference keys (:195-213), optimiser states
in ``torch.optim.Adam.state_dict()`` form."""
import json
import os
import random
import shutil

import numpy as np
import torch
import torch.distributed as dist
from torch.utils.data import DataLoader

from .. import engine, parallel
from ..data.bar_dataset import NoteDataset, SyntheticBars
from ..graph.bar_discriminator import BarDiscriminator
from ..graph.bar_discriminator_with_feature import BarFeatureDiscriminator
from ..graph.loss.bar_loss import DLoss, Loss
from ..graph.model_with_gan import Model
from ..graph.z_discriminator import BarZDiscriminator, PhraseZDiscriminator
from ..maker_bar import sample_songs
from .barGen import _Plateau


class FlatAdam:
    """torch.optim.Adam(module.parameters(), lr) on the module's flat bucket: one bvae_adam_step launch (+ one repack of the
    bf16 GEMM operands); data-parallel gradient SUM over ranks first, the 1/world average folded into the step."""

    def __init__(self, module, lr, reducer=None):
        self.module, self.lr, self.reducer = module, lr, reducer
        self.flat = engine.flatten(module)
        self.step_count = 0

    def zero_grad(self):
        self.flat.attach_grads(zero=True)

    def step(self):
        scale = 1.0
        if self.reducer is not None:
            scale = self.reducer.finish()
        elif dist.is_initialized() and dist.get_world_size() > 1:
            dist.all_reduce(self.flat.grad)
            scale = 1.0 / dist.get_world_size()
        self.step_count += 1
        engine.adam_step(self.flat, self.lr, self.step_count, grad_scale=scale)

    def state_dict(self):
        """torch.optim.Adam.state_dict() form (what the reference stores, agent/barGen_with_gan.py:197-212)"""
        flat, state = self.flat, {}
        if flat.exp_avg is not None:
            for i, (p, o) in enumerate(zip(flat.params, flat.offsets)):
                n = p.numel()
                state[i] = {"step": torch.tensor(float(self.step_count)), "exp_avg": flat.exp_avg[o:o + n].view(p.shape).clone(),
                            "exp_avg_sq": flat.exp_avg_sq[o:o + n].view(p.shape).clone()}
        return {"state": state, "param_groups": [{"lr": self.lr, "betas": (0.9, 0.999), "eps": 1e-8, "weight_decay": 0,
                                                  "amsgrad": False, "params": list(range(len(flat.params)))}]}

    def load_state_dict(self, sd):
        flat = self.flat
        group = sd["param_groups"][0]
        self.lr = group.get("lr", self.lr)
        ids = list(group["params"])
        m, v, step = torch.zeros_like(flat.data), torch.zeros_like(flat.data), 0
        for i, (p, o) in enumerate(zip(flat.params, flat.offsets)):
            st = sd["state"].get(ids[i]) if i < len(ids) else None
            if st is None:
                continue
            if tuple(st["exp_avg"].shape) != tuple(p.shape):
                raise ValueError("optimizer state %d has shape %s, parameter has %s" % (i, tuple(st["exp_avg"].shape), tuple(p.shape)))
            n = p.numel()
            m[o:o + n].copy_(st["exp_avg"].reshape(-1).to(m.device))
            v[o:o + n].copy_(st["exp_avg_sq"].reshape(-1).to(m.device))
            step = max(step, int(st["step"]))
        if sd["state"]:
            flat.exp_avg, flat.exp_avg_sq, self.step_count = m, v, step


def free(module):
    for p in module.parameters():
        p.requires_grad = True


def frozen(module):
    for p in module.parameters():
        p.requires_grad = False


class BarGen(object):
    def __init__(self, config, dataset=None):
        self.config = config
        self.flag_gan = False
        self.train_count = 0
        self.pretraining_step_size = config.pretraining_step_size
        self.batch_size = config.batch_size
        self.rank, self.world, self.local_rank = parallel.init_from_env()
        torch.cuda.set_device(self.local_rank)
        self.device = dev = torch.device("cuda", self.local_rank)

        data_dir = os.path.join(config.root_path, config.data_path)
        if dataset is not None:
            self.dataset = dataset
        elif os.path.isdir(data_dir):
            self.dataset = NoteDataset(config.root_path, config)
        elif getattr(config, "synthetic", False):
            self.dataset = SyntheticBars(64, 4, self.batch_size)
        else:
            raise FileNotFoundError("no dataset directory %r; set config.synthetic = True to train on random bars" % data_dir)
        self.indices = parallel.shard_indices(len(self.dataset), self.rank, self.world)
        self.dataloader = DataLoader(torch.utils.data.Subset(self.dataset, self.indices), batch_size=self.batch_size,
                                     shuffle=False, num_workers=1, pin_memory=config.pin_memory, collate_fn=self.make_batch)

        self.manual_seed = random.randint(1, 10000)
        torch.manual_seed(self.manual_seed)
        torch.cuda.manual_seed_all(self.manual_seed)
        random.seed(self.manual_seed)

        self.generator = Model().to(dev)
        self.discriminator = BarDiscriminator().to(dev)
        self.discriminator_feature = BarFeatureDiscriminator().to(dev)
        self.z_discriminator_phrase = PhraseZDiscriminator().to(dev)
        self.z_discriminator_bar = BarZDiscriminator().to(dev)
        self.loss_generator, self.loss_disc = Loss(), DLoss()
        self.loss_feature_disc, self.loss_bar, self.loss_phrase = DLoss(), DLoss(), DLoss()

        lr = config.learning_rate
        gflat = self.generator.flatten_parameters()
        self.reducer = parallel.GradReducer.for_model(self.generator, gflat, getattr(config, "bucket_mb", 64),
                                                      overlap=False) if self.world > 1 else None
        self.opt_generator = FlatAdam(self.generator, lr, self.reducer)
        self.opt_discriminator = FlatAdam(self.discriminator, lr)
        self.opt_discriminator_feature = FlatAdam(self.discriminator_feature, lr)
        self.opt_Zdiscriminator_bar = FlatAdam(self.z_discriminator_bar, lr)
        self.opt_Zdiscriminator_phrase = FlatAdam(self.z_discriminator_phrase, lr)
        self._opts = {"generator": self.opt_generator, "discriminator": self.opt_discriminator,
                      "discriminator_feature": self.opt_discriminator_feature,
                      "z_discriminator_bar": self.opt_Zdiscriminator_bar,
                      "z_discriminator_phrase": self.opt_Zdiscriminator_phrase}
        self._sched = {k: _Plateau(factor=0.8, cooldown=6) for k in self._opts}

        self.iteration = 0
        self.epoch = 0
        self.load_checkpoint(config.checkpoint_file)
        if self.world > 1:                          # rank 0's weights win (agent/barGen_horovod.py:130-134), all five modules
            for opt in self._opts.values():
                dist.broadcast(opt.flat.data, src=0)
            for m in (self.discriminator,):         # BatchNorm buffers too
                for b in m.buffers():
                    dist.broadcast(b, src=0)
            engine.bump_param_epoch()
        self.summary = None
        if self.rank == 0:
            os.makedirs(os.path.join(config.root_path, config.summary_dir), exist_ok=True)
            self.summary = open(os.path.join(config.root_path, config.summary_dir, "scalars.jsonl"), "a")

    def make_batch(self, samples):
        cat = lambda k: np.concatenate([s[k] for s in samples], axis=0)
        return (torch.tensor(cat("note"), dtype=torch.float), torch.tensor(cat("pre_note"), dtype=torch.float),
                torch.tensor(cat("pre_phrase"), dtype=torch.float), torch.tensor(cat("position"), dtype=torch.long))

    # ---- checkpoints (agent/barGen_with_gan.py:169-218) -----------------------------------------------------
    _KEYS = (("generator", "generator_state_dict", "generator_optimizer"),
             ("discriminator", "discriminator_state_dict", "disc_optimizer"),
             ("discriminator_feature", "discriminator_feature_state_dict", "disc_feature_optimizer"),
             ("z_discriminator_bar", "z_discriminator_bar_state_dict", "opt_Zdiscriminator_bar_optimizer"),
             ("z_discriminator_phrase", "z_discriminator_phrase_state_dict", "opt_Zdiscriminator_phrase_optimizer"))

    def _ckpt_dir(self):
        return os.path.join(self.config.root_path, self.config.checkpoint_dir)

    def load_checkpoint(self, file_name):
        try:
            ck = torch.load(os.path.join(self._ckpt_dir(), file_name), map_location=self.device, weights_only=False)
        except OSError:
            if self.rank == 0:
                print("No checkpoint exists from '{}'. Skipping...".format(self._ckpt_dir()))
            return
        for name, sd_key, opt_key in self._KEYS:
            sd = {(k[len("module."):] if k.startswith("module.") else k): v for k, v in ck[sd_key].items()}
            getattr(self, name).load_state_dict(sd)
            self._opts[name].load_state_dict(ck[opt_key])
        engine.bump_param_epoch()
        self.epoch = ck.get("epoch", self.epoch)

    def save_checkpoint(self, file_name, epoch):
        if self.rank != 0:
            return
        os.makedirs(self._ckpt_dir(), exist_ok=True)
        tmp_name = os.path.join(self._ckpt_dir(), "checkpoint_{}.pth.tar".format(epoch))
        state = {"epoch": self.epoch}
        for name, sd_key, opt_key in self._KEYS:
            # nn.DataParallel's ``module.`` prefix, as the reference's files carry it (:108-112,196)
            state[sd_key] = {"module." + k: v.detach().clone() for k, v in getattr(self, name).state_dict().items()}
            state[opt_key] = self._opts[name].state_dict()
        torch.save(state, tmp_name)
        shutil.copyfile(tmp_name, os.path.join(self._ckpt_dir(), file_name))

    # ---- training loop (agent/barGen_with_gan.py:219-349) ----------------------------------------------------
    def run(self):
        try:
            self.train()
        except KeyboardInterrupt:
            print("You have entered CTRL+C.. Wait to finalize")

    def train(self):
        for _ in range(self.config.epoch):
            self.epoch += 1
            self.train_epoch()
            if self.epoch > self.pretraining_step_size + 20:
                self.save_checkpoint(self.config.checkpoint_file, self.epoch)

    def train_epoch(self):
        if self.epoch > self.pretraining_step_size:
            self.train_count += 1
        dev = self.device
        horovod = getattr(self.config, "gan_schedule", "with_gan") == "horovod"
        meters = {k: [torch.zeros((), device=dev), 0] for k in self._opts}     # running loss sums stay on the device

        def upd(name):
            def f(loss):
                meters[name][0] += loss.detach()
                meters[name][1] += 1
            return f

        for curr_it, (note, pre_note, pre_phrase, position) in enumerate(self.dataloader):
            self.iteration += 1
            note, pre_note = note.to(dev, non_blocking=True), pre_note.to(dev, non_blocking=True)
            pre_phrase, position = pre_phrase.to(dev, non_blocking=True), position.to(dev, non_blocking=True)
            valid_target = torch.ones(note.size(0), device=dev)
            fake_target = torch.zeros(note.size(0), device=dev)
            if self.epoch <= self.pretraining_step_size:
                self.train_pretrain(note, pre_note, pre_phrase, position, upd("generator"))
            elif horovod:                                   # agent/barGen_horovod.py:312-324
                self.train_discriminator(note, pre_note, pre_phrase, position, upd("z_discriminator_bar"),
                                         upd("z_discriminator_phrase"), upd("discriminator"),
                                         upd("discriminator_feature"), fake_target, valid_target)
                if self.flag_gan:
                    self.train_add_gan(note, pre_note, pre_phrase, position, upd("generator"), valid_target)
                else:
                    self.train_wae_only(note, pre_note, pre_phrase, position, upd("generator"), valid_target)
            elif self.flag_gan:
                self.train_gan(note, pre_note, pre_phrase, position, upd("generator"), upd("discriminator"),
                               upd("discriminator_feature"), fake_target, valid_target, curr_it)
            else:
                self.train_wae(note, pre_note, pre_phrase, position, upd("generator"), upd("z_discriminator_bar"),
                               upd("z_discriminator_phrase"), fake_target, valid_target, curr_it)

        gan_len, wae_len = (160, 40) if horovod else (100, 50)      # barGen_horovod.py:336-341 / barGen_with_gan.py:297-305
        if self.flag_gan and self.train_count >= gan_len:
            self.flag_gan, self.train_count = not self.flag_gan, 0
        elif not self.flag_gan and self.train_count >= wae_len:
            self.flag_gan, self.train_count = not self.flag_gan, 0

        # epoch means, identical on every rank (one all-reduce of 10 numbers), then the plateau schedulers (:337-342)
        tot = torch.stack([torch.stack((meters[k][0].double(), torch.tensor(float(meters[k][1]), dtype=torch.float64,
                                                                           device=dev))) for k in self._opts])
        if self.world > 1:
            dist.all_reduce(tot)
        tot = tot.tolist()
        means = {k: (t[0] / t[1] if t[1] > 0 else 0.0) for k, t in zip(self._opts, tot)}
        for k, opt in self._opts.items():
            if k == "generator" or self.epoch > self.pretraining_step_size:
                opt.lr = self._sched[k].step(means[k], opt.lr)
        if self.summary is not None:
            self.summary.write(json.dumps({"epoch": self.epoch, "iteration": self.iteration, "gan_phase": self.flag_gan,
                                           "loss": means, "lr": {k: o.lr for k, o in self._opts.items()}}) + "\n")
            self.summary.flush()
        return means

    def _modes(self, train):
        for name in self._opts:
            getattr(self, name).train(name in train)

    def train_pretrain(self, note, pre_note, pre_phrase, position, avg_generator_loss):
        self._modes({"generator"})
        self.opt_generator.zero_grad()
        free(self.generator)
        for m in (self.discriminator, self.discriminator_feature, self.z_discriminator_bar, self.z_discriminator_phrase):
            frozen(m)
        gen_note, z, pre_z, phrase_feature, _ = self.generator(note, pre_note, pre_phrase, position)
        loss = self.loss_generator(gen_note, note, True)
        loss.backward()
        self.opt_generator.step()
        avg_generator_loss(loss)
        return gen_note[:3]

    def train_wae(self, note, pre_note, pre_phrase, position, avg_generator_loss, avg_barZ_disc_loss, avg_phraseZ_disc_loss,
                  fake_target, valid_target, curr_it):
        self._modes({"generator", "z_discriminator_bar", "z_discriminator_phrase"})
        dev = note.device
        if (self.epoch + curr_it) % 2:
            # ---- z discriminators (generator frozen: its forward saves nothing) :389-424
            self.opt_Zdiscriminator_bar.zero_grad()
            self.opt_Zdiscriminator_phrase.zero_grad()
            free(self.z_discriminator_bar)
            free(self.z_discriminator_phrase)
            for m in (self.generator, self.discriminator, self.discriminator_feature):
                frozen(m)
            _, z, pre_z, phrase_feature, _ = self.generator(note, pre_note, pre_phrase, position)
            phrase_fake = torch.randn(phrase_feature.size(0), phrase_feature.size(1), device=dev) * self.config.sigma
            d_phrase_fake = self.z_discriminator_phrase(phrase_fake).view(-1)
            d_phrase_real = self.z_discriminator_phrase(phrase_feature).view(-1)
            phraseZ_disc_loss = self.loss_phrase(d_phrase_real, fake_target) + self.loss_phrase(d_phrase_fake, valid_target)
            bar_fake = torch.randn(z.size(0), z.size(1), device=dev) * self.config.sigma
            d_bar_fake = self.z_discriminator_bar(bar_fake).view(-1)
            d_bar_real = self.z_discriminator_bar(z).view(-1)
            barZ_disc_loss = self.loss_bar(d_bar_real, fake_target) + self.loss_bar(d_bar_fake, valid_target)
            phraseZ_disc_loss.backward()
            barZ_disc_loss.backward()
            self.opt_Zdiscriminator_bar.step()
            self.opt_Zdiscriminator_phrase.step()
            avg_barZ_disc_loss(barZ_disc_loss)
            avg_phraseZ_disc_loss(phraseZ_disc_loss)
        # ---- generator :426-452
        self.opt_generator.zero_grad()
        free(self.generator)
        for m in (self.z_discriminator_bar, self.z_discriminator_phrase, self.discriminator, self.discriminator_feature):
            frozen(m)
        gen_note, z, pre_z, phrase_feature, _ = self.generator(note, pre_note, pre_phrase, position)
        loss = self.loss_phrase(self.z_discriminator_phrase(phrase_feature).view(-1), valid_target)
        loss = loss + self.loss_bar(self.z_discriminator_bar(z).view(-1), valid_target) + \
            self.loss_bar(self.z_discriminator_bar(pre_z).view(-1), valid_target)
        loss = loss + self.loss_generator(gen_note, note, False)
        loss.backward()
        self.opt_generator.step()
        avg_generator_loss(loss)
        return gen_note[:3]

    def train_gan(self, note, pre_note, pre_phrase, position, avg_generator_loss, avg_discriminator_loss,
                  avg_feature_discriminator_loss, fake_target, valid_target, curr_it):
        self._modes({"generator", "discriminator", "discriminator_feature"})
        dev = note.device
        if (self.epoch + curr_it) % 2:
            # ---- bar / feature discriminators :470-504
            self.opt_discriminator.zero_grad()
            self.opt_discriminator_feature.zero_grad()
            free(self.discriminator)
            free(self.discriminator_feature)
            for m in (self.generator, self.z_discriminator_bar, self.z_discriminator_phrase):
                frozen(m)
            gen_note, z, pre_z, phrase_feature, gen_z = self.generator(note, pre_note, pre_phrase, position)
            fake_note = torch.cat((pre_note, gen_note), dim=2)
            real_note = torch.cat((pre_note, note), dim=2)
            d_note_fake = self.discriminator(fake_note).view(-1)
            d_note_real = self.discriminator(real_note).view(-1)
            note_disc_loss = self.loss_disc(d_note_real, fake_target) + self.loss_disc(d_note_fake, valid_target)
            d_feature_fake = self.discriminator_feature(gen_z).view(-1)
            d_feature_real = self.discriminator_feature(z).view(-1)
            feature_disc_loss = self.loss_disc(d_feature_real, fake_target) + self.loss_disc(d_feature_fake, valid_target)
            note_disc_loss.backward()
            feature_disc_loss.backward()
            self.opt_discriminator.step()
            self.opt_discriminator_feature.step()
            avg_discriminator_loss(note_disc_loss)
            avg_feature_discriminator_loss(feature_disc_loss)
        # ---- generator, from noise :506-531
        self.opt_generator.zero_grad()
        free(self.generator)
        for m in (self.discriminator, self.discriminator_feature, self.z_discriminator_bar, self.z_discriminator_phrase):
            frozen(m)
        noise = torch.randn(note.size(0), 1152, device=dev) * 1.5
        gen_note, gen_z = self.generator(noise, pre_note, pre_phrase, position, False)
        d_note_fake = self.discriminator(torch.cat((pre_note, gen_note), dim=2)).view(-1)
        loss = self.loss_disc(d_note_fake, valid_target)
        loss = loss + self.loss_disc(self.discriminator_feature(gen_z).view(-1), valid_target)
        loss.backward()
        self.opt_generator.step()
        avg_generator_loss(loss)
        return gen_note[:3]

    # ---- the per-iteration schedule of agent/barGen_horovod.py ------------------------------------------------
    def train_discriminator(self, note, pre_note, pre_phrase, position, avg_barZ_disc_loss, avg_phraseZ_disc_loss,
                            avg_discriminator_loss, avg_feature_discriminator_loss, fake_target, valid_target):
        """agent/barGen_horovod.py:380-432: one frozen-generator forward feeds all four discriminators"""
        self._modes(set(self._opts))
        dev = note.device
        discs = (self.discriminator, self.discriminator_feature, self.z_discriminator_bar, self.z_discriminator_phrase)
        opts = (self.opt_discriminator, self.opt_discriminator_feature, self.opt_Zdiscriminator_bar,
                self.opt_Zdiscriminator_phrase)
        for o in opts:
            o.zero_grad()
        for m in discs:
            free(m)
        frozen(self.generator)
        gen_note, z, pre_z, phrase_feature, gen_z = self.generator(note, pre_note, pre_phrase, position)
        phrase_fake = torch.randn(phrase_feature.size(0), phrase_feature.size(1), device=dev) * self.config.sigma
        phraseZ = self.loss_phrase(self.z_discriminator_phrase(phrase_feature).view(-1), fake_target) + \
            self.loss_phrase(self.z_discriminator_phrase(phrase_fake).view(-1), valid_target)
        bar_fake = torch.randn(z.size(0), z.size(1), device=dev) * self.config.sigma
        barZ = self.loss_bar(self.z_discriminator_bar(z).view(-1), fake_target) + \
            self.loss_bar(self.z_discriminator_bar(bar_fake).view(-1), valid_target)
        note_loss = self.loss_disc(self.discriminator(torch.cat((pre_note, note), dim=2)).view(-1), fake_target) + \
            self.loss_disc(self.discriminator(torch.cat((pre_note, gen_note), dim=2)).view(-1), valid_target)
        feat_loss = self.loss_disc(self.discriminator_feature(z).view(-1), fake_target) + \
            self.loss_disc(self.discriminator_feature(gen_z).view(-1), valid_target)
        for l in (phraseZ, barZ, note_loss, feat_loss):
            l.backward()
        for o in (self.opt_Zdiscriminator_bar, self.opt_Zdiscriminator_phrase, self.opt_discriminator,
                  self.opt_discriminator_feature):
            o.step()
        avg_barZ_disc_loss(barZ)
        avg_phraseZ_disc_loss(phraseZ)
        avg_discriminator_loss(note_loss)
        avg_feature_discriminator_loss(feat_loss)

    def _generator_wae_terms(self, note, pre_note, pre_phrase, position, valid_target, bce_weight):
        gen_note, z, pre_z, phrase_feature, _ = self.generator(note, pre_note, pre_phrase, position)
        loss = self.loss_phrase(self.z_discriminator_phrase(phrase_feature).view(-1), valid_target)
        loss = loss + self.loss_bar(self.z_discriminator_bar(z).view(-1), valid_target) + \
            self.loss_bar(self.z_discriminator_bar(pre_z).view(-1), valid_target)
        return gen_note, loss + self.loss_generator(gen_note, note, False) * bce_weight

    def _generator_step_modes(self):
        self._modes({"generator", "z_discriminator_bar", "z_discriminator_phrase"})       # :511-516,556-561
        self.opt_generator.zero_grad()
        free(self.generator)
        for m in (self.z_discriminator_bar, self.z_discriminator_phrase, self.discriminator, self.discriminator_feature):
            frozen(m)

    def train_wae_only(self, note, pre_note, pre_phrase, position, avg_generator_loss, valid_target):
        """agent/barGen_horovod.py:510-553"""
        self._generator_step_modes()
        gen_note, loss = self._generator_wae_terms(note, pre_note, pre_phrase, position, valid_target, 1.0)
        loss.backward()
        self.opt_generator.step()
        avg_generator_loss(loss)
        return gen_note[:3]

    def train_add_gan(self, note, pre_note, pre_phrase, position, avg_generator_loss, valid_target):
        """agent/barGen_horovod.py:555-607: reconstruction + latent terms AND the from-noise adversarial terms in one
        backward pass through two generator forwards"""
        self._generator_step_modes()
        _, loss = self._generator_wae_terms(note, pre_note, pre_phrase, position, valid_target, 1.1)
        noise = torch.randn(note.size(0), 1152, device=note.device) * 1.5
        gen_note, gen_z = self.generator(noise, pre_note, pre_phrase, position, False)
        loss = loss + self.loss_disc(self.discriminator(torch.cat((pre_note, gen_note), dim=2)).view(-1), valid_target) * 0.8
        loss = loss + self.loss_disc(self.discriminator_feature(gen_z).view(-1), valid_target) * 0.8
        loss.backward()
        self.opt_generator.step()
        avg_generator_loss(loss)
        return gen_note[:3]

    def generate(self, music_length=10, songs=1, seed=0, sampler="threshold", temperature=1.0, primer=None):
        """the per-epoch sample generation of :307-328 (same loop as maker_bar.py)"""
        g = torch.Generator(device=self.device).manual_seed(seed)
        lat = torch.randn(music_length * 4, songs, 1152, device=self.device, generator=g)
        self.generator.eval()
        return sample_songs(self.generator, lat, music_length, sampler=sampler, temperature=temperature,
                            seed=g.initial_seed(), primer=primer)
