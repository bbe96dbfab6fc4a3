"""CelebA 64x64 training step (celebA/EAD-GAN_celebA.py): generator, discriminator-with-Q-head,
three optimisation phases (G / D / info), three Adams.

The module classes are written exactly as the reference writes them -- ``nn.Sequential`` of
``nn.ConvTranspose2d / nn.BatchNorm2d / nn.ReLU / ...`` with the same constructor arguments
(celebA/EAD-GAN_celebA.py:67-138) -- but against ``eadgan_b200.nn``, so the state_dict layout
is the reference's and every forward/backward runs on the sm_100a kernels.
"""
from __future__ import annotations

import itertools

import torch

from .. import affine, chain, functional as Fn, parallel
from .. import nn as nn
from ..optim import Adam
from .._lib import ACT_SIGMOID

LATENT, CODE, CLASSES, CHANNELS = 200, 8, 10, 3  # argparse defaults, celebA/EAD-GAN_celebA.py:46-50


class Generator(torch.nn.Module):
    def __init__(self):
        super().__init__()
        widths = [LATENT + CODE + CLASSES, 1024, 512, 256, 128]
        layers = [nn.ConvTranspose2d(widths[0], widths[1], 4, 1, 0)]
        for cin, cout in zip(widths[1:-1], widths[2:]):
            layers += [nn.ConvTranspose2d(cin, cout, 4, stride=2, padding=1), nn.BatchNorm2d(cout), nn.ReLU()]
        layers += [nn.ConvTranspose2d(widths[-1], CHANNELS, 4, stride=2, padding=1), nn.Tanh()]
        self.conv_blocks = nn.Sequential(*layers)

    def forward(self, noise, labels, code):
        g_in = torch.cat((noise, labels, code), -1)
        return self.conv_blocks(g_in.view(g_in.size(0), g_in.size(1), 1, 1))


class Discriminator(torch.nn.Module):
    def __init__(self):
        super().__init__()
        widths = [3, 128, 256, 512, 1024]
        layers = []
        for cin, cout in zip(widths[:-1], widths[1:]):
            layers += [nn.spectral_norm(nn.Conv2d(cin, cout, 4, 2, 1)), nn.LeakyReLU(0.1, inplace=True)]
        layers.append(nn.Conv2d(widths[-1], 1 + CLASSES + CODE, 4, 1, 0))
        self.main = nn.Sequential(*layers)

    def forward(self, img):
        out = self.main(img).squeeze()
        if out.dim() == 1:  # batch of one: the reference's .squeeze() would break here (SURVEY appendix C.2)
            out = out.unsqueeze(0)
        validity = Fn.activation(out[:, 0], ACT_SIGMOID)
        cat = Fn.softmax(out[:, CODE + 1: CODE + 1 + CLASSES])
        cont = out[:, 1: CODE + 1]
        return cat, cont, validity


class CelebAStep:
    """Owns G, D, the three Adams and the loss modules; ``__call__`` runs one iteration."""

    def __init__(self, seed=0, device="cuda"):
        torch.manual_seed(seed)  # same construction order as the reference: G, then D (:172-173)
        self.G, self.D = Generator(), Discriminator()
        self.G.to(device)
        self.D.to(device)
        betas = (0.5, 0.999)
        self.opt_G = Adam(self.G.parameters(), lr=0.001, betas=betas)        # :211
        self.opt_D = Adam(self.D.parameters(), lr=0.0002, betas=betas)       # :212
        self.opt_info = Adam(itertools.chain(self.G.parameters(), self.D.parameters()), lr=0.0002, betas=betas)
        self.bce, self.mse, self.ce = nn.BCELoss(), nn.MSELoss(), nn.CrossEntropyLoss()
        self.device = torch.device(device)
        self._defer_D = None    # None: defer opt_D.step() under data parallelism only; True / False force it (see __call__)

    def optimizers(self):
        return [self.opt_G, self.opt_D, self.opt_info]

    @staticmethod
    def _snap(opt, rec, name):
        if rec is None:
            return
        ps = [p for g in opt.param_groups for p in g["params"]]
        rec.append({"name": name, "grads": [None if p.grad is None else p.grad.detach().clone() for p in ps]})

    @staticmethod
    def _after(opt, rec):
        if rec is not None:
            rec[-1]["params_after"] = [p.detach().clone() for g in opt.param_groups for p in g["params"]]

    def __call__(self, imgs, z, code, labels, record=None, after_phase=None):
        """imgs [B,3,64,64] in [-1,1]; z [B,200]; code [B,8]; labels [B] int64 -- all on the device.
        ``after_phase(i)`` (tests only) runs after the optimiser step of phase i = 0, 1."""
        G, D = self.G, self.D
        B = imgs.shape[0]
        valid = torch.ones(B, device=imgs.device)
        fake = torch.zeros(B, device=imgs.device)
        onehot = torch.zeros(B, CLASSES, device=imgs.device)
        onehot.scatter_(1, labels.view(-1, 1), 1.0)
        scaled = affine.stn(imgs, affine.celeba_matrix(code[:, :5])[:, 0:2])

        # D's weights do not change until opt_D.step(): the power iterations of its next three forwards (D(gen) below,
        # then the two of phase D) depend only on the weights and on u / v, so they are issued now, on a side stream,
        # and overlap G's forward instead of preceding every D conv stack on the critical path
        # Phase G differentiates THROUGH D but only opt_G steps: D is frozen for it, so D's weight gradients (which
        # the reference computes and then discards at :353) are never launched.  The weight tensors W / sigma are
        # produced by the prefetch, hence one prefetch with D frozen (phase G's forward) and two with D trainable
        chain.clear_prefetch(D.main)          # leftovers of an aborted step, if any
        # ... and so do the bf16 operand packs of both networks (the last opt_info.step() changed G and D): G's are
        # needed first, D's overlap G's forward
        chain.prefetch_packs(G)
        chain.prefetch_packs(D)
        chain.set_trainable(D, False)
        chain.prefetch_spectral_norm(D.main, 1)
        chain.set_trainable(D, True)
        chain.prefetch_spectral_norm(D.main, 2)

        # phase G -- :334-345
        self.opt_G.zero_grad()
        chain.set_trainable(D, False)
        gen = G(z, onehot, code)
        _, _, validity = D(gen)
        g_loss = self.bce(validity, valid)
        g_loss.backward()
        chain.set_trainable(D, True)
        # Optimiser steps are DEFERRED to the last point where nothing has read the weights they change (same
        # arithmetic, independent work reordered): phase D never touches G (it sees gen.detach(), computed above), so
        # opt_G.step() -- which under data parallelism first waits for the all-reduce of G's gradients -- runs after
        # phase D's backward, and that all-reduce overlaps the whole of phase D; under data parallelism opt_D.step()
        # runs after the info phase's G forward, which hides the all-reduce of D's last buckets (on one device it
        # stays where it is, and the side-stream work it releases -- D's operand packs and power iterations --
        # overlaps that G forward instead).  With a recorder or a test hook attached the reference's literal order
        # is kept.
        defer = record is None and after_phase is None
        defer_D = defer and (self._defer_D if self._defer_D is not None else parallel.get() is not None)
        if not defer:
            self._snap(self.opt_G, record, "G")
            self.opt_G.step()
            self._after(self.opt_G, record)
            if after_phase is not None:
                after_phase(0)

        # phase D -- :353-366
        self.opt_D.zero_grad()
        _, _, real_pred = D(scaled)
        _, _, fake_pred = D(gen.detach())
        d_loss = (self.bce(real_pred, valid) + self.bce(fake_pred, fake)) / 2
        d_loss.backward()
        if defer:
            self.opt_G.step()
            chain.prefetch_packs(G)
        if not defer_D:
            self._snap(self.opt_D, record, "D")
            self.opt_D.step()
            self._after(self.opt_D, record)
            if after_phase is not None:
                after_phase(1)
            chain.prefetch_packs(D)
            chain.prefetch_spectral_norm(D.main, 3)     # the info phase's three D forwards (weights fixed until opt_info.step)

        # phase info -- :375-401
        if not defer_D:
            self.opt_info.zero_grad()
        gen = G(z, onehot, code)
        if defer_D:
            self.opt_D.step()
            chain.prefetch_packs(D)
            chain.prefetch_spectral_norm(D.main, 3)
            self.opt_info.zero_grad()
        pred_label, pred_code, _ = D(gen)
        info = self.ce(pred_label, labels) + self.mse(pred_code, code)
        _, transform_code, _ = D(scaled)
        _, real_code, _ = D(imgs)
        info = info + self.mse(affine.celeba_relative_code(real_code, transform_code), code[:, :5])
        info.backward()
        self._snap(self.opt_info, record, "info")
        self.opt_info.step()
        self._after(self.opt_info, record)
        return {"g_loss": g_loss.detach(), "d_loss": d_loss.detach(), "info_loss": info.detach()}
