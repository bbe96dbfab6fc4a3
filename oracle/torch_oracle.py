"""TEST INFRASTRUCTURE ONLY (the oracle).  Never imported by eadgan_b200/.

Stand-alone restatement, in stock ``torch.nn`` on CPU (or any torch device), of the
reference's adversarial training step.  It exists because /root/reference does not
travel to the GPU box; it is pinned, in the build container, against the reference
scripts themselves executed by oracle/ref_runner.py (tests/test_oracle_pin.py) and
against the committed fixtures in tests/golden/ (generated from the *reference*, see
oracle/make_golden.py).  The reference has no tests or golden vectors of its own
(SURVEY.md section 4), so those self-generated fixtures are the pin.

Every function cites the reference lines it follows (paths relative to
/root/reference).  Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
cpu-baseline / ``--impl reference`` legs may import this module.
"""
from __future__ import annotations

import itertools
import math

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.nn.utils import spectral_norm

# --------------------------------------------------------------------------- #
# affine glue (utils_*.py)                                                    #
# --------------------------------------------------------------------------- #


def _eye_batch(n, like):
    return torch.eye(3, dtype=like.dtype, device=like.device).unsqueeze(0).repeat(n, 1, 1)


def _rot(theta):
    m = _eye_batch(theta.shape[0], theta)
    c, s = torch.cos(theta), torch.sin(theta)
    m[:, 0, 0] = c
    m[:, 0, 1] = -s
    m[:, 1, 0] = s
    m[:, 1, 1] = c
    return m


def _zoom(p, q):
    m = _eye_batch(p.shape[0], p)
    m[:, 0, 0] = p
    m[:, 1, 1] = q
    return m


def _shift(x, y):
    m = _eye_batch(x.shape[0], x)
    m[:, 0, 2] = x
    m[:, 1, 2] = y
    return m


def celeba_get_matrix(code5):
    """celebA/utils_rpqxy.py:25-38 (rescale) and :59-80 (R @ Z @ T)."""
    theta = code5[:, 0] * np.pi / 9
    p = code5[:, 1] * 0.2 + 1
    q = code5[:, 2] * 0.2 + 1
    x = code5[:, 3] * 0.1
    y = code5[:, 4] * 0.1
    return _rot(theta) @ _zoom(p, q) @ _shift(x, y)


def celeba_affine_regularizer(real_code, trans_code):
    """celebA/utils_rpqxy.py:82-116: closed-form recovery of the relative affine code."""
    rel = celeba_get_matrix(trans_code[:, :5]) @ torch.inverse(celeba_get_matrix(real_code[:, :5]))
    t1 = rel[:, 0, 0] * rel[:, 1, 0] - rel[:, 0, 1] * rel[:, 1, 1]
    t2 = rel[:, 0, 0] ** 2 + rel[:, 1, 1] ** 2 - rel[:, 0, 1] ** 2 - rel[:, 1, 0] ** 2
    th = 0.5 * torch.atan(2 * t1 / t2)
    p = rel[:, 0, 0] * torch.cos(th) + rel[:, 1, 0] * torch.sin(th)
    q = -rel[:, 0, 1] * torch.sin(th) + rel[:, 1, 1] * torch.cos(th)
    x = (rel[:, 0, 2] * torch.cos(th) + rel[:, 1, 2] * torch.sin(th)) / p
    y = (rel[:, 1, 2] * torch.cos(th) - rel[:, 0, 2] * torch.sin(th)) / q
    # celebA/utils_rpqxy.py:41-55 (inverse rescale)
    out = torch.stack((th / np.pi * 9, (p - 1) / 0.2, (q - 1) / 0.2, x / 0.1, y / 0.1), dim=1)
    return out.to(real_code.dtype)  # the reference's .float() (:116); dtype-preserving so an fp64 referee run works


def stn(img, theta23, padding_mode="border"):
    """transformation_2D.stn, celebA/EAD-GAN_celebA.py:149-153."""
    grid = F.affine_grid(theta23, img.size(), align_corners=False)
    return F.grid_sample(img, grid, padding_mode=padding_mode, align_corners=False)


# --------------------------------------------------------------------------- #
# CelebA (celebA/EAD-GAN_celebA.py)                                           #
# --------------------------------------------------------------------------- #


class CelebAGenerator(nn.Module):
    """celebA/EAD-GAN_celebA.py:67-102 (latent 200 + classes 10 + code 8 -> 3x64x64)."""

    def __init__(self, latent_dim=200, code_dim=8, n_classes=10, channels=3):
        super().__init__()
        d = latent_dim + code_dim + n_classes
        self.conv_blocks = nn.Sequential(
            nn.ConvTranspose2d(d, 1024, 4, 1, 0),
            nn.ConvTranspose2d(1024, 512, 4, stride=2, padding=1), nn.BatchNorm2d(512), nn.ReLU(),
            nn.ConvTranspose2d(512, 256, 4, stride=2, padding=1), nn.BatchNorm2d(256), nn.ReLU(),
            nn.ConvTranspose2d(256, 128, 4, stride=2, padding=1), nn.BatchNorm2d(128), nn.ReLU(),
            nn.ConvTranspose2d(128, channels, 4, stride=2, padding=1), nn.Tanh(),
        )

    def forward(self, noise, labels, code):
        x = torch.cat((noise, labels, code), -1)
        return self.conv_blocks(x.view(x.size(0), x.size(1), 1, 1))


class CelebADiscriminator(nn.Module):
    """celebA/EAD-GAN_celebA.py:105-138; channel 0 validity, 1..8 code, 9..18 class."""

    def __init__(self, code_dim=8, n_classes=10):
        super().__init__()
        self.code_dim, self.n_classes = code_dim, n_classes
        self.main = nn.Sequential(
            spectral_norm(nn.Conv2d(3, 128, 4, 2, 1)), nn.LeakyReLU(0.1, inplace=True),
            spectral_norm(nn.Conv2d(128, 256, 4, 2, 1)), nn.LeakyReLU(0.1, inplace=True),
            spectral_norm(nn.Conv2d(256, 512, 4, 2, 1)), nn.LeakyReLU(0.1, inplace=True),
            spectral_norm(nn.Conv2d(512, 1024, 4, 2, 1)), nn.LeakyReLU(0.1, inplace=True),
            nn.Conv2d(1024, 1 + n_classes + code_dim, 4, 1, 0),
        )

    def forward(self, img):
        out = self.main(img).squeeze()
        validity = torch.sigmoid(out[:, 0])
        cat = F.softmax(out[:, self.code_dim + 1: self.code_dim + 1 + self.n_classes], dim=1)
        cont = out[:, 1: self.code_dim + 1]
        return cat, cont, validity


def one_hot(labels, n, like):
    out = torch.zeros(labels.shape[0], n, dtype=like.dtype, device=like.device)
    out[torch.arange(labels.shape[0]), torch.as_tensor(labels, dtype=torch.long)] = 1.0
    return out


def sample_celeba(rs: np.random.RandomState, batch, latent_dim=200, code_dim=8, n_classes=10):
    """Host sampling in the reference's order, celebA/EAD-GAN_celebA.py:308-317."""
    z = rs.normal(0, 1, (batch, latent_dim))
    code = rs.uniform(-1, 1, (batch, code_dim))
    labels = rs.randint(0, n_classes, batch)
    return {"z": torch.tensor(z, dtype=torch.float32), "code": torch.tensor(code, dtype=torch.float32),
            "labels": torch.tensor(labels, dtype=torch.long)}


def build_celeba(seed=0, device="cpu", dtype=torch.float32):
    """Models + the three Adams of celebA/EAD-GAN_celebA.py:172-173,211-217.
    Construction order (G then D) after ``torch.manual_seed`` fixes the random init."""
    torch.manual_seed(seed)
    G, D = CelebAGenerator(), CelebADiscriminator()
    G.to(device=device, dtype=dtype)
    D.to(device=device, dtype=dtype)
    betas = (0.5, 0.999)
    st = {
        "G": G, "D": D,
        "opt_G": torch.optim.Adam(G.parameters(), lr=0.001, betas=betas),
        "opt_D": torch.optim.Adam(D.parameters(), lr=0.0002, betas=betas),
        "opt_info": torch.optim.Adam(itertools.chain(G.parameters(), D.parameters()), lr=0.0002, betas=betas),
    }
    return st


def _snap(opt):
    ps = [p for g in opt.param_groups for p in g["params"]]
    return [None if p.grad is None else p.grad.detach().clone() for p in ps]


def _params(opt):
    return [p.detach().clone() for g in opt.param_groups for p in g["params"]]


def _state(G, D):
    """full module state (weights, BN running stats, spectral-norm u/v) after a phase: lets a test restart
    the next phase of another implementation from THIS run's state (SURVEY.md section 7.3-1 iv)."""
    return {"G": {k: v.detach().clone() for k, v in G.state_dict().items()},
            "D": {k: v.detach().clone() for k, v in D.state_dict().items()}}


def step_celeba(st, imgs, draws, record=True, after_phase=None):
    """One iteration of celebA/EAD-GAN_celebA.py:297-401 on batch ``imgs`` [B,3,64,64].
    ``after_phase(i)`` (parity tests only) runs after the optimiser step of phase i = 0, 1: it lets a test restart
    the next phase from another run's state, exactly like the hook of eadgan_b200.steps.celeba.CelebAStep."""
    G, D = st["G"], st["D"]
    dev, dt = imgs.device, imgs.dtype
    B = imgs.shape[0]
    bce, mse, ce = nn.BCELoss(), nn.MSELoss(), nn.CrossEntropyLoss()
    valid = torch.ones(B, device=dev, dtype=dt)            # :302
    fake = torch.zeros(B, device=dev, dtype=dt)            # :303
    z = draws["z"].to(dev, dt)
    code = draws["code"].to(dev, dt)
    labels = draws["labels"].to(dev)
    label_input = one_hot(labels, 10, z)
    imgs = imgs.to(dt)
    A = celeba_get_matrix(code[:, :5])                      # :325
    scaled = stn(imgs, A[:, 0:2])                           # :327
    rec = {"phases": []}

    # ---- phase G  (:334-345)
    st["opt_G"].zero_grad()
    gen = G(z, label_input, code)
    _, _, validity = D(gen)
    g_loss = bce(validity, valid)
    g_loss.backward()
    if record:
        rec["phases"].append({"name": "G", "grads": _snap(st["opt_G"])})
    st["opt_G"].step()
    if record:
        rec["phases"][-1]["params_after"] = _params(st["opt_G"])
        rec["phases"][-1]["state_after"] = _state(G, D)
    if after_phase is not None:
        after_phase(0)

    # ---- phase D  (:353-366)
    st["opt_D"].zero_grad()
    _, _, real_pred = D(scaled)
    d_real = bce(real_pred, valid)
    _, _, fake_pred = D(gen.detach())
    d_fake = bce(fake_pred, fake)
    d_loss = (d_real + d_fake) / 2
    d_loss.backward()
    if record:
        rec["phases"].append({"name": "D", "grads": _snap(st["opt_D"])})
    st["opt_D"].step()
    if record:
        rec["phases"][-1]["params_after"] = _params(st["opt_D"])
        rec["phases"][-1]["state_after"] = _state(G, D)
    if after_phase is not None:
        after_phase(1)

    # ---- phase info  (:375-401)
    st["opt_info"].zero_grad()
    gen = G(z, label_input, code)
    pred_label, pred_code, _ = D(gen)
    info1 = ce(pred_label, labels) + mse(pred_code, code)   # CE on softmax output (:383)
    _, transform_code, _ = D(scaled)
    _, real_code, _ = D(imgs)
    pred_aff = celeba_affine_regularizer(real_code, transform_code)
    info_loss = info1 + mse(pred_aff, code[:, :5])
    info_loss.backward()
    if record:
        rec["phases"].append({"name": "info", "grads": _snap(st["opt_info"])})
    st["opt_info"].step()
    if record:
        rec["phases"][-1]["params_after"] = _params(st["opt_info"])

    rec["losses"] = {"g_loss": g_loss.item(), "d_loss": d_loss.item(), "info_loss": info_loss.item()}
    return rec


# --------------------------------------------------------------------------- #
# synthetic inputs (SURVEY.md section 8 d)                                    #
# --------------------------------------------------------------------------- #


def synth_celeba_images(batch, seed=0):
    g = torch.Generator().manual_seed(1000 + seed)
    return torch.rand(batch, 3, 64, 64, generator=g) * 2 - 1


def summarize(t: torch.Tensor):
    """Size-independent fingerprint of a tensor used by the golden fixtures."""
    t = t.detach().double().flatten()
    idx = torch.linspace(0, t.numel() - 1, steps=min(8, t.numel())).long()
    return {"sum": float(t.sum()), "l2": float(t.norm()), "absmax": float(t.abs().max()),
            "probe": [float(v) for v in t[idx]]}


# --------------------------------------------------------------------------- #
# dSprites stage 2 (dSprites/rp.py)                                           #
# --------------------------------------------------------------------------- #


def _conv_trunk(cin, slope, sn):
    wrap = spectral_norm if sn else (lambda m: m)
    layers = []
    for a, b in ((cin, 32), (32, 32), (32, 64), (64, 64)):
        layers += [wrap(nn.Conv2d(a, b, 4, 2, 1)), nn.LeakyReLU(slope, inplace=True)]
    return nn.Sequential(*layers)


class DSpritesEncoderPxy(nn.Module):
    """dSprites/rp.py:56-82 (frozen stage-1 encoder: zoom / position code)."""

    def __init__(self, channels=1, out_dim=3):
        super().__init__()
        self.conv_block = _conv_trunk(channels, 0.1, False)
        self.fc1 = nn.Linear(1024, out_dim)

    def forward(self, img):
        x = self.conv_block(img)
        return self.fc1(x.view(x.shape[0], -1))


class DSpritesDiscriminator(nn.Module):
    """dSprites/rp.py:85-114."""

    def __init__(self, channels=1):
        super().__init__()
        self.conv_block = _conv_trunk(channels, 0.2, True)
        self.fc1 = nn.Sequential(spectral_norm(nn.Linear(1024, 128)), nn.LeakyReLU(0.2, inplace=True))
        self.fc2 = nn.Linear(128, 1)

    def forward(self, img):
        x = self.conv_block(img)
        x = self.fc1(x.view(x.shape[0], -1))
        return torch.sigmoid(self.fc2(x))


class DSpritesGenerator(nn.Module):
    """dSprites/rp.py:118-152 (registration order: conv_block, fc1, fc2)."""

    def __init__(self, n_classes=3, code_dim=4, channels=1):
        super().__init__()
        blk = []
        for _ in range(3):
            blk += [nn.ConvTranspose2d(64, 64, 4, 2, 1), nn.BatchNorm2d(64), nn.ReLU()]
        blk.append(nn.ConvTranspose2d(64, channels, 4, 2, 1))
        self.conv_block = nn.Sequential(*blk)
        self.fc1 = nn.Sequential(nn.Linear(n_classes + code_dim, 128), nn.ReLU())
        self.fc2 = nn.Sequential(nn.Linear(128, 64 * 4 * 4), nn.ReLU())

    def forward(self, z_c):
        x = self.fc2(self.fc1(z_c))
        return torch.sigmoid(self.conv_block(x.view(x.shape[0], 64, 4, 4)))


class DSpritesEncoder(nn.Module):
    """dSprites/rp.py:155-190."""

    def __init__(self, n_classes=3, code_dim=4, channels=1):
        super().__init__()
        self.conv_block = _conv_trunk(channels, 0.2, True)
        self.fc1 = nn.Sequential(spectral_norm(nn.Linear(1024, 128)), nn.LeakyReLU(0.2, inplace=True))
        self.fc2 = nn.Sequential(spectral_norm(nn.Linear(128, 128)), nn.LeakyReLU(0.2, inplace=True))
        self.cat_layer = nn.Sequential(spectral_norm(nn.Linear(128, n_classes)), nn.Softmax(dim=1))
        self.cont_layer = nn.Sequential(spectral_norm(nn.Linear(128, code_dim)))

    def forward(self, img):
        x = self.conv_block(img)
        x = self.fc2(self.fc1(x.view(x.shape[0], -1)))
        return self.cat_layer(x), self.cont_layer(x)


def mutual_info_loss(c_given_x, c):
    """dSprites/rp.py:225-232 (eps inside both logs; the target's own entropy is added)."""
    eps = 1e-8
    cond = torch.mean(-torch.sum(torch.log(c_given_x + eps) * c, dim=1))
    ent = torch.mean(-torch.sum(torch.log(c + eps) * c, dim=1))
    return cond + ent


def dsprites_align_matrix(code3):
    """dSprites/utils_pxy.py:69-87 (get_matrix_pxy_align: translation only, zoom ignored)."""
    return _shift(code3[:, 1] * 0.1, code3[:, 2] * 0.1)


def dsprites_get_matrix(code4):
    """dSprites/utils_rp.py:38-59 (get_matrix_D) == :94-115 (get_matrix): R(theta) @ Z(p,p) @ T(x,y)."""
    theta = code4[:, 0] * np.pi / 9
    p = code4[:, 1] * 0.2 + 1
    return _rot(theta) @ _zoom(p, p) @ _shift(code4[:, 2] * 0.1, code4[:, 3] * 0.1)


def dsprites_affine_regularizer(real_code, trans_code):
    """dSprites/utils_rp.py:117-147."""
    rel = dsprites_get_matrix(trans_code[:, :4]) @ torch.inverse(dsprites_get_matrix(real_code[:, :4]))
    th = torch.atan((rel[:, 1, 0] - rel[:, 0, 1]) / (rel[:, 0, 0] + rel[:, 1, 1]))
    p = 0.5 * (torch.cos(th) * (rel[:, 0, 0] + rel[:, 1, 1]) + torch.sin(th) * (rel[:, 1, 0] - rel[:, 0, 1]))
    x = (rel[:, 0, 2] * torch.cos(th) + rel[:, 1, 2] * torch.sin(th)) / p
    y = (rel[:, 1, 2] * torch.cos(th) - rel[:, 0, 2] * torch.sin(th)) / p
    out = torch.stack((th / np.pi * 9, (p - 1) / 0.2, x / 0.1, y / 0.1), dim=1)
    return out.to(real_code.dtype)


def build_dsprites(seed=0, device="cpu", dtype=torch.float32, colored=False):
    """dSprites/rp.py:255-282 (colored_dSprites/rp_color.py:253-280): construction order encoder_pxy, encoder,
    discriminator, generator; the frozen Encoder_pxy then loads a checkpoint -- here a stand-in drawn from
    seed + 1000 (dsprites_pxy_state).  colored: 3 channels, 7-d code, Encoder_pxy emits 6, both Adams at
    opt.lr = 2e-4 (rp_color.py:39,275-280); gray: D 2e-4 (rp.py:277), info opt.lr = 1e-4 (rp.py:42,280-282)."""
    torch.manual_seed(seed)
    ch, cd, pd = (3, 7, 6) if colored else (1, 4, 3)
    Epxy, E = DSpritesEncoderPxy(ch, pd), DSpritesEncoder(3, cd, ch)
    D, G = DSpritesDiscriminator(ch), DSpritesGenerator(3, cd, ch)
    Epxy.load_state_dict(dsprites_pxy_state(seed, colored))
    Epxy.eval()
    for m in (Epxy, E, D, G):
        m.to(device=device, dtype=dtype)
    betas = (0.5, 0.999)
    return {"Epxy": Epxy, "E": E, "D": D, "G": G,
            "opt_D": torch.optim.Adam(D.parameters(), lr=0.0002, betas=betas),
            "opt_info": torch.optim.Adam(itertools.chain(G.parameters(), E.parameters()),
                                         lr=0.0002 if colored else 0.0001, betas=betas)}


def dsprites_pxy_state(seed=0, colored=False):
    """random-init stand-in for encoder_pxy_50000.pt / encoder_pxy_color_50000.pt (unavailable offline,
    SURVEY.md section 8c)."""
    g = torch.random.get_rng_state()
    torch.manual_seed(seed + 1000)
    net = DSpritesEncoderPxy(3, 6) if colored else DSpritesEncoderPxy()
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    torch.random.set_rng_state(g)
    return sd


def synth_dsprites_images(batch, seed=0):
    """binary {0,1} uint8 sprites [B,64,64]: one filled axis-aligned ellipse / square per image."""
    rs = np.random.RandomState(2000 + seed)
    yy, xx = np.mgrid[0:64, 0:64]
    out = np.zeros((batch, 64, 64), dtype=np.uint8)
    for b in range(batch):
        cx, cy = rs.uniform(20, 44, 2)
        r = rs.uniform(5, 12)
        if rs.rand() < 0.5:
            out[b] = (((xx - cx) / r) ** 2 + ((yy - cy) / (0.7 * r)) ** 2 <= 1).astype(np.uint8)
        else:
            out[b] = ((abs(xx - cx) <= r) & (abs(yy - cy) <= r)).astype(np.uint8)
    return torch.from_numpy(out)


def sample_dsprites(rs: np.random.RandomState, batch, code_dim=4, n_classes=3):
    """host draws in the reference's order: code, labels (phase D, dSprites/rp.py:389-394), then code,
    labels again (phase info, :424-431)."""
    d = {}
    for ph in ("d", "info"):
        d["code_" + ph] = torch.tensor(rs.uniform(-1, 1, (batch, code_dim)), dtype=torch.float32)
        d["labels_" + ph] = torch.tensor(rs.randint(0, n_classes, batch), dtype=torch.long)
    return d


def step_dsprites(st, img_u8, draws, record=True, after_phase=None):
    """One iteration of dSprites/rp.py:362-482 on ``img_u8`` uint8 [B,64,64].  ``after_phase(0)`` runs after the
    optimiser step of phase D, as in step_celeba."""
    Epxy, E, D, G = st["Epxy"], st["E"], st["D"], st["G"]
    dt = next(G.parameters()).dtype
    dev = next(G.parameters()).device
    bce, mse = nn.BCELoss(), nn.MSELoss()
    B = img_u8.shape[0]
    img = img_u8.unsqueeze(1).to(dev).to(dt)                                   # :369-370
    valid = torch.ones(B, 1, device=dev, dtype=dt)
    fake = torch.zeros(B, 1, device=dev, dtype=dt)
    rec = {"phases": []}

    def aligned():
        code = Epxy(img)                                                       # :374 (grad-tracked, frozen)
        inv = torch.inverse(dsprites_align_matrix(code))
        return stn(img, inv[:, 0:2])                                           # :375-377

    # ---- phase D  (:379-419)
    align_img = aligned()
    code = draws["code_d"].to(dev, dt)
    lab = one_hot(draws["labels_d"], 3, code)
    trans_img = stn(align_img, dsprites_get_matrix(code[:, :4])[:, 0:2])       # :399-400
    gen = G(torch.cat((lab, code), dim=1))
    d_real = D(trans_img)            # order matters: every D forward advances the spectral-norm u, v (:410-411)
    d_fake = D(gen.detach())
    d_loss = (bce(d_fake, fake) + bce(d_real, valid)) / 2
    st["opt_D"].zero_grad()
    d_loss.backward()
    if record:
        rec["phases"].append({"name": "D", "grads": _snap(st["opt_D"])})
    st["opt_D"].step()
    if record:
        rec["phases"][-1]["params_after"] = _params(st["opt_D"])
        rec["phases"][-1]["state_after"] = {k: {n: v.detach().clone() for n, v in st[k].state_dict().items()}
                                            for k in ("G", "D", "E")}
    if after_phase is not None:
        after_phase(0)

    # ---- phase info  (:424-482)
    code = draws["code_info"].to(dev, dt)
    lab = one_hot(draws["labels_info"], 3, code)
    gen = G(torch.cat((lab, code), dim=1))
    rec_cat, rec_cont = E(gen)
    g_loss = bce(D(gen), valid)
    cat_loss = mutual_info_loss(rec_cat, lab)
    cont_loss = mse(rec_cont, code)
    align_img = aligned()
    trans_img = stn(align_img, dsprites_get_matrix(code[:, :4])[:, 0:2])
    align_cat, align_cont = E(align_img)
    trans_cat, trans_cont = E(trans_img)
    affine_loss = mse(dsprites_affine_regularizer(align_cont, trans_cont), code)
    rel_cat_loss = mutual_info_loss(trans_cat, align_cat.detach())             # Variable(..., requires_grad=False)
    total = cat_loss + cont_loss + affine_loss + g_loss + rel_cat_loss
    st["opt_info"].zero_grad()
    total.backward()
    if record:
        rec["phases"].append({"name": "info", "grads": _snap(st["opt_info"])})
    st["opt_info"].step()
    if record:
        rec["phases"][-1]["params_after"] = _params(st["opt_info"])
    rec["losses"] = {"d_loss": d_loss.item(), "g_loss": g_loss.item(), "cat_loss": cat_loss.item(),
                     "cont_loss": cont_loss.item(), "affine_loss": affine_loss.item(),
                     "relative_cat_loss": rel_cat_loss.item(), "total": total.item()}
    return rec


# --------------------------------------------------------------------------- #
# colored dSprites stage 2 (colored_dSprites/rp_color.py)                     #
# --------------------------------------------------------------------------- #


def colored_affine_color_regularizer(real_code, trans_code):
    """colored_dSprites/utils_rp_color.py:99-139: the 4 affine entries as in dSprites/utils_rp.py, the 3 colour
    entries as the ratio of the gains c * 0.5 + 1 (:38-47, :63-72)."""
    aff = dsprites_affine_regularizer(real_code[:, :4], trans_code[:, :4])
    rel = (trans_code[:, 4:] * 0.5 + 1) / (real_code[:, 4:] * 0.5 + 1)
    return torch.cat((aff, (rel - 1) / 0.5), dim=1).to(real_code.dtype)


def sample_colored(rs: np.random.RandomState, batch, code_dim=7, n_classes=3):
    """host draws in the reference's order: the per-image RGB gains U(0.5, 1) (rp_color.py:372-378), then code,
    labels (phase D, :409-414), then code, labels again (phase info, :447-453)."""
    d = {"color": torch.tensor(rs.uniform(0.5, 1, [batch, 3, 1, 1]), dtype=torch.float64)}
    d.update(sample_dsprites(rs, batch, code_dim, n_classes))
    return d


def step_colored(st, img_u8, draws, record=True, after_phase=None):
    """One iteration of colored_dSprites/rp_color.py:362-516 on ``img_u8`` uint8 [B,64,64].  ``after_phase(0)`` runs
    after the optimiser step of phase D, as in step_celeba."""
    Epxy, E, D, G = st["Epxy"], st["E"], st["D"], st["G"]
    dt = next(G.parameters()).dtype
    dev = next(G.parameters()).device
    bce, mse = nn.BCELoss(), nn.MSELoss()
    B = img_u8.shape[0]
    # uint8 x float64 gains -> float64 -> .float()  (:366-381)
    img = (img_u8.unsqueeze(1).repeat(1, 3, 1, 1).to(dev) * draws["color"].to(dev)).float().to(dt)
    valid = torch.ones(B, 1, device=dev, dtype=dt)
    fake = torch.zeros(B, 1, device=dev, dtype=dt)
    rec = {"phases": []}

    def aligned():
        code = Epxy(img)                                                       # :385 (grad-tracked, frozen)
        inv = torch.inverse(dsprites_align_matrix(code))
        gains = (code[:, 3:] * 0.1 + 1).unsqueeze(2).unsqueeze(3)              # utils_pxy.py:48-57
        return stn(img, inv[:, 0:2]) / gains                                   # :386-394

    def distorted(align_img, code):
        gains = (code[:, 4:] * 0.5 + 1).unsqueeze(2).unsqueeze(3)              # utils_rp_color.py:38-47
        return stn(align_img, dsprites_get_matrix(code[:, :4])[:, 0:2]) * gains   # :416-424

    # ---- phase D  (:397-441)
    align_img = aligned()
    code = draws["code_d"].to(dev, dt)
    lab = one_hot(draws["labels_d"], 3, code)
    trans_img = distorted(align_img, code)
    gen = G(torch.cat((lab, code), dim=1))
    d_real = D(trans_img)
    d_fake = D(gen.detach())
    d_loss = (bce(d_fake, fake) + bce(d_real, valid)) / 2
    st["opt_D"].zero_grad()
    d_loss.backward()
    if record:
        rec["phases"].append({"name": "D", "grads": _snap(st["opt_D"])})
    st["opt_D"].step()
    if record:
        rec["phases"][-1]["params_after"] = _params(st["opt_D"])
        rec["phases"][-1]["state_after"] = {k: {n: v.detach().clone() for n, v in st[k].state_dict().items()}
                                            for k in ("G", "D", "E")}
    if after_phase is not None:
        after_phase(0)

    # ---- phase info  (:444-516)
    code = draws["code_info"].to(dev, dt)
    lab = one_hot(draws["labels_info"], 3, code)
    gen = G(torch.cat((lab, code), dim=1))
    rec_cat, rec_cont = E(gen)
    g_loss = bce(D(gen), valid)
    cat_loss = mutual_info_loss(rec_cat, lab)
    cont_loss = mse(rec_cont, code)
    align_img = aligned()
    trans_img = distorted(align_img, code)
    align_cat, align_cont = E(align_img)
    trans_cat, trans_cont = E(trans_img)
    affine_loss = mse(colored_affine_color_regularizer(align_cont, trans_cont), code)
    rel_cat_loss = mutual_info_loss(trans_cat, align_cat.detach())
    total = cat_loss + cont_loss + affine_loss + rel_cat_loss + g_loss         # :511 (this summation order)
    st["opt_info"].zero_grad()
    total.backward()
    if record:
        rec["phases"].append({"name": "info", "grads": _snap(st["opt_info"])})
    st["opt_info"].step()
    if record:
        rec["phases"][-1]["params_after"] = _params(st["opt_info"])
    rec["losses"] = {"d_loss": d_loss.item(), "g_loss": g_loss.item(), "cat_loss": cat_loss.item(),
                     "cont_loss": cont_loss.item(), "affine_loss": affine_loss.item(),
                     "relative_cat_loss": rel_cat_loss.item(), "total": total.item()}
    return rec


# --------------------------------------------------------------------------- #
# MNIST (MNIST/EAD-GAN_rpqmnxy.py, MNIST/utils_rpqmnxy.py) -- BASELINE configs[0] #
# --------------------------------------------------------------------------- #


class MnistAffineApproximator(nn.Module):
    """MNIST/utils_rpqmnxy.py:12-34 (Affine_classifier): the 6 -> 256x4 -> 7 MLP that maps the top two rows of a
    relative affine matrix back to the 7 affine parameters; pre-trained and frozen in the reference."""

    def __init__(self):
        super().__init__()
        self.fc_block = nn.Sequential(nn.Linear(6, 256), nn.LeakyReLU(), nn.Linear(256, 256), nn.LeakyReLU(),
                                      nn.Linear(256, 256), nn.LeakyReLU(), nn.Linear(256, 256), nn.LeakyReLU(),
                                      nn.Linear(256, 7))

    def forward(self, x):
        return self.fc_block(x)


def mnist_weights_init_normal(m):
    """MNIST/EAD-GAN_rpqmnxy.py:54-60 (dispatches on class-name substrings)."""
    classname = m.__class__.__name__
    if classname.find("Conv") != -1:
        torch.nn.init.normal_(m.weight.data, 0.0, 0.02)
    elif classname.find("BatchNorm") != -1:
        torch.nn.init.normal_(m.weight.data, 1.0, 0.02)
        torch.nn.init.constant_(m.bias.data, 0.0)


class MnistGenerator(nn.Module):
    """MNIST/EAD-GAN_rpqmnxy.py:71-98 (latent 62 + 10 classes + 7 code; 32x32x1 output)."""

    def __init__(self, latent_dim=62, n_classes=10, code_dim=7, img_size=32, channels=1):
        super().__init__()
        self.init_size = img_size // 4
        self.l1 = nn.Sequential(nn.Linear(latent_dim + n_classes + code_dim, 128 * self.init_size ** 2))
        self.conv_blocks = nn.Sequential(
            nn.BatchNorm2d(128), nn.Upsample(scale_factor=2), nn.Conv2d(128, 128, 3, stride=1, padding=1),
            nn.BatchNorm2d(128, 0.8), nn.LeakyReLU(0.2, inplace=True), nn.Upsample(scale_factor=2),
            nn.Conv2d(128, 64, 3, stride=1, padding=1), nn.BatchNorm2d(64, 0.8), nn.LeakyReLU(0.2, inplace=True),
            nn.Conv2d(64, channels, 3, stride=1, padding=1), nn.Tanh())

    def forward(self, noise, labels, code):
        out = self.l1(torch.cat((noise, labels, code), -1))
        return self.conv_blocks(out.view(out.shape[0], 128, self.init_size, self.init_size))


def _mnist_trunk(channels, bn):
    layers = []
    for i, (a, b) in enumerate(((channels, 16), (16, 32), (32, 64), (64, 128))):
        layers += [spectral_norm(nn.Conv2d(a, b, 3, 2, 1)), nn.LeakyReLU(0.2, inplace=True)]
        if bn and i > 0:
            layers.append(nn.BatchNorm2d(b, 0.8))
    return nn.Sequential(*layers)


class MnistDiscriminator(nn.Module):
    """MNIST/EAD-GAN_rpqmnxy.py:101-134 (LSGAN: raw linear output)."""

    def __init__(self, img_size=32, channels=1):
        super().__init__()
        self.conv_blocks = _mnist_trunk(channels, False)
        self.adv_layer = nn.Sequential(spectral_norm(nn.Linear(128 * (img_size // 16) ** 2, 1)))

    def forward(self, img):
        out = self.conv_blocks(img)
        return self.adv_layer(out.view(out.shape[0], -1))


class MnistEncoder(nn.Module):
    """MNIST/EAD-GAN_rpqmnxy.py:137-175."""

    def __init__(self, latent_dim=62, n_classes=10, code_dim=7, img_size=32, channels=1):
        super().__init__()
        self.conv_blocks = _mnist_trunk(channels, True)
        feat = 128 * (img_size // 16) ** 2
        self.aux_layer = nn.Sequential(spectral_norm(nn.Linear(feat, n_classes)), nn.Softmax(dim=1))
        self.latent_layer = nn.Sequential(spectral_norm(nn.Linear(feat, code_dim)))
        self.noise_layer = nn.Sequential(spectral_norm(nn.Linear(feat, latent_dim)))

    def forward(self, img):
        out = self.conv_blocks(img)
        out = out.view(out.shape[0], -1)
        return self.aux_layer(out), self.latent_layer(out), self.noise_layer(out)


def _skew(m, n):
    out = _eye_batch(m.shape[0], m)
    out[:, 0, 1] = m
    out[:, 1, 0] = n
    return out


def mnist_get_matrix(code7):
    """MNIST/utils_rpqmnxy.py:46-60,87-114: R(theta) @ Z(p,q) @ Skew(m,n) @ T(x,y)."""
    theta = code7[:, 0] * np.pi / 9
    p, q = code7[:, 1] * 0.2 + 1, code7[:, 2] * 0.2 + 1
    return (_rot(theta) @ _zoom(p, q) @ _skew(code7[:, 3] * 0.2, code7[:, 4] * 0.2)
            @ _shift(code7[:, 5] * 0.1, code7[:, 6] * 0.1))


def mnist_affine_regularizer(real_code, trans_code, approximator):
    """MNIST/utils_rpqmnxy.py:117-134: relative matrix -> frozen MLP approximator -> code scale (:64-84)."""
    rel = mnist_get_matrix(trans_code) @ torch.inverse(mnist_get_matrix(real_code))
    pred = approximator(torch.cat((rel[:, 0], rel[:, 1]), dim=1))
    return torch.stack((pred[:, 0] / np.pi * 9, (pred[:, 1] - 1) / 0.2, (pred[:, 2] - 1) / 0.2, pred[:, 3] / 0.2,
                        pred[:, 4] / 0.2, pred[:, 5] / 0.1, pred[:, 6] / 0.1), dim=1)


def mnist_approximator_state(seed=0):
    """seeded random-init stand-in for rpqmnxy_approximator.pt (unavailable offline, SURVEY.md section 8c)."""
    g = torch.random.get_rng_state()
    torch.manual_seed(seed + 2000)
    sd = {k: v.clone() for k, v in MnistAffineApproximator().state_dict().items()}
    torch.random.set_rng_state(g)
    return sd


def build_mnist(seed=0, device="cpu", dtype=torch.float32):
    """Construction order of the script: ``from utils_rpqmnxy import *`` builds (and then loads) the approximator
    FIRST (utils_rpqmnxy.py:36-43, consuming the seeded RNG), then Generator, Discriminator, Encoder
    (EAD-GAN_rpqmnxy.py:205-207), then weights_init_normal on each (:229-231).  Optimisers :249-255:
    G lr, D 2*lr, info lr over G + E, lr = 1e-4, betas (0.5, 0.999)."""
    torch.manual_seed(seed)
    A = MnistAffineApproximator()
    A.load_state_dict(mnist_approximator_state(seed))
    A.eval()
    G, D, E = MnistGenerator(), MnistDiscriminator(), MnistEncoder()
    for m in (G, D, E):
        m.apply(mnist_weights_init_normal)
    for m in (A, G, D, E):
        m.to(device=device, dtype=dtype)
    betas, lr = (0.5, 0.999), 0.0001
    return {"A": A, "G": G, "D": D, "E": E,
            "opt_G": torch.optim.Adam([{"params": G.parameters()}], lr=lr, betas=betas),
            "opt_D": torch.optim.Adam(D.parameters(), lr=lr * 2, betas=betas),
            "opt_info": torch.optim.Adam(itertools.chain(G.parameters(), E.parameters()), lr=lr, betas=betas)}


def synth_mnist_images(batch, seed=0):
    """synthetic "digits": random 28x28 blobs bilinearly resized to 32x32 (the reference resizes MNIST to
    opt.img_size = 32, EAD-GAN_rpqmnxy.py:45,241) and normalised to [-1, 1]."""
    g = torch.Generator().manual_seed(3000 + seed)
    x = torch.rand(batch, 1, 7, 7, generator=g)
    x = F.interpolate(x, size=(28, 28), mode="bilinear", align_corners=False)
    x = F.interpolate(x, size=(32, 32), mode="bilinear", align_corners=False)
    return ((x > 0.55).float() * x - 0.5) / 0.5


def sample_mnist(rs: np.random.RandomState, batch, latent_dim=62, code_dim=7, n_classes=10):
    """host draws in the reference's order (EAD-GAN_rpqmnxy.py:351-358): labels, z, code."""
    labels = rs.randint(0, n_classes, batch)
    z = rs.normal(0, 1, (batch, latent_dim))
    code = rs.uniform(-1, 1, (batch, code_dim))
    return {"z": torch.tensor(z, dtype=torch.float32), "code": torch.tensor(code, dtype=torch.float32),
            "labels": torch.tensor(labels, dtype=torch.long)}


def step_mnist(st, imgs, draws, record=True, after_phase=None):
    """One iteration of MNIST/EAD-GAN_rpqmnxy.py:337-446 on ``imgs`` [B,1,32,32] in [-1,1].  ``after_phase(i)`` runs
    after the optimiser step of phase i = 0 (G), 1 (D), as in step_celeba."""
    A, G, D, E = st["A"], st["G"], st["D"], st["E"]
    dt = next(G.parameters()).dtype
    dev = next(G.parameters()).device
    mse, ce = nn.MSELoss(), nn.CrossEntropyLoss()
    lambda_cat, lambda_con, lambda_affine = 1, 0.1, 0.1                        # :201-203
    B = imgs.shape[0]
    real = imgs.to(dev, dt)
    valid = torch.ones(B, 1, device=dev, dtype=dt)
    fake = torch.zeros(B, 1, device=dev, dtype=dt)
    z, code = draws["z"].to(dev, dt), draws["code"].to(dev, dt)
    gt = draws["labels"].to(dev)
    lab = one_hot(gt, 10, code)
    scaled = stn(real, mnist_get_matrix(code)[:, 0:2])                         # :363-365
    rec = {"phases": []}

    def snap(name, opt, phase):
        if record:
            rec["phases"].append({"name": name, "grads": _snap(opt)})
        opt.step()
        if record:
            rec["phases"][-1]["params_after"] = _params(opt)
            rec["phases"][-1]["state_after"] = {k: {n: v.detach().clone() for n, v in st[k].state_dict().items()}
                                                for k in ("G", "D", "E")}
        if after_phase is not None and phase is not None:
            after_phase(phase)

    # ---- phase G  (:373-386)
    st["opt_G"].zero_grad()
    gen = G(z, lab, code)
    g_loss = mse(D(gen), valid)
    g_loss.backward()
    snap("G", st["opt_G"], 0)
    # ---- phase D  (:393-407)
    st["opt_D"].zero_grad()
    d_loss = (mse(D(scaled), valid) + mse(D(gen.detach()), fake)) / 2
    d_loss.backward()
    snap("D", st["opt_D"], 1)
    # ---- phase info  (:413-446)
    st["opt_info"].zero_grad()
    gen = G(z, lab, code)
    pred_label, pred_code, _ = E(gen)
    info1 = lambda_cat * ce(pred_label, gt) + lambda_con * mse(pred_code, code)
    _, transform_code, _ = E(scaled)
    _, real_code, _ = E(real)
    info_loss = info1 + lambda_affine * mse(mnist_affine_regularizer(real_code, transform_code, A), code)
    info_loss.backward()
    snap("info", st["opt_info"], None)
    rec["losses"] = {"g_loss": g_loss.item(), "d_loss": d_loss.item(), "info_loss": info_loss.item()}
    return rec


# --------------------------------------------------------------------------- #
# stage 1: Encoder_pxy pre-training (dSprites/pxy.py, colored_dSprites/pxy_color.py) #
# --------------------------------------------------------------------------- #


def pxy_get_matrix(code):
    """get_matrix_pxy (dSprites/utils_pxy.py:49-66): Z(p,p) @ T(x,y), p = c0 * 0.1 + 1, (x, y) = (c1, c2) * 0.1."""
    p = code[:, 0] * 0.1 + 1
    return _zoom(p, p) @ _shift(code[:, 1] * 0.1, code[:, 2] * 0.1)


def pxy_affine_regularizer(real_code, trans_code):
    """affine_regularzier_pxy (dSprites/utils_pxy.py:107-126; colored_dSprites/utils_pxy.py:150-175 adds the
    ratio of the colour gains c * 0.1 + 1 for code entries 3..5)."""
    rel = pxy_get_matrix(trans_code[:, :3]) @ torch.inverse(pxy_get_matrix(real_code[:, :3]))
    p = (rel[:, 0, 0] + rel[:, 1, 1]) / 2
    out = torch.stack(((p - 1) / 0.1, rel[:, 0, 2] / p / 0.1, rel[:, 1, 2] / p / 0.1), dim=1)
    if real_code.shape[1] > 3:
        relc = (trans_code[:, 3:] * 0.1 + 1) / (real_code[:, 3:] * 0.1 + 1)
        out = torch.cat((out, (relc - 1) / 0.1), dim=1)
    return out.to(real_code.dtype)


def build_pxy(seed=0, device="cpu", dtype=torch.float32, colored=False):
    """dSprites/pxy.py:113-122 / colored_dSprites/pxy_color.py: one Encoder_pxy, one Adam (lr 2e-4)."""
    torch.manual_seed(seed)
    E = DSpritesEncoderPxy(3, 6) if colored else DSpritesEncoderPxy()
    E.to(device=device, dtype=dtype)
    return {"E": E, "opt_E": torch.optim.Adam(E.parameters(), lr=0.0002, betas=(0.5, 0.999)), "colored": colored}


def sample_pxy(rs: np.random.RandomState, batch, colored=False):
    """host draws in the reference's order: (colored: RGB gains U(0.5,1), pxy_color.py:172-178), then the code."""
    d = {}
    if colored:
        d["color"] = torch.tensor(rs.uniform(0.5, 1, [batch, 3, 1, 1]), dtype=torch.float64)
    d["code"] = torch.tensor(rs.uniform(-1, 1, (batch, 6 if colored else 3)), dtype=torch.float32)
    return d


def step_pxy(st, img_u8, draws, record=True):
    """One iteration of dSprites/pxy.py:156-187 (gray, grid_sample padding 'border') or
    colored_dSprites/pxy_color.py:162-216 (RGB gains, padding 'zeros', :90)."""
    E, colored = st["E"], st["colored"]
    dt = next(E.parameters()).dtype
    dev = next(E.parameters()).device
    if colored:
        img = (img_u8.unsqueeze(1).repeat(1, 3, 1, 1).to(dev) * draws["color"].to(dev)).float().to(dt)
    else:
        img = img_u8.unsqueeze(1).to(dev).to(dt)
    code = draws["code"].to(dev, dt)
    real_code = E(img)
    trans = stn(img, pxy_get_matrix(code)[:, 0:2], padding_mode="zeros" if colored else "border")
    if colored:
        trans = trans * (code[:, 3:] * 0.1 + 1).unsqueeze(2).unsqueeze(3)
    trans_code = E(trans)
    loss = nn.MSELoss()(pxy_affine_regularizer(real_code, trans_code), code)
    st["opt_E"].zero_grad()
    loss.backward()
    rec = {"phases": []}
    if record:
        rec["phases"].append({"name": "E", "grads": _snap(st["opt_E"])})
    st["opt_E"].step()
    if record:
        rec["phases"][-1]["params_after"] = _params(st["opt_E"])
    rec["losses"] = {"affine_loss": loss.item()}
    return rec


# --------------------------------------------------------------------------- #
# pre-training of the MNIST affine approximator (MNIST/approximate_rpqmnxy.py) #
# --------------------------------------------------------------------------- #


def build_approximator(seed=0, device="cpu", dtype=torch.float32):
    """MNIST/approximate_rpqmnxy.py:20-53: the MLP, MSELoss, Adam(lr 2e-4, betas (0.5, 0.999))."""
    torch.manual_seed(seed)
    A = MnistAffineApproximator().to(device=device, dtype=dtype)
    return {"A": A, "opt": torch.optim.Adam(A.parameters(), lr=0.0002, betas=(0.5, 0.999))}


def sample_approximator(rs: np.random.RandomState, batch=128):
    """:121-122: codes (rand - 0.5) * 2, float32"""
    return torch.tensor((rs.rand(batch, 7) - 0.5) * 2, dtype=torch.float32)


def step_approximator(st, code, record=True):
    """One iteration of MNIST/approximate_rpqmnxy.py:118-138: code -> 3x3 matrix (R Z Skew T, :77-108) -> its top two
    rows -> MLP -> MSE against the 7 affine PARAMETERS (not the raw code)."""
    A = st["A"]
    dt = next(A.parameters()).dtype
    code = code.to(next(A.parameters()).device, dt)
    para = torch.stack((code[:, 0] * np.pi / 9, code[:, 1] * 0.2 + 1, code[:, 2] * 0.2 + 1, code[:, 3] * 0.2,
                        code[:, 4] * 0.2, code[:, 5] * 0.1, code[:, 6] * 0.1), dim=1)
    m = mnist_get_matrix(code)
    st["opt"].zero_grad()
    loss = nn.MSELoss()(A(torch.cat((m[:, 0], m[:, 1]), dim=1)), para)
    loss.backward()
    rec = {"loss": loss.item()}
    if record:
        rec["grads"] = _snap(st["opt"])
    st["opt"].step()
    if record:
        rec["params_after"] = _params(st["opt"])
    return rec
