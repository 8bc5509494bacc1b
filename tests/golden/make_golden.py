#!/usr/bin/env python
"""Generate the golden fixtures in tests/golden/ from the UNMODIFIED reference.

Needs a checkout of the reference, found as build() finds it
(oracle/ship_reference.py: $DISVAE_REFERENCE, BASELINE.json reference_path, or
a directory named `reference` next to this repository):

    python tests/golden/make_golden.py

The reference is imported read-only with the two non-arithmetic shims of
SURVEY.md Appendix C (an `imageio` stub; `np.product = np.prod`).  Every output
below is produced by reference code (disvae.models.*, disvae.training.Trainer,
disvae.utils.math); the oracle and the CUDA path are then tested against these
files.  Inputs are seeded; small ones are stored, big ones are re-derived from
the seed in the tests and protected by a checksum stored here.

Also copies two shipped checkpoints (reference DATA files, not source) so that
trained / saturating weights are available on the GPU box:
results/btcvae_dsprites/model.pt and results/VAE_mnist/model.pt.
"""
import os
import shutil
import sys
import types
from collections import defaultdict

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle.ship_reference import find_checkout  # noqa: E402

REF = find_checkout()
assert REF is not None, "no checkout of the reference found"

sys.dont_write_bytecode = True
sys.path.insert(0, REF)
_io = types.ModuleType("imageio")
_io.mimsave = lambda *a, **k: None
_io.mimread = lambda *a, **k: []
sys.modules["imageio"] = _io
import numpy as np  # noqa: E402

np.product = np.prod
import torch  # noqa: E402
from torch import optim  # noqa: E402

import disvae  # noqa: E402  (the reference)
from disvae.models.losses import get_loss_f, _get_log_pz_qz_prodzi_qzCx, _permute_dims  # noqa: E402
from disvae.models.discriminator import Discriminator  # noqa: E402
from disvae.utils.math import log_importance_weight_matrix  # noqa: E402
from disvae.training import Trainer  # noqa: E402

assert os.path.realpath(disvae.__file__).startswith(os.path.realpath(REF)), disvae.__file__

SEED = 1234  # hyperparam.ini:6
LOSS_KW = dict(rec_dist="bernoulli", reg_anneal=0, betaH_B=4, betaB_initC=0, betaB_finC=25,
               betaB_G=100, factor_G=6, latent_dim=10, lr_disc=5e-5, btcvae_A=1, btcvae_B=6,
               btcvae_G=1, device=torch.device("cpu"), n_data=737280)


def tensor_digest(t):
    t = t.detach().double().flatten()
    return dict(sum=t.sum().item(), abssum=t.abs().sum().item(), n=t.numel(),
                head=t[:8].float().clone(), tail=t[-8:].float().clone())


def state_digest(sd):
    return {k: tensor_digest(v) for k, v in sd.items()}


def gen_init():
    out = {}
    for img_size, z in [((1, 32, 32), 10), ((1, 64, 64), 10), ((3, 64, 64), 10), ((3, 64, 64), 64)]:
        torch.manual_seed(SEED)
        model = disvae.init_specific_model("Burgess", img_size, z)
        key = "vae_%dx%dx%d_z%d" % (img_size + (z,))
        out[key] = dict(keys=list(model.state_dict().keys()),
                        shapes={k: tuple(v.shape) for k, v in model.state_dict().items()},
                        digest=state_digest(model.state_dict()))
    for z in (10, 64):
        torch.manual_seed(SEED)
        d = Discriminator(latent_dim=z)
        out["disc_z%d" % z] = dict(keys=list(d.state_dict().keys()),
                                   shapes={k: tuple(v.shape) for k, v in d.state_dict().items()},
                                   digest=state_digest(d.state_dict()))
    torch.save(out, os.path.join(HERE, "init.pt"))


def gen_forward():
    """Seeded-init model forward+backward on small batches, plus a trained checkpoint."""
    out = {}
    cases = [("c1_1x32x32", (1, 32, 32), 10, 8, None),
             ("c2_1x64x64", (1, 64, 64), 10, 4, None),
             ("c3_3x64x64", (3, 64, 64), 10, 2, None),
             ("c5_3x64x64_z64", (3, 64, 64), 64, 2, None),
             ("ckpt_btcvae_dsprites", (1, 64, 64), 10, 4, "btcvae_dsprites"),
             ("ckpt_VAE_mnist", (1, 32, 32), 10, 8, "VAE_mnist")]
    for name, img_size, z, b, ckpt in cases:
        torch.manual_seed(SEED)
        model = disvae.init_specific_model("Burgess", img_size, z)
        if ckpt is not None:
            model.load_state_dict(torch.load(os.path.join(REF, "results", ckpt, "model.pt")), strict=False)
        model.train()
        torch.manual_seed(SEED + 1)
        x = torch.rand(b, *img_size)
        if ckpt == "btcvae_dsprites":
            x = (x > 0.7).float()          # dSprites-like binary input (saturating regime, trap T8)
        eps = torch.randn(b, z)
        mu, logvar = model.encoder(x)
        zs = mu + torch.exp(0.5 * logvar) * eps          # vae.py:66-68 with the eps recorded
        recon = model.decoder(zs)
        # a scalar that touches everything, to pin the backward pass
        wr = torch.linspace(0.5, 1.5, recon.numel()).view_as(recon)
        probe = (recon * wr).sum() + (mu * 0.3).sum() - (logvar * 0.2).sum()
        model.zero_grad()
        probe.backward()
        grads = {k: v.grad.clone() for k, v in model.named_parameters()}
        out[name] = dict(img_size=img_size, latent_dim=z, batch=b, ckpt=ckpt, x=x, eps=eps,
                         mu=mu.detach().clone(), logvar=logvar.detach().clone(), z=zs.detach().clone(),
                         recon=recon.detach().clone(), probe=probe.item(),
                         grad_digest=state_digest(grads),
                         grad_small={k: g for k, g in grads.items() if g.numel() <= 64})
    torch.save(out, os.path.join(HERE, "forward.pt"))


def gen_losses():
    """Every loss x every rec_dist on fixed tensors: value, storer, grads."""
    out = {}
    torch.manual_seed(SEED + 2)
    b, c, s, z = 6, 3, 64, 10
    data = torch.rand(b, c, s, s)
    recon0 = torch.sigmoid(torch.randn(b, c, s, s) * 3)
    recon0[0, 0, 0, :4] = torch.tensor([0.0, 1.0, 1e-30, 1 - 1e-7])   # saturated pixels (trap T8)
    mu0 = torch.randn(b, z)
    lv0 = torch.randn(b, z) * 0.5 - 1
    eps = torch.randn(b, z)
    out["inputs"] = dict(data=data, recon=recon0, mu=mu0, logvar=lv0, eps=eps)
    for loss_name in ["VAE", "betaH", "betaB", "btcvae"]:
        for rec_dist in ["bernoulli", "laplace", "gaussian"]:
            for reg_anneal, n_calls in [(0, 1), (100, 3)]:
                kw = dict(LOSS_KW, rec_dist=rec_dist, reg_anneal=reg_anneal)
                loss_f = get_loss_f(loss_name, **kw)
                for _ in range(n_calls):     # advance n_train_steps; record the last call
                    recon = recon0.clone().requires_grad_(True)
                    mu = mu0.clone().requires_grad_(True)
                    lv = lv0.clone().requires_grad_(True)
                    zz = mu + torch.exp(0.5 * lv) * eps
                    storer = defaultdict(list)
                    loss_f.n_train_steps = loss_f.n_train_steps   # explicit: state lives here
                    # record_loss_every=50: only step 1 records; force recording by eval storer
                    loss = loss_f(data, recon, (mu, lv), True, storer, latent_sample=zz)
                g = torch.autograd.grad(loss, [recon, mu, lv])
                # eval-mode call for the storer on the same tensors (always records, anneal=1)
                st_eval = defaultdict(list)
                loss_eval = loss_f(data, recon0, (mu0, lv0), False, st_eval, latent_sample=mu0 + torch.exp(0.5 * lv0) * eps)
                out["%s_%s_a%d" % (loss_name, rec_dist, reg_anneal)] = dict(
                    loss=loss.item(), n_train_steps=loss_f.n_train_steps,
                    storer_train={k: list(v) for k, v in storer.items()},
                    loss_eval=loss_eval.item(), storer_eval={k: list(v) for k, v in st_eval.items()},
                    g_recon=tensor_digest(g[0]), g_mu=g[1].clone(), g_logvar=g[2].clone())
    torch.save(out, os.path.join(HERE, "losses.pt"))


def gen_btcvae_density():
    out = {}
    for b, d, n_data in [(64, 10, 737280), (256, 64, 202599), (7, 3, 1000), (2, 1, 50)]:
        torch.manual_seed(SEED + 3)
        mu = torch.randn(b, d)
        lv = torch.randn(b, d) * 0.5 - 1
        eps = torch.randn(b, d)
        mu.requires_grad_(True)
        lv.requires_grad_(True)
        z = mu + torch.exp(0.5 * lv) * eps
        zd = z.detach().clone().requires_grad_(True)     # treat z as an independent input too
        for mss in (True, False):
            outs = _get_log_pz_qz_prodzi_qzCx(zd, (mu, lv), n_data, is_mss=mss)
            coef = [0.7, -1.3, 2.1, 0.4]
            probe = sum(c * o.mean() for c, o in zip(coef, outs))
            g = torch.autograd.grad(probe, [zd, mu, lv])
            out["b%d_d%d_mss%d" % (b, d, int(mss))] = dict(
                b=b, d=d, n_data=n_data, z=zd.detach().clone(), mu=mu.detach().clone(),
                logvar=lv.detach().clone(),
                log_pz=outs[0].detach().clone(), log_qz=outs[1].detach().clone(),
                log_prod_qzi=outs[2].detach().clone(), log_q_zCx=outs[3].detach().clone(),
                coef=coef, g_z=g[0].clone(), g_mu=g[1].clone(), g_logvar=g[2].clone())
        out["logiw_b%d" % b] = log_importance_weight_matrix(b, n_data)
    torch.save(out, os.path.join(HERE, "btcvae_density.pt"))


class _Loader(list):
    """Minimal stand-in for a DataLoader: list of (data, label) with .dataset."""
    def __init__(self, batches, n_data):
        super().__init__(batches)
        self.dataset = list(range(n_data))


def gen_train_steps():
    """k seeded Trainer._train_iteration steps per loss through the reference Trainer."""
    out = {}
    import logging
    import tempfile
    cases = [("VAE", (1, 32, 32), 8, 60000, dict(lr=5e-4)),
             ("betaH", (3, 64, 64), 4, 202599, dict(lr=5e-4, betaH_B=10)),
             ("betaB", (1, 32, 32), 8, 60000, dict(lr=1e-3, reg_anneal=100)),
             ("btcvae", (1, 64, 64), 8, 737280, dict(lr=5e-4, btcvae_B=6.4, reg_anneal=10)),
             ("factor", (3, 64, 64), 8, 202599, dict(lr=1e-4, factor_G=6.4, lr_disc=1e-5))]
    for loss_name, img_size, b, n_data, over in cases:
        torch.manual_seed(SEED)
        model = disvae.init_specific_model("Burgess", img_size, 10)
        optimizer = optim.Adam(model.parameters(), lr=over["lr"])
        kw = dict(LOSS_KW, n_data=n_data)
        kw.update({k: v for k, v in over.items() if k != "lr"})
        loss_f = get_loss_f(loss_name, **kw)      # factor: discriminator drawn here, after the model
        torch.manual_seed(SEED + 4)
        xs = [torch.rand(b, *img_size) for _ in range(3)]
        tmp = tempfile.mkdtemp()
        trainer = Trainer(model, optimizer, loss_f, device=torch.device("cpu"),
                          logger=logging.getLogger("golden"), save_dir=tmp, is_progress_bar=False)
        model.train()
        steps = []
        torch.manual_seed(SEED + 5)               # noise stream of the training iterations
        names = {id(p): k for k, p in model.named_parameters()}
        opt_state_step1 = None
        for x in xs:
            storer = defaultdict(list)
            lv = trainer._train_iteration(x, storer)
            steps.append(dict(loss=lv, storer={k: list(v) for k, v in storer.items()}))
            if opt_state_step1 is None:
                # after the FIRST step exp_avg = (1 - beta1) * grad and exp_avg_sq = (1 - beta2) * grad^2 exactly: the
                # gradient seen THROUGH the optimizer.  (Later steps depend on which way Adam moved the entries whose
                # first gradient is numerically zero -- +-lr regardless of magnitude -- and are only loosely comparable.)
                opt_state_step1 = {names[id(p)]: dict(exp_avg=tensor_digest(st["exp_avg"]),
                                                      exp_avg_sq=tensor_digest(st["exp_avg_sq"]))
                                   for p, st in optimizer.state.items()}
                if loss_name == "factor":
                    dn = {id(p): k for k, p in loss_f.discriminator.named_parameters()}
                    disc_step1 = {dn[id(p)]: dict(exp_avg=tensor_digest(st["exp_avg"]), exp_avg_sq=tensor_digest(st["exp_avg_sq"]))
                                  for p, st in loss_f.optimizer_d.state.items()}
        rec = dict(img_size=img_size, batch=b, n_data=n_data, over=over, xs_digest=[tensor_digest(x) for x in xs],
                   steps=steps, params=state_digest(model.state_dict()))
        # Adam moments after the 3 steps: linear / quadratic in the gradients, so -- unlike the parameters, which
        # move by ~lr whatever the gradient is -- they pin the gradients' magnitudes through the optimizer
        rec["opt_state_step1"] = opt_state_step1
        if loss_name == "factor":
            rec["disc_opt_state_step1"] = disc_step1
        rec["opt_state"] = {names[id(p)]: dict(exp_avg=tensor_digest(st["exp_avg"]), exp_avg_sq=tensor_digest(st["exp_avg_sq"]),
                                               step=float(st["step"]))
                            for p, st in optimizer.state.items()}
        if loss_name == "factor":
            rec["disc_params"] = state_digest(loss_f.discriminator.state_dict())
            dnames = {id(p): k for k, p in loss_f.discriminator.named_parameters()}
            rec["disc_opt_state"] = {dnames[id(p)]: dict(exp_avg=tensor_digest(st["exp_avg"]),
                                                          exp_avg_sq=tensor_digest(st["exp_avg_sq"]), step=float(st["step"]))
                                     for p, st in loss_f.optimizer_d.state.items()}
        out[loss_name] = rec
        shutil.rmtree(tmp, ignore_errors=True)
    torch.save(out, os.path.join(HERE, "train_steps.pt"))


def gen_permute():
    torch.manual_seed(SEED + 6)
    z = torch.randn(16, 10)
    torch.manual_seed(SEED + 7)
    zp = _permute_dims(z)
    torch.save(dict(z=z, z_perm=zp), os.path.join(HERE, "permute.pt"))


def gen_metrics():
    """MIG / AAM metrics (evaluate.py:119-317) from the reference Evaluator.
    (A) direct calls of Evaluator._estimate_latent_entropies on seeded statistics with explicit n_samples;
    (B) the whole Evaluator.__call__(loader, is_metrics=True) on a procedural dataset with 4 known factors
        (tests/synthetic_factors.py) through the shipped VAE_mnist checkpoint.  The estimator's default n_samples=10000
        needs >= 10000 examples in every factor slice (>= 10^5 images); the fixture lowers the DEFAULT ARGUMENT to 1000
        (`__defaults__`, no code change) so that 10^4 images suffice.  The index draws (`torch.randperm`, :267) are
        recorded so the CUDA path -- whose device generator draws differently -- can replay them."""
    import logging
    import tempfile
    from disvae.evaluate import Evaluator
    sys.path.insert(0, os.path.dirname(HERE))
    from synthetic_factors import FactorRectangles, loader
    out = {}
    drawn = []
    real_randperm = torch.randperm

    def recording_randperm(n, *a, **k):
        p = real_randperm(n, *a, **k)
        drawn.append(p.clone())
        return p

    torch.manual_seed(SEED)
    model = disvae.init_specific_model("Burgess", (1, 32, 32), 10)
    model.load_state_dict(torch.load(os.path.join(REF, "results", "VAE_mnist", "model.pt")))
    tmp = tempfile.mkdtemp()
    ev = Evaluator(model, None, device=torch.device("cpu"), logger=logging.getLogger("golden"), save_dir=tmp,
                   is_progress_bar=True)       # (evaluate.py:276 disables its bar when this is True)
    torch.randperm = recording_randperm
    try:
        # (A)
        for name, (n, d, s) in dict(n3000_d10_s500=(3000, 10, 500), n1200_d6_s1200=(1200, 6, 1200)).items():
            torch.manual_seed(SEED + 8)
            mean = torch.randn(n, d)
            logvar = torch.randn(n, d) * 0.7 - 1.5
            samples = mean + torch.exp(0.5 * logvar) * torch.randn(n, d)
            drawn.clear()
            H = ev._estimate_latent_entropies(samples, (mean, logvar), n_samples=s)
            out[name] = dict(n=n, d=d, s=s, mean=mean, logvar=logvar, samples=samples, perm=drawn[0][:s].clone(), H=H.clone())
        # (B)
        old_defaults = Evaluator._estimate_latent_entropies.__defaults__
        Evaluator._estimate_latent_entropies.__defaults__ = (1000,)
        ds = FactorRectangles()
        drawn.clear()
        torch.manual_seed(SEED + 9)
        ev(loader(ds), is_metrics=True, is_losses=False)
        Evaluator._estimate_latent_entropies.__defaults__ = old_defaults
        import json
        metrics = json.load(open(os.path.join(tmp, "metrics.log")))
        helpers = torch.load(os.path.join(tmp, "metric_helpers.pth"), weights_only=False)
        out["full"] = dict(n_samples=1000, k=10, metrics=metrics, helpers={k: v.clone() for k, v in helpers.items()},
                           perms=[p[:1000].clone() for p in drawn], imgs_digest=tensor_digest(ds.imgs))
        # (C) the two metric formulas on a table where they are not clamped away (evaluate.py:163-198)
        torch.manual_seed(SEED + 10)
        mi_table = torch.rand(4, 10) * 0.05
        mi_table[0, 2], mi_table[1, 7], mi_table[3, 0], mi_table[3, 5] = 1.5, 0.9, 0.6, 0.5
        mi_table[2] = 0.0                                  # a factor no latent informs: AAM's 0/0 -> 0 branch
        smi = torch.sort(mi_table, dim=1, descending=True)[0].clamp(min=0)
        st = {}
        mig = ev._mutual_information_gap(smi, np.array([10, 10, 10, 10]), storer=st)
        aam = ev._axis_aligned_metric(smi, storer=st)
        out["formulas"] = dict(sorted_mut_info=smi, mig=mig.clone(), aam=aam.clone(), mig_k=st["mig_k"].clone(),
                               aam_k=st["aam_k"].clone())
    finally:
        torch.randperm = real_randperm
    shutil.rmtree(tmp, ignore_errors=True)
    torch.save(out, os.path.join(HERE, "metrics.pt"))


def copy_checkpoints():
    dst = os.path.join(HERE, "ckpt")
    os.makedirs(dst, exist_ok=True)
    for name in ("btcvae_dsprites", "VAE_mnist"):
        shutil.copyfile(os.path.join(REF, "results", name, "model.pt"), os.path.join(dst, name + ".pt"))


if __name__ == "__main__":
    torch.set_num_threads(1)        # deterministic reduction order for the fixtures
    gen_init()
    gen_forward()
    gen_losses()
    gen_btcvae_density()
    gen_train_steps()
    gen_permute()
    gen_metrics()
    copy_checkpoints()
    for f in sorted(os.listdir(HERE)):
        p = os.path.join(HERE, f)
        if os.path.isfile(p):
            print("%-24s %8d bytes" % (f, os.path.getsize(p)))
