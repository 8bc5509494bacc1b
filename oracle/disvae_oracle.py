"""CPU oracle for the disvae training hot path.  TEST INFRASTRUCTURE ONLY.

This file is a plain-PyTorch (fp32, CPU, stock ATen ops + autograd) restatement
of the algorithm the reference implements for the path named in
BASELINE.json:north_star.  It exists to *check* the CUDA product path; nothing
under `disentangling-vae_b200/` may import it.  Only `tests/`,
`__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference`
legs use it.

Pinning status: the reference ships no tests or golden vectors for this path
(SURVEY.md section 4), so the oracle is pinned against OUTPUTS OF THE REFERENCE
ITSELF: `tests/golden/make_golden.py` imports the unmodified reference from a
checkout of it, runs it on seeded inputs and commits
the results under `tests/golden/*.pt`; `tests/test_oracle_golden.py` checks
every function below against those files.

The arithmetic lives in PyTorch (requirements.txt:1 of the reference, unpinned;
2.11.0+cu128 here).  Each function cites the reference file:line it restates
(paths relative to the reference checkout).

Style: purely functional -- parameters are a flat dict name -> tensor using the
reference's state_dict keys, so a reference checkpoint (results/*/model.pt) can
be passed in directly.
"""
import math
from collections import OrderedDict

import torch
import torch.nn.functional as F

LOG_2PI = math.log(2.0 * math.pi)
HID_CH = 32      # encoders.py:43, decoders.py:43
KSIZE = 4        # encoders.py:44
HID_FC = 256     # encoders.py:45
DISC_HID = 1000  # discriminator.py:12
DISC_SLOPE = 0.2  # discriminator.py:10


# --------------------------------------------------------------------------
# parameter construction (seeded-init parity)
# --------------------------------------------------------------------------
def _default_layer_draw(w_shape, fan_in):
    """What torch's Conv/Linear constructors draw: weight ~ kaiming_uniform(a=sqrt 5)
    == U(+-1/sqrt(fan_in)), then bias ~ U(+-1/sqrt(fan_in)).  (torch/nn/modules/
    conv.py and linear.py reset_parameters -- third-party behaviour the
    reference relies on through encoders.py:54-67, decoders.py:53-65.)"""
    bound = 1.0 / math.sqrt(fan_in)
    w = torch.empty(w_shape).uniform_(-bound, bound)
    return w, bound


def _relu_kaiming_(w):
    """initialization.py:50-52: kaiming_uniform_(nonlinearity='relu'):
    bound = sqrt(2) * sqrt(3 / fan_in), fan_in = size(1) * receptive field."""
    fan_in = w.size(1) * (w[0][0].numel() if w.dim() > 2 else 1)
    bound = math.sqrt(2.0) * math.sqrt(3.0 / fan_in)
    with torch.no_grad():
        w.uniform_(-bound, bound)
    return w


def vae_layer_table(img_size, latent_dim):
    """(key, weight shape, bias length, fan_in of the constructor) in module
    construction order: encoders.py:54-67 then decoders.py:53-65."""
    n_chan, h, w = img_size
    is64 = (h == 64 and w == 64)
    kk = KSIZE * KSIZE
    t = []
    t.append(("encoder.conv1", (HID_CH, n_chan, 4, 4), HID_CH, n_chan * kk))
    t.append(("encoder.conv2", (HID_CH, HID_CH, 4, 4), HID_CH, HID_CH * kk))
    t.append(("encoder.conv3", (HID_CH, HID_CH, 4, 4), HID_CH, HID_CH * kk))
    if is64:
        t.append(("encoder.conv_64", (HID_CH, HID_CH, 4, 4), HID_CH, HID_CH * kk))
    t.append(("encoder.lin1", (HID_FC, HID_CH * kk), HID_FC, HID_CH * kk))
    t.append(("encoder.lin2", (HID_FC, HID_FC), HID_FC, HID_FC))
    t.append(("encoder.mu_logvar_gen", (2 * latent_dim, HID_FC), 2 * latent_dim, HID_FC))
    t.append(("decoder.lin1", (HID_FC, latent_dim), HID_FC, latent_dim))
    t.append(("decoder.lin2", (HID_FC, HID_FC), HID_FC, HID_FC))
    t.append(("decoder.lin3", (HID_CH * kk, HID_FC), HID_CH * kk, HID_FC))
    # ConvTranspose2d weight is [Cin, Cout, k, k]; torch computes its fan_in
    # from size(1) (= Cout) * k*k.
    if is64:
        t.append(("decoder.convT_64", (HID_CH, HID_CH, 4, 4), HID_CH, HID_CH * kk))
    t.append(("decoder.convT1", (HID_CH, HID_CH, 4, 4), HID_CH, HID_CH * kk))
    t.append(("decoder.convT2", (HID_CH, HID_CH, 4, 4), HID_CH, HID_CH * kk))
    t.append(("decoder.convT3", (HID_CH, n_chan, 4, 4), n_chan, n_chan * kk))
    return t


def disc_layer_table(latent_dim, hidden=DISC_HID):
    """discriminator.py:51-56."""
    dims = [latent_dim] + [hidden] * 5 + [2]
    return [("lin%d" % (i + 1), (dims[i + 1], dims[i]), dims[i + 1], dims[i]) for i in range(6)]


def _build(table):
    params = OrderedDict()
    for key, w_shape, n_bias, fan_in in table:
        w, bound = _default_layer_draw(w_shape, fan_in)
        b = torch.empty(n_bias).uniform_(-bound, bound)
        params[key + ".weight"] = w
        params[key + ".bias"] = b
    # vae.py:87-88 / discriminator.py:72-73: apply(weights_init) re-draws every
    # weight in module order; biases untouched (initialization.py:56-61).
    for key, _, _, _ in table:
        _relu_kaiming_(params[key + ".weight"])
    return params


def init_vae_params(img_size, latent_dim):
    """Seeded construction of a Burgess VAE: vae.py:15-26,47-50."""
    if list(img_size[1:]) not in [[32, 32], [64, 64]]:
        raise RuntimeError("{} sized images not supported".format(img_size))  # vae.py:41-42
    return _build(vae_layer_table(img_size, latent_dim))


def init_disc_params(latent_dim):
    """Seeded construction of the FactorVAE discriminator: discriminator.py:51-58."""
    return _build(disc_layer_table(latent_dim))


# --------------------------------------------------------------------------
# model forward
# --------------------------------------------------------------------------
def _has(p, key):
    return (key + ".weight") in p


# Test hook for FLIP-ROBUST gradient parity (oracle/same_branch.py).  Two correct fp32 evaluations of this network round
# a few (Leaky)ReLU pre-activations of a large batch to opposite sides of zero; every such unit switches a whole
# back-propagated path on or off, so full-batch gradients of two correct implementations differ by far more than their
# arithmetic error.  With `_ACT = dict(record={}, masks={...}, calls={})` the forward passes below (a) record every
# pre-activation and (b) apply GIVEN on/off patterns instead of their own sign test (`pre * mask`), which makes the
# backward pass a smooth function of the inputs again.  None (the default) = plain reference semantics.
_ACT = None


def _call_index(prefix):
    if _ACT is None:
        return 0
    c = _ACT.setdefault("calls", {})
    c[prefix] = c.get(prefix, -1) + 1
    return c[prefix]


def _act(pre, name, slope=0.0):
    if _ACT is None:
        return torch.relu(pre) if slope == 0.0 else F.leaky_relu(pre, slope)
    if _ACT.get("record") is not None:
        _ACT["record"][name] = pre.detach()
    m = (_ACT.get("masks") or {}).get(name)
    if m is None:
        return torch.relu(pre) if slope == 0.0 else F.leaky_relu(pre, slope)
    m = m.to(pre.dtype)
    return pre * (m if slope == 0.0 else m + slope * (1 - m))


def encoder_forward(p, x):
    """encoders.py:69-89.  Returns (mu, logvar), interleaved split (trap T1)."""
    h = x
    tag = "encoder#%d." % _call_index("encoder")
    for name in ("conv1", "conv2", "conv3", "conv_64"):
        k = "encoder." + name
        if _has(p, k):
            h = _act(F.conv2d(h, p[k + ".weight"], p[k + ".bias"], stride=2, padding=1), tag + name)
    h = h.reshape(x.size(0), -1)
    h = _act(F.linear(h, p["encoder.lin1.weight"], p["encoder.lin1.bias"]), tag + "lin1")
    h = _act(F.linear(h, p["encoder.lin2.weight"], p["encoder.lin2.bias"]), tag + "lin2")
    ml = F.linear(h, p["encoder.mu_logvar_gen.weight"], p["encoder.mu_logvar_gen.bias"])
    ml = ml.view(x.size(0), -1, 2)
    return ml[..., 0], ml[..., 1]


def decoder_forward(p, z):
    """decoders.py:67-84."""
    tag = "decoder#%d." % _call_index("decoder")
    h = _act(F.linear(z, p["decoder.lin1.weight"], p["decoder.lin1.bias"]), tag + "lin1")
    h = _act(F.linear(h, p["decoder.lin2.weight"], p["decoder.lin2.bias"]), tag + "lin2")
    h = _act(F.linear(h, p["decoder.lin3.weight"], p["decoder.lin3.bias"]), tag + "lin3")
    h = h.view(z.size(0), HID_CH, KSIZE, KSIZE)
    for name in ("convT_64", "convT1", "convT2"):
        k = "decoder." + name
        if _has(p, k):
            h = _act(F.conv_transpose2d(h, p[k + ".weight"], p[k + ".bias"], stride=2, padding=1), tag + name)
    k = "decoder.convT3"
    return torch.sigmoid(F.conv_transpose2d(h, p[k + ".weight"], p[k + ".bias"], stride=2, padding=1))


def reparameterize(mu, logvar, eps=None, training=True):
    """vae.py:52-71.  `eps` replaces randn_like so CUDA and CPU can share noise."""
    if not training:
        return mu
    std = torch.exp(0.5 * logvar)
    if eps is None:
        eps = torch.randn_like(std)
    return mu + std * eps


def vae_forward(p, x, eps=None, training=True):
    """vae.py:73-85: (recon, (mu, logvar), z)."""
    mu, logvar = encoder_forward(p, x)
    z = reparameterize(mu, logvar, eps, training)
    return decoder_forward(p, z), (mu, logvar), z


def discriminator_forward(dp, z):
    """discriminator.py:60-70."""
    h = z
    tag = "disc#%d." % _call_index("disc")
    for i in range(1, 6):
        h = _act(F.linear(h, dp["lin%d.weight" % i], dp["lin%d.bias" % i]), tag + "lin%d" % i, DISC_SLOPE)
    return F.linear(h, dp["lin6.weight"], dp["lin6.bias"])


# --------------------------------------------------------------------------
# loss pieces
# --------------------------------------------------------------------------
def reconstruction_loss(data, recon, distribution="bernoulli"):
    """losses.py:394-449 (sum over everything, / batch)."""
    b = recon.size(0)
    if distribution == "bernoulli":
        loss = F.binary_cross_entropy(recon, data, reduction="sum")
    elif distribution == "gaussian":
        loss = F.mse_loss(recon * 255, data * 255, reduction="sum") / 255
    elif distribution == "laplace":
        loss = F.l1_loss(recon, data, reduction="sum") * 3
        loss = loss * (loss != 0)
    else:
        raise ValueError("Unkown distribution: {}".format(distribution))
    return loss / b


def kl_normal(mu, logvar):
    """losses.py:452-480: returns (total, per-dimension vector)."""
    per_dim = 0.5 * (-1 - logvar + mu.pow(2) + logvar.exp()).mean(dim=0)
    return per_dim.sum(), per_dim


def log_density_gaussian(x, mu, logvar):
    """math.py:34-51."""
    return -0.5 * (LOG_2PI + logvar) - 0.5 * ((x - mu) ** 2 * torch.exp(-logvar))


def log_importance_weight_matrix(batch_size, n_data):
    """math.py:54-73 (column-structured, trap T3); built in fp32 like the
    reference's torch.Tensor(...).fill_()."""
    m = batch_size - 1
    strat = (n_data - m) / (n_data * m)
    w = torch.full((batch_size, batch_size), 1.0 / m, dtype=torch.float32)
    flat = w.view(-1)
    flat[::m + 1] = 1.0 / n_data
    flat[1::m + 1] = strat
    w[m - 1, 0] = strat
    return w.log()


def btcvae_log_densities(z, mu, logvar, n_data, is_mss=True):
    """losses.py:523-544: (log_pz, log_qz, log_prod_qzi, log_q_zCx), each [B]."""
    b, d = z.shape
    log_q_zcx = log_density_gaussian(z, mu, logvar).sum(1)
    log_pz = log_density_gaussian(z, torch.zeros_like(z), torch.zeros_like(z)).sum(1)
    mat = log_density_gaussian(z.reshape(b, 1, d), mu.reshape(1, b, d), logvar.reshape(1, b, d))
    if is_mss:
        mat = mat + log_importance_weight_matrix(b, n_data).to(z.device).view(b, b, 1)
    log_qz = torch.logsumexp(mat.sum(2), dim=1)
    log_prod_qzi = torch.logsumexp(mat, dim=1).sum(1)
    return log_pz, log_qz, log_prod_qzi, log_q_zcx


def btcvae_terms(z, mu, logvar, n_data, is_mss=True):
    """losses.py:369-373: (mi, tc, dw_kl) scalars."""
    log_pz, log_qz, log_prod, log_qzcx = btcvae_log_densities(z, mu, logvar, n_data, is_mss)
    return (log_qzcx - log_qz).mean(), (log_qz - log_prod).mean(), (log_prod - log_pz).mean()


def linear_annealing(init, fin, step, annealing_steps):
    """losses.py:511-518."""
    if annealing_steps == 0:
        return fin
    assert fin > init
    return min(init + (fin - init) * step / annealing_steps, fin)


def permute_dims(z, perms=None):
    """losses.py:483-508.  `perms` is a [D, B] long tensor of per-dimension batch
    permutations; if None they are drawn from the CPU generator like the
    reference (trap T7)."""
    b, d = z.shape
    out = torch.zeros_like(z)
    for j in range(d):
        pi = torch.randperm(b) if perms is None else perms[j]
        out[:, j] = z[pi.to(z.device), j]
    return out


# --------------------------------------------------------------------------
# full losses (value + every logged scalar)
# --------------------------------------------------------------------------
def loss_betaH(data, recon, mu, logvar, beta, rec_dist, step, steps_anneal, is_train=True):
    """losses.py:139-153 (VAE == beta 1, losses.py:28-29)."""
    rec = reconstruction_loss(data, recon, rec_dist)
    kl, kl_dims = kl_normal(mu, logvar)
    anneal = linear_annealing(0, 1, step, steps_anneal) if is_train else 1
    loss = rec + anneal * (beta * kl)
    return loss, dict(recon_loss=rec, kl_loss=kl, kl_dims=kl_dims, loss=loss)


def loss_betaB(data, recon, mu, logvar, c_init, c_fin, gamma, rec_dist, step, steps_anneal, is_train=True):
    """losses.py:186-202."""
    rec = reconstruction_loss(data, recon, rec_dist)
    kl, kl_dims = kl_normal(mu, logvar)
    c = linear_annealing(c_init, c_fin, step, steps_anneal) if is_train else c_fin
    loss = rec + gamma * (kl - c).abs()
    return loss, dict(recon_loss=rec, kl_loss=kl, kl_dims=kl_dims, loss=loss)


def loss_btcvae(data, recon, mu, logvar, z, n_data, alpha, beta, gamma, rec_dist, step,
                steps_anneal, is_train=True, is_mss=True):
    """losses.py:356-391."""
    rec = reconstruction_loss(data, recon, rec_dist)
    mi, tc, dw = btcvae_terms(z, mu, logvar, n_data, is_mss)
    anneal = linear_annealing(0, 1, step, steps_anneal) if is_train else 1
    loss = rec + (alpha * mi + beta * tc + anneal * gamma * dw)
    kl, kl_dims = kl_normal(mu, logvar)
    return loss, dict(recon_loss=rec, mi_loss=mi, tc_loss=tc, dw_kl_loss=dw, loss=loss,
                      kl_loss=kl, kl_dims=kl_dims)


# --------------------------------------------------------------------------
# training steps (Trainer._train_iteration, training.py:137-164)
# --------------------------------------------------------------------------
def make_leaf_params(p):
    return OrderedDict((k, v.detach().clone().requires_grad_(True)) for k, v in p.items())


def train_step(p, opt, x, loss_name, cfg, step, eps=None):
    """One non-factor step: forward, loss, zero_grad, backward, Adam.
    `p` leaf params (requires_grad), `opt` a torch.optim.Adam over p.values().
    `step` is loss_f.n_train_steps AFTER the _pre_call increment (losses.py:105-107).
    Returns (loss, logged dict, recon)."""
    recon, (mu, logvar), z = vae_forward(p, x, eps, True)
    rd, sa = cfg.get("rec_dist", "bernoulli"), cfg.get("reg_anneal", 0)
    if loss_name == "VAE":
        loss, logs = loss_betaH(x, recon, mu, logvar, 1, rd, step, sa)
    elif loss_name == "betaH":
        loss, logs = loss_betaH(x, recon, mu, logvar, cfg["betaH_B"], rd, step, sa)
    elif loss_name == "betaB":
        loss, logs = loss_betaB(x, recon, mu, logvar, cfg["betaB_initC"], cfg["betaB_finC"],
                                cfg["betaB_G"], rd, step, sa)
    elif loss_name == "btcvae":
        loss, logs = loss_btcvae(x, recon, mu, logvar, z, cfg["n_data"], cfg["btcvae_A"],
                                 cfg["btcvae_B"], cfg["btcvae_G"], rd, step, sa)
    else:
        raise ValueError("Uknown loss : {}".format(loss_name))
    opt.zero_grad()
    loss.backward()
    opt.step()
    return loss.detach(), logs, recon.detach()


def factor_step(p, dp, opt, opt_d, x, cfg, step, eps_full=None, eps1=None, eps2=None, perms=None):
    """FactorVAE iteration: training.py:152-162 + losses.py:243-313.
    Includes the discarded full-batch forward (trap T6; it only consumes RNG so
    with injected eps it is skipped unless eps_full is None and eps1 is None)."""
    rd, sa, gamma = cfg.get("rec_dist", "bernoulli"), cfg.get("reg_anneal", 0), cfg["factor_G"]
    if eps1 is None and eps_full is None:
        with torch.no_grad():
            vae_forward(p, x, None, True)           # training.py:153 (result discarded)
    half = x.size(0) // 2
    parts = x.split(half)
    x1, x2 = parts[0], parts[1]
    recon, (mu, logvar), z1 = vae_forward(p, x1, eps1, True)
    rec = reconstruction_loss(x1, recon, rd)
    kl, kl_dims = kl_normal(mu, logvar)
    d_z = discriminator_forward(dp, z1)
    tc = (d_z[:, 0] - d_z[:, 1]).mean()
    anneal = linear_annealing(0, 1, step, sa)
    vae_loss = rec + kl + anneal * gamma * tc
    opt.zero_grad()
    vae_loss.backward(retain_graph=True)
    mu2, lv2 = encoder_forward(p, x2)
    z2 = reparameterize(mu2, lv2, eps2, True)
    z_perm = permute_dims(z2, perms).detach()
    d_perm = discriminator_forward(dp, z_perm)
    ones = torch.ones(half, dtype=torch.long, device=x.device)
    d_tc = 0.5 * (F.cross_entropy(d_z, torch.zeros_like(ones)) + F.cross_entropy(d_perm, ones))
    opt_d.zero_grad()
    d_tc.backward()                                  # also reaches the encoder (trap T5)
    opt.step()
    opt_d.step()
    logs = dict(recon_loss=rec, kl_loss=kl, kl_dims=kl_dims, loss=vae_loss, tc_loss=tc,
                discrim_loss=d_tc)
    return vae_loss.detach(), logs, recon.detach()


def make_adam(params, lr, betas=(0.9, 0.999)):
    """main.py:208 / losses.py:238."""
    return torch.optim.Adam(list(params.values()), lr=lr, betas=betas)


# --------------------------------------------------------------------------
# disentanglement metrics (Evaluator.compute_metrics, evaluate.py:119-317)
# --------------------------------------------------------------------------
def estimate_latent_entropies(samples_zCx, mean, logvar, samples_x, chunk=50):
    """evaluate.py:233-297 with the drawn indices `samples_x` given ([n_samples] int64; the reference draws
    torch.randperm(len_dataset)[:n_samples], :267).  Includes the reference's reshape-not-transpose of the selected
    block (:270).  -> H_z [latent_dim].  `chunk` samples at a time (the reference uses 10, :272): a sum over samples in
    a different grouping, not different arithmetic."""
    len_dataset, latent_dim = samples_zCx.shape
    n_samples = samples_x.numel()
    zs = samples_zCx.index_select(0, samples_x).view(latent_dim, n_samples)
    log_N = math.log(len_dataset)
    H_z = torch.zeros(latent_dim, dtype=samples_zCx.dtype)
    for k in range(0, n_samples, chunk):
        zk = zs[:, k:k + chunk].unsqueeze(0)                            # [1, D, c]
        log_q_zCx = log_density_gaussian(zk, mean.unsqueeze(-1), logvar.unsqueeze(-1))   # [N, D, c]
        log_q_z = -log_N + torch.logsumexp(log_q_zCx, dim=0)            # :284
        H_z += (-log_q_z).sum(1)                                        # :287
    return H_z / n_samples                                              # :291


def estimate_H_zCv(samples_zCx, mean, logvar, lat_sizes, perms):
    """evaluate.py:299-317; `perms` = iterator over the index draws of the successive estimator calls."""
    latent_dim = samples_zCx.size(-1)
    lat_sizes = [int(v) for v in lat_sizes]
    len_dataset = 1
    for v in lat_sizes:
        len_dataset *= v
    s = samples_zCx.view(*lat_sizes, latent_dim)
    m, lv = mean.view(*lat_sizes, latent_dim), logvar.view(*lat_sizes, latent_dim)
    H_zCv = torch.zeros(len(lat_sizes), latent_dim, dtype=samples_zCx.dtype)
    for f, lat_size in enumerate(lat_sizes):
        idcs = [slice(None)] * len(lat_sizes)
        for i in range(lat_size):
            idcs[f] = i
            sub = [t[tuple(idcs)].contiguous().view(len_dataset // lat_size, latent_dim) for t in (s, m, lv)]
            H_zCv[f] += estimate_latent_entropies(sub[0], sub[1], sub[2], next(perms)) / lat_size
    return H_zCv


def mig_aam(H_z, H_zCv, lat_sizes):
    """evaluate.py:148-158, 163-198 -> (MIG, AAM, mig_k, aam_k)."""
    mut_info = -H_zCv + H_z
    sorted_mut_info = torch.sort(mut_info, dim=1, descending=True)[0].clamp(min=0)
    delta = sorted_mut_info[:, 0] - sorted_mut_info[:, 1]
    mig_k = delta / torch.as_tensor([float(v) for v in lat_sizes]).log()
    numerator = (sorted_mut_info[:, 0] - sorted_mut_info[:, 1:].sum(dim=1)).clamp(min=0)
    aam_k = numerator / sorted_mut_info[:, 0]
    aam_k[torch.isnan(aam_k)] = 0
    return mig_k.mean(), aam_k.mean(), mig_k, aam_k
