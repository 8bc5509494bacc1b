"""CPU-side tests: package surface, seeded init, checkpoint compatibility, loss host logic,
C-ABI symbol export, no-CPU-fallback guarantee, data-parallel plumbing on gloo."""
import ctypes
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "disentangling-vae_b200")
GOLDEN = os.path.join(ROOT, "tests", "golden")
SEED = 1234

import disvae  # noqa: E402
from disvae.models import losses as L  # noqa: E402
from disvae.models.discriminator import Discriminator  # noqa: E402
from disvae.models.vae import MODELS  # noqa: E402


def digest_close(t, dg, rtol=0.0):
    t = t.detach().double().flatten()
    assert t.numel() == dg["n"]
    assert torch.allclose(t[:8].float(), dg["head"], rtol=rtol, atol=0)
    assert torch.allclose(t[-8:].float(), dg["tail"], rtol=rtol, atol=0)
    assert abs(t.sum().item() - dg["sum"]) <= 1e-12 * max(1.0, dg["abssum"])


@pytest.mark.parametrize("img_size,z", [((1, 32, 32), 10), ((1, 64, 64), 10), ((3, 64, 64), 10), ((3, 64, 64), 64)])
def test_seeded_init_and_state_dict_match_reference(golden, img_size, z):
    g = golden("init.pt")["vae_%dx%dx%d_z%d" % (img_size + (z,))]
    torch.manual_seed(SEED)
    m = disvae.init_specific_model("Burgess", img_size, z)
    sd = m.state_dict()
    assert list(sd.keys()) == g["keys"]
    for k, v in sd.items():
        assert tuple(v.shape) == g["shapes"][k]
        digest_close(v, g["digest"][k])
    assert m.model_type == "Burgess" and m.latent_dim == z and m.num_pixels == img_size[1] * img_size[2]


@pytest.mark.parametrize("z", [10, 64])
def test_seeded_discriminator_init_matches_reference(golden, z):
    g = golden("init.pt")["disc_z%d" % z]
    torch.manual_seed(SEED)
    d = Discriminator(latent_dim=z)
    assert list(d.state_dict().keys()) == g["keys"]
    for k, v in d.state_dict().items():
        digest_close(v, g["digest"][k])


def test_model_factory_errors():
    assert MODELS == ["Burgess"]
    with pytest.raises(ValueError):
        disvae.init_specific_model("resnet", (1, 32, 32), 10)
    with pytest.raises(RuntimeError):
        disvae.init_specific_model("Burgess", (1, 28, 28), 10)


@pytest.mark.parametrize("name,img_size", [("btcvae_dsprites", (1, 64, 64)), ("VAE_mnist", (1, 32, 32))])
def test_reference_checkpoints_load(name, img_size):
    m = disvae.init_specific_model("Burgess", img_size, 10)
    sd = torch.load(os.path.join(GOLDEN, "ckpt", name + ".pt"))
    missing, unexpected = m.load_state_dict(sd, strict=True)
    assert not missing and not unexpected


def test_save_and_load_model_roundtrip(tmp_path):
    from disvae.utils.modelIO import load_metadata, load_model, save_model
    torch.manual_seed(0)
    m = disvae.init_specific_model("Burgess", (1, 32, 32), 10)
    save_model(m, str(tmp_path), metadata=dict(img_size=[1, 32, 32], latent_dim=10, model_type="Burgess", dataset="mnist"))
    assert load_metadata(str(tmp_path))["dataset"] == "mnist"
    m2 = load_model(str(tmp_path), is_gpu=False)
    assert not m2.training
    for (k, a), (_, b) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert torch.equal(a, b), k


def test_no_cpu_fallback():
    m = disvae.init_specific_model("Burgess", (1, 32, 32), 10)
    with pytest.raises(RuntimeError, match="CUDA only"):
        m(torch.rand(2, 1, 32, 32))
    with pytest.raises(RuntimeError, match="CUDA only"):
        m.decoder(torch.rand(2, 10))
    with pytest.raises(RuntimeError, match="CUDA only"):
        Discriminator()(torch.rand(2, 10))
    lf = L.get_loss_f("VAE", rec_dist="bernoulli", reg_anneal=0)
    with pytest.raises(RuntimeError, match="CUDA only"):
        lf(torch.rand(2, 1, 32, 32), torch.rand(2, 1, 32, 32), (torch.rand(2, 10), torch.rand(2, 10)), True, None)


def test_product_package_never_imports_oracle():
    for dp, _, files in os.walk(PKG):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dp, f)).read()
                assert "oracle" not in src.replace("# oracle", ""), os.path.join(dp, f)


KW = dict(rec_dist="bernoulli", reg_anneal=0, betaH_B=4, betaB_initC=0, betaB_finC=25, betaB_G=100, factor_G=6,
          latent_dim=10, lr_disc=5e-5, btcvae_A=1, btcvae_B=6, btcvae_G=1, device=torch.device("cpu"), n_data=1000,
          some_unrelated_argparse_key=3)


def test_get_loss_f_dispatch_and_attributes():
    assert L.LOSSES == ["VAE", "betaH", "betaB", "factor", "btcvae"]
    assert L.RECON_DIST == ["bernoulli", "laplace", "gaussian"]
    assert isinstance(L.get_loss_f("VAE", **KW), L.BetaHLoss) and L.get_loss_f("VAE", **KW).beta == 1
    assert L.get_loss_f("betaH", **KW).beta == 4
    b = L.get_loss_f("betaB", **KW)
    assert (b.C_init, b.C_fin, b.gamma) == (0, 25, 100)
    t = L.get_loss_f("btcvae", **KW)
    assert (t.n_data, t.alpha, t.beta, t.gamma, t.is_mss) == (1000, 1, 6, 1, True)
    f = L.get_loss_f("factor", **KW)
    assert f.gamma == 6 and isinstance(f.discriminator, Discriminator)
    assert f.optimizer_d.defaults["lr"] == 5e-5 and f.optimizer_d.defaults["betas"] == (0.5, 0.9)
    for lf in (b, t, f):
        assert lf.n_train_steps == 0 and lf.record_loss_every == 50 and lf.rec_dist == "bernoulli" and lf.steps_anneal == 0
    with pytest.raises(ValueError):
        L.get_loss_f("nope", **KW)
    with pytest.raises(ValueError):
        f(None, None, None, True, None)           # training.py:160 relies on this


def test_linear_annealing_and_record_policy():
    assert L.linear_annealing(0, 1, 5, 0) == 1
    assert L.linear_annealing(0, 1, 5, 10) == 0.5
    assert L.linear_annealing(0, 25, 200, 100) == 25
    with pytest.raises(AssertionError):
        L.linear_annealing(1, 0, 1, 10)
    lf = L.get_loss_f("VAE", **KW)
    st = {}
    assert lf._pre_call(True, st) is st and lf.n_train_steps == 1           # step 1 records
    assert lf._pre_call(True, st) is None and lf.n_train_steps == 2
    for _ in range(48):
        lf._pre_call(True, st)
    assert lf._pre_call(True, st) is st and lf.n_train_steps == 51          # 51 % 50 == 1
    assert lf._pre_call(False, st) is st and lf.n_train_steps == 51         # eval: always, no increment


def test_importance_weight_matrix_structure(golden):
    from disvae.utils.math import log_importance_weight_matrix
    G = golden("btcvae_density.pt")
    for b, n in [(64, 737280), (256, 202599), (7, 1000), (2, 50)]:
        assert torch.equal(log_importance_weight_matrix(b, n), G["logiw_b%d" % b])


def _header_symbols():
    src = open(os.path.join(ROOT, "include", "disvae_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(dv_[a-z0-9_]+)\s*\(", src)))


def test_library_loads_and_exports_every_declared_symbol():
    from disvae import _native
    if not os.path.exists(_native.LIB_PATH):
        sys.path.insert(0, PKG)
        import build as dv_build
        dv_build.build()
    lib = ctypes.CDLL(_native.LIB_PATH)
    syms = _header_symbols()
    assert len(syms) >= 30
    for s in syms:
        assert hasattr(lib, s), "missing export " + s
    assert set(_native.SIGNATURES) == set(syms)
    h = _native.lib()
    assert h.dv_built_arch() == 100 and h.dv_version() >= 100
    assert h.dv_status_string(-1).decode() == "unsupported shape"
    assert h.dv_conv_packed_floats(32) == 2 * 32 * 32 * 16 + 2 * 16 * 64 * 32   # ffma + tcgen05 (hi|lo) sections
    out = subprocess.run(["cuobjdump", "-lelf", _native.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_ctypes_signatures_match_the_header_prototypes():
    """Every prototype of include/disvae_b200.h has as many parameters as the ctypes binding passes (ABI drift guard:
    a mismatch would still load and then corrupt the call)."""
    from disvae import _native
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    text = open(os.path.join(root, "include", "disvae_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    protos = dict(re.findall(r"\b(dv_\w+)\s*\(([^;{]*?)\)\s*;", text, flags=re.S))
    assert set(protos) == set(_native.SIGNATURES)
    for name, params in protos.items():
        params = params.strip()
        n = 0 if params in ("", "void") else len(params.split(","))
        assert n == len(_native.SIGNATURES[name][1]), (name, n, len(_native.SIGNATURES[name][1]))
        # pointer parameters are bound as void pointers, sizes/flags as integers
        for decl, ctype in zip(params.split(",") if n else [], _native.SIGNATURES[name][1]):
            assert ("*" in decl) == (ctype is ctypes.c_void_p), (name, decl.strip())


def _ddp_worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from disvae.parallel import FlatGradSync, broadcast_parameters, shard_batch
    torch.manual_seed(rank)                                   # different init per rank on purpose
    m = disvae.init_specific_model("Burgess", (1, 32, 32), 10)
    broadcast_parameters(m)
    ref = torch.cat([p.detach().flatten() for p in m.parameters()])
    gathered = [torch.empty_like(ref) for _ in range(world)]
    dist.all_gather(gathered, ref)
    same = all(torch.equal(gathered[0], g) for g in gathered)
    for i, p in enumerate(m.parameters()):
        p.grad = torch.full_like(p, float(rank + 1) * (i + 1))
    sync = FlatGradSync(list(m.parameters()))
    sync.sync()
    expect = sum(range(1, world + 1)) / world
    ok = all(torch.allclose(p.grad, torch.full_like(p, expect * (i + 1))) for i, p in enumerate(m.parameters()))
    views = all(p.grad.data_ptr() == v.data_ptr() for p, v in zip(sync.params, sync.views))
    x = torch.arange(8).view(8, 1)
    shard = shard_batch(x)
    ok_shard = shard.flatten().tolist() == list(range(rank * 4, rank * 4 + 4))
    if rank == 0:
        torch.save(dict(same=same, ok=ok, views=views, ok_shard=ok_shard), out)
    dist.destroy_process_group()


def test_flat_grad_allreduce_world2_gloo(tmp_path):
    import torch.multiprocessing as mp
    out = str(tmp_path / "r.pt")
    mp.spawn(_ddp_worker, args=(2, 29561, out), nprocs=2, join=True)
    r = torch.load(out)
    assert r == dict(same=True, ok=True, views=True, ok_shard=True)


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` runs without a GPU (it times the unmodified reference shipped to oracle/_ref, or
    the CPU oracle port when that copy is absent) and prints ONE JSON line with the keys the bench contract names; its
    metric/unit/config match our own arm's."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--workload", "c1",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "images/sec" and d["unit"] == "img/s" and d["higher_is_better"] is True
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config",
              "cpu_baseline", "e2e"):
        assert k in d, k
    shipped = os.path.isfile(os.path.join(root, "oracle", "_ref", "main.py"))
    assert d["cpu_baseline"]["kind"] == ("reference" if shipped else "port") and d["cpu_baseline"]["value"] == d["value"]
    assert set(d["config"]) == {"workload", "loss", "img_size", "batch_per_gpu", "global_batch", "latent_dim", "n_data",
                                "rec_dist", "optimizer", "parallelism", "l2"}          # == our own arm's keys
    assert d["e2e"] == {"value": d["value"], "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["loss"] == "VAE" and d["config"]["batch_per_gpu"] == 64


def _row_collectives_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from disvae import parallel
    b, n = 3, 4
    mine = torch.arange(b * n, dtype=torch.float32).view(b, n) + 100 * rank
    g = parallel.all_gather_rows(mine)
    ok = tuple(g.shape) == (world * b, n) and all(torch.equal(g[r * b:(r + 1) * b], torch.arange(b * n, dtype=torch.float32).view(b, n) + 100 * r) for r in range(world))
    part = torch.full((world * b, n), float(rank + 1)) * torch.arange(world * b).view(-1, 1)
    rs = parallel.reduce_scatter_rows(part)
    expect = (sum(range(1, world + 1)) * torch.arange(world * b).view(-1, 1).float()).expand(-1, n)[rank * b:(rank + 1) * b]
    ok = ok and torch.equal(rs, expect)
    q.put((rank, bool(ok)))
    dist.destroy_process_group()


def test_row_collectives_world2_gloo():
    """all_gather_rows / reduce_scatter_rows (the two collectives of the global-batch beta-TCVAE estimator, SURVEY.md
    8f-1) on the gloo fallback path, world size 2: rank-major row order, sum semantics, this rank's block."""
    import socket
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_row_collectives_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(60)
    assert sorted(res) == [(0, True), (1, True)]


def test_shard_sampler_partitions_every_epoch():
    """disvae.parallel.ShardSampler (SURVEY.md 8f-3): the ranks' index lists are disjoint, equally long and cover the
    dataset (padding by wrap-around), identical permutation on every rank, a new one per epoch, deterministic."""
    from disvae.parallel import ShardSampler
    n, world = 1003, 4
    samplers = [ShardSampler(n, rank=r, world_size=world, shuffle=True, seed=7) for r in range(world)]
    for epoch in range(3):
        for s in samplers:
            s.set_epoch(epoch)
        parts = [list(s) for s in samplers]
        assert all(len(p) == len(samplers[0]) == 251 for p in parts)
        flat = [i for p in parts for i in p]
        assert set(flat) == set(range(n)) and len(flat) == 1004                 # one wrapped-around duplicate
        assert parts == [list(s) for s in samplers]                               # deterministic
        if epoch:
            assert parts[0] != prev
        prev = parts[0]
    assert list(ShardSampler(10, rank=1, world_size=2, shuffle=False)) == [1, 3, 5, 7, 9]
    assert len(ShardSampler(10, rank=0, world_size=4, drop_last=True)) == 2
    loader = torch.utils.data.DataLoader(list(range(20)), batch_size=4, sampler=ShardSampler(20, rank=0, world_size=2, seed=1))
    assert sum(len(b) for b in loader) == 10


def test_mlp_modes_restore_their_state_and_the_trace_lists_two_discriminator_calls():
    """FactorVAE evaluates the discriminator ONCE on [z1; z_perm] (losses.FactorKLoss.call_optimize); the ReLU-branch trace
    must still present the two calls of the reference to the fp64 referee (oracle/same_branch.py)."""
    from disvae import ops
    assert ops._mlp_note_parts == 1 and ops._mlp_skip_param_grads is False
    with pytest.raises(RuntimeError):
        with ops.mlp_note_parts(2), ops.mlp_input_grad_only():
            assert ops._mlp_note_parts == 2 and ops._mlp_skip_param_grads is True
            raise RuntimeError("leave the contexts through an exception")
    assert ops._mlp_note_parts == 1 and ops._mlp_skip_param_grads is False
    # the trace MlpFn.forward writes for a 2-part batch: all layers of part 0, then all layers of part 1
    sys.path.insert(0, ROOT)
    from oracle.same_branch import _to_oracle_names
    h1, h2 = torch.randn(6, 5), torch.randn(6, 5)
    trace = [("mlp.lin1", h1[:3]), ("mlp.lin2", h2[:3]), ("mlp.lin1", h1[3:]), ("mlp.lin2", h2[3:])]
    masks = _to_oracle_names(trace, {})
    assert list(masks) == ["disc#0.lin1", "disc#0.lin2", "disc#1.lin1", "disc#1.lin2"]
    assert torch.equal(masks["disc#1.lin2"], h2[3:] > 0)
