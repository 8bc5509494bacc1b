#!/usr/bin/env python
"""bench.py -- disvae training hot path on B200 (contract: see the task statement / DESIGN.md section 6).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|reference-cuda]
                  [--workload c1..c5] [--scaling weak|strong] [--dump-outputs DIR]

One "step" = one full optimisation step (forward, loss, backward, gradient all-reduce for N>1, Adam) over one
synthetic batch.  Default workload at every N: BASELINE.json configs[1] (btcvae, 1x64x64, batch 1024 PER GPU, z=10,
bernoulli, MSS, Adam lr 5e-4) -- weak scaling.  `--scaling strong` divides the config's batch over the ranks.

  value  : images/s with the batches already resident in HBM (CUDA events, max over ranks)
  e2e    : the same through disvae.Trainer._train_epoch over a loader of PINNED HOST batches with a real storer: H2D
           copy of every batch and D2H copy of every step's loss inside the timed region
  parity : full-size forward, loss AND every parameter gradient of the timed model against the CPU oracle (fp32, with
           an fp64 run of the oracle as the arbiter of what fp32 allows)
  ddp_parity (N>1): rank r's loss == oracle on shard r, rank-averaged gradients == mean of the oracle's shard gradients
  roofline / roofline_logdensity / cpu_baseline / cuda_eager_baseline / clocks / gpu_launches : DESIGN.md section 6

--impl reference      : the UNMODIFIED reference (oracle/_ref, shipped by oracle/ship_reference.py) through its own
                        Trainer._train_iteration on the host cores (kind "reference"); the oracle port if the copy is
                        not there (kind "port").
--impl reference-cuda : the same unmodified reference with device=cuda (stock PyTorch eager: cuDNN/cuBLAS, TF32 off) --
                        the "existing Blackwell kernels" bar of SURVEY.md 8d.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "disentangling-vae_b200")
sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = {
    # name: (loss, img_size, per-GPU batch for weak scaling, latent, n_data, loss kwargs, lr, the config's own batch)
    "c2": ("btcvae", (1, 64, 64), 1024, 10, 737280, dict(btcvae_A=1, btcvae_B=6, btcvae_G=1), 5e-4, 1024),
    "c3": ("betaH", (3, 64, 64), 512, 10, 202599, dict(betaH_B=10), 5e-4, 512),
    "c5": ("btcvae", (3, 64, 64), 256, 64, 202599, dict(btcvae_A=1, btcvae_B=6, btcvae_G=1), 5e-4, 2048),
    "c1": ("VAE", (1, 32, 32), 64, 10, 60000, dict(), 5e-4, 64),
    # FactorVAE: `-b 256` doubled by main.py:191-194 -> loader batch 512 (two halves of 256); factor_celeba gamma 6.4
    "c4": ("factor", (3, 64, 64), 512, 10, 202599, dict(factor_G=6.4, lr_disc=1e-5), 1e-4, 512),
}
WORKLOAD_NAMES = {"c1": "BASELINE.json configs[0]: VAE mnist-shape", "c2": "BASELINE.json configs[1]: btcvae dsprites-shape",
                  "c3": "BASELINE.json configs[2]: betaH celeba-shape", "c4": "BASELINE.json configs[3]: factor celeba-shape",
                  "c5": "BASELINE.json configs[4]: btcvae celeba-shape z=64"}
# algorithmic work per image, forward + backward (SURVEY.md 8d): conv FLOPs
CONV_FLOP_PER_IMG = {(1, 64, 64): 71.30e6, (3, 64, 64): 81.79e6, (1, 32, 32): 17.04e6}
N_ROTATE = 8            # distinct batches cycled through (8 x 16.8 MB > 126 MB L2)


def loss_kwargs(workload, device):
    loss_name, img, B, z, n_data, lkw, lr, _ = WORKLOADS[workload]
    kw = dict(rec_dist="bernoulli", reg_anneal=0, betaH_B=4, betaB_initC=0, betaB_finC=25, betaB_G=100, factor_G=6,
              latent_dim=z, lr_disc=5e-5, btcvae_A=1, btcvae_B=6, btcvae_G=1, device=device, n_data=n_data)
    kw.update(lkw)
    return kw


def per_gpu_batch(args, world):
    _, _, B, _, _, _, _, B_cfg = WORKLOADS[args.workload]
    if args.batch:
        return args.batch
    if args.scaling == "strong":
        assert B_cfg % world == 0
        return B_cfg // world
    return B


def config_block(args, world, B):
    """Identical in every arm (ours / reference / reference-cuda): it names the WORKLOAD."""
    loss_name, img, _, z, n_data, _, lr, _ = WORKLOADS[args.workload]
    return {"workload": WORKLOAD_NAMES[args.workload], "loss": loss_name, "img_size": list(img), "batch_per_gpu": B,
            "global_batch": B * world, "latent_dim": z, "n_data": n_data, "rec_dist": "bernoulli",
            "optimizer": "Adam lr %g" % lr, "parallelism": "dp%d" % world if world > 1 else "single",
            "l2": "inputs larger than L2: %d distinct batches rotated (%.0f MB)" % (
                N_ROTATE, N_ROTATE * B * img[0] * img[1] * img[2] * 4 / 1e6)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], bf16=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi sampling DURING the timed region (profiling guide, clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = max(mx, float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return None
        load = sorted(s for s in sm if s >= 0.5 * max(sm)) or sorted(sm)
        return dict(sm_mhz=load[len(load) // 2], sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


def dump_outputs(out_dir, trainer, loss):
    """What the last timed step handed its caller, as DIR/<name>.npy (float32): the loss it returned and, updated in
    place, every parameter and its gradient (the discriminator's too for FactorVAE).  Inputs, weights and noise are
    seeded, so two builds run with the same arguments can be compared array for array.  At most 36 MB (c4: FactorVAE
    with its discriminator's parameters and gradients); the assertion keeps it within 64 MB."""
    import numpy as np
    arrays = {"loss": loss}
    nets = [("", trainer.model)]
    if getattr(trainer.loss_f, "discriminator", None) is not None:
        nets.append(("disc.", trainer.loss_f.discriminator))
    for prefix, net in nets:
        for k, p in net.named_parameters():
            arrays["param." + prefix + k] = p
            if p.grad is not None:
                arrays["grad." + prefix + k] = p.grad
    arrays = {k: t.detach().float().cpu().numpy() for k, t in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= 64 * 1024 * 1024, "outputs to dump take %d bytes" % total
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# =====================================================================================================
# our arm
# =====================================================================================================
def build_job(workload, device):
    sys.path.insert(0, PKG)
    import disvae
    from disvae.models.losses import get_loss_f
    loss_name, img, B, z, n_data, lkw, lr, _ = WORKLOADS[workload]
    torch.manual_seed(1234)
    model = disvae.init_specific_model("Burgess", img, z).to(device)
    from disvae.parallel import broadcast_parameters
    broadcast_parameters(model)
    opt = torch.optim.Adam(model.parameters(), lr=lr)
    loss_f = get_loss_f(loss_name, **loss_kwargs(workload, device))
    if loss_name == "factor":
        broadcast_parameters(loss_f.discriminator)
    import logging
    import tempfile
    trainer = disvae.Trainer(model, opt, loss_f, device=device, logger=logging.getLogger("bench"),
                             save_dir=tempfile.mkdtemp(prefix="dvbench"), is_progress_bar=False)
    model.train()
    return trainer


def run_ours(args):
    import torch.distributed as dist
    from collections import defaultdict
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (ours) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    sys.path.insert(0, PKG)
    from disvae import _native
    L = _native.lib()
    assert L.dv_device_check() == 0, "not an sm_100 device"

    loss_name, img, _, z, n_data, lkw, lr, _ = WORKLOADS[args.workload]
    B = per_gpu_batch(args, world)
    trainer = build_job(args.workload, device)
    g = torch.Generator().manual_seed(1234 + rank)
    host = [torch.rand(B, *img, generator=g).pin_memory() for _ in range(N_ROTATE)]
    resident = [h.to(device) for h in host]
    K, W = args.steps, args.warmup     # the Trainer captures its CUDA graph on the 3rd eligible step: W >= 3 keeps it untimed

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last = {}

    def timed(fn, n):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            r = fn(i)
        e1.record()
        barrier()
        last["out"] = r
        ms = torch.tensor([e0.elapsed_time(e1)], device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    step_res = lambda i: trainer._step(resident[i % N_ROTATE], None)            # noqa: E731
    # end to end: the Trainer's epoch loop over a loader of PINNED HOST batches (H2D of every batch on the Trainer's
    # copy stream one step ahead, async D2H of every step's loss, one blocking read of the epoch mean at the end) with a
    # real storer, so the steps that log scalars (every 50th, losses.py:105-114) run their eager + host-sync path
    loader = [(host[i % N_ROTATE], None) for i in range(K)]
    epoch_e2e = lambda: trainer._train_epoch(loader, defaultdict(list), 0)       # noqa: E731

    for i in range(W):
        step_res(i)
    clk = ClockSampler(local)
    if rank == 0:
        clk.start()
    l0 = _native.launch_count()
    ms = timed(step_res, K)
    launches = _native.launch_count() - l0
    clocks = clk.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # before the end-to-end and parity passes below move the model on (and replays overwrite the graph's loss)
        dump_outputs(args.dump_outputs, trainer, last["out"])
    # untimed warm-up of the end-to-end path: three loader steps, and one EAGER step -- torch.cuda.graph empties the
    # caching allocator when it captures, so the first eager step afterwards (the every-50th logging step of a real
    # run) would otherwise pay ~2 GB of cudaMalloc inside the timed epoch, once
    trainer._train_epoch(loader[:3], None, 0)
    graph_was = trainer.use_cuda_graph
    trainer.use_cuda_graph = False
    trainer._step(resident[0], None)
    trainer.use_cuda_graph = graph_was
    ms_e2e = timed(lambda i: epoch_e2e(), 1)

    out = None
    if rank == 0:
        pk = peaks()
        imgs = B * world * K
        value = imgs / (ms / 1e3)
        e2e_v = imgs / (ms_e2e / 1e3)
        conv_flop = CONV_FLOP_PER_IMG[img]
        out = {
            "metric": "images/sec", "value": round(value, 1), "unit": "img/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": round(ms / K, 4), "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32", "data": "synthetic (torch.rand, seed 1234+rank); random-init weights (seed 1234)",
            "config": config_block(args, world, B),
            "e2e": {"value": round(e2e_v, 1), "unit": "img/s", "h2d_bytes_per_step": B * img[0] * img[1] * img[2] * 4,
                    "d2h_bytes_per_step": 4, "ms_per_step": round(ms_e2e / K, 4),
                    "api": "disvae.Trainer._train_epoch(loader of pinned host batches, storer) -> mean loss (float)"},
            "cuda_graph": bool(trainer._graphs),
            "gpu_launches": int(launches),
            "launches_per_step": round(launches / K, 1),
            "conv_flop_fraction_of_bf16_peak": round(value / world * conv_flop / (pk["bf16_sustained"] * 1e12), 5),
            "clocks": clocks,
        }
    # ---- roofline of the dominant kernel + the named log-density kernel ----
    # Every rank runs the profiled steps (they contain the gradient all-reduce); only rank 0 reports.
    try:
        roof = kernel_rooflines(trainer, resident, min(K, 20), B, img, z, n_data, device, detail=args.detail and rank == 0)
    except Exception as e:                                     # never lose the headline line
        roof = {"roofline_error": repr(e)}
    if rank == 0:
        out.update(roof)
    if not args.no_parity:
        try:
            par = parity_check(trainer, args.workload, B, device, rank, world)
        except Exception as e:
            import traceback
            traceback.print_exc()
            par = {"error": repr(e), "ok": False}
        if rank == 0:
            out["ddp_parity" if world > 1 else "parity"] = par
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = sub_arm("reference", args, steps=8, warmup=1, key="cpu_baseline")
        if world == 1 and not args.no_eager_baseline:
            torch.cuda.synchronize()
            eager = sub_arm("reference-cuda", args, steps=min(K, 30), warmup=5)
            if isinstance(eager, dict) and "value" in eager:
                out["cuda_eager_baseline"] = {
                    "value": eager["value"], "unit": "img/s", "ms_per_step": eager["ms_per_step"],
                    "what": eager.get("what"), "torch": torch.__version__,
                    "ours_over_eager": round(out["value"] / eager["value"], 3)}
            else:
                out["cuda_eager_baseline"] = eager
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def sub_arm(impl, args, steps, warmup, key=None):
    """Run another arm of this script in a child process (the reference's `disvae` package cannot share a process with
    ours: same module name) and return its JSON line (or `key` of it)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", impl, "--workload", args.workload, "--steps", str(steps),
           "--warmup", str(warmup)]
    if args.batch:
        cmd += ["--batch", str(args.batch)]
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
        line = [l for l in r.stdout.strip().splitlines() if l.startswith("{")][-1]
        d = json.loads(line)
        return d[key] if key else d
    except Exception as e:
        return {"error": repr(e)}


def kernel_rooflines(trainer, resident, K, B, img, z, n_data, device, detail=False):
    """Per-entry-point device time inside K more steps (CUDA events around every C-ABI call on the
    launching stream), then the roofline of the dominant one and of the beta-TCVAE kernel."""
    from disvae import _native, ops
    pk = peaks()
    graph_was = trainer.use_cuda_graph
    trainer.use_cuda_graph = False               # per-call events need direct launches (the graph replays them opaquely)
    side_was = os.environ.get("DISVAE_SIDE_STREAM")
    os.environ["DISVAE_SIDE_STREAM"] = "0"       # ... and every kernel alone on the GPU: with the weight-gradient side stream
                                                 # two kernels share the SMs and each one's events span both
    _native.enable_profiling()
    for i in range(K):
        trainer._step(resident[i % len(resident)], None)
    torch.cuda.synchronize()
    table = _native.disable_profiling()          # name -> (total ms, calls)
    trainer.use_cuda_graph = graph_was
    if side_was is None:
        os.environ.pop("DISVAE_SIDE_STREAM", None)
    else:
        os.environ["DISVAE_SIDE_STREAM"] = side_was
    total = sum(t for t, _ in table.values())
    top = sorted(table.items(), key=lambda kv: -kv[1][0])
    if detail:
        for k, (t, n) in top:
            sys.stderr.write("%-44s %4d calls/step  %8.2f us/call  %8.2f us/step  %5.1f%%\n" % (
                k, n // K, t / n * 1e3, t / K * 1e3, 100 * t / total))
    # share per entry point (all layers) and the single heaviest (entry point, layer geometry)
    by_entry = {}
    for k, (t, n) in table.items():
        e = k.split("[")[0]
        by_entry[e] = by_entry.get(e, 0.0) + t
    res = {"kernel_share": {k: round(v / total, 4) for k, v in sorted(by_entry.items(), key=lambda kv: -kv[1])[:8]},
           # sum of the per-call device times of one eager step (events around every C-ABI call): what is left of
           # ms_per_step after subtracting it is torch glue kernels + launch gaps
           "profiled_call_ms_per_step": round(total / K, 4),
           "profiled_calls_per_step": sum(n for _, n in table.values()) // K}
    traffic_table = {}
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tp):                                          # dram__bytes_read+write of one launch (ncu --set full)
        traffic_table = json.load(open(tp))
    conv = [(k, v) for k, v in top if k.startswith("dv_conv_") and "[" in k]
    name, (tms, calls) = conv[0] if conv else top[0]
    if conv:
        import re
        H, CH = map(int, re.search(r"H=(\d+),CH=(\d+)", name).groups())
        per_call_ms = tms / calls
        flops = 2.0 * B * H * H * 32 * 16 * CH                      # algorithmic MACs*2 of one launch (counted once,
        ach = flops / (per_call_ms / 1e3) / 1e12                    # the kernels issue 3 tf32 passes per product)
        # algorithmic HBM bytes of one launch: read/write the hi and the lo side once
        hi_b, lo_b = 4.0 * B * 4 * H * H * CH, 4.0 * B * H * H * 32
        alg_bytes = hi_b + lo_b
        ent = traffic_table.get(name) or {}
        res["roofline"] = {"kernel": name, "bound": "tensor", "achieved": round(ach, 3), "peak": pk["bf16_sustained"],
                           "unit": "TFLOP/s", "frac": round(ach / pk["bf16_sustained"], 5),
                           "traffic": ent.get("dram_bytes"), "traffic_source": ent.get("source"),
                           "algorithmic_flops_per_launch": flops, "algorithmic_hbm_bytes_per_launch": alg_bytes,
                           "hbm_achieved_gbs": round(alg_bytes / (per_call_ms / 1e3) / 1e9, 1),
                           "hbm_frac": round(alg_bytes / (per_call_ms / 1e3) / 1e9 / pk["hbm"], 4),
                           "us_per_launch": round(per_call_ms * 1e3, 2), "launches_per_step": calls // K,
                           "peak_source": pk["src"] + " bf16 sustained (kernel timed inside a long step)",
                           "note": "tcgen05 kind::tf32, error-compensated 3xTF32 (three tensor passes per algorithmic "
                                   "product; FLOPs counted once); time = CUDA events around the C-ABI call on its stream"}
        if CH != 32:
            # image-boundary layer (K = 16*CH): a streaming problem on the CUDA cores (dv_conv_img.cu), bounded by HBM
            r = res["roofline"]
            r.update({"bound": "hbm", "achieved": r["hbm_achieved_gbs"], "peak": pk["hbm"], "unit": "GB/s", "frac": r["hbm_frac"],
                      "flop_achieved_tflops": round(ach, 3),
                      "peak_source": pk["src"] + " HBM copy bandwidth",
                      "note": "exact-fp32 CUDA-core kernel (dv_conv_img.cu); achieved = algorithmic bytes (hi + lo side once) / "
                              "CUDA-event time around the C-ABI call on its stream"})
    else:
        res["roofline"] = {"kernel": name, "bound": "hbm", "achieved": None, "peak": pk["hbm"], "unit": "GB/s", "frac": None,
                           "traffic": None, "ms_per_step": round(tms / K, 4)}
    # the named kernel, timed alone (burst peak): virtual bytes 4*B^2*D + 12*B*D + 16*B (SURVEY.md 8d)
    Bk, Dk = 1024, 10
    torch.manual_seed(1)
    mu = torch.randn(Bk, Dk, device=device)
    lv = torch.randn(Bk, Dk, device=device) * 0.5 - 1
    zz = mu + torch.exp(0.5 * lv) * torch.randn(Bk, Dk, device=device)
    flush = torch.empty(256 * 1024 * 1024 // 4, device=device)
    for _ in range(5):
        ops.btcvae_rowstats(zz, mu, lv, n_data, True)
    ts = []
    for _ in range(20):
        flush.fill_(1.0)                                         # L2 flush between timed iterations
        _native.PROFILE_ONLY = "dv_btcvae_fwd"
        _native.enable_profiling()
        ops.btcvae_rowstats(zz, mu, lv, n_data, True)
        torch.cuda.synchronize()
        t = _native.disable_profiling()
        ts.append(t["dv_btcvae_fwd"][0])
    _native.PROFILE_ONLY = None
    ts.sort()
    t_med = ts[len(ts) // 2]
    # the same measurement around a kernel that does nothing measurable (16 bytes through dv_u8_to_f32): what the method
    # itself costs (event records + launch on an idle, L2-flushed GPU)
    tiny_src = torch.zeros(16, dtype=torch.uint8, device=device)
    tiny_dst = torch.empty(16, device=device)
    fl = []
    for _ in range(10):
        flush.fill_(1.0)
        _native.PROFILE_ONLY = "dv_u8_to_f32"
        _native.enable_profiling()
        ops.u8_to_f32(tiny_src, out=tiny_dst)
        torch.cuda.synchronize()
        fl.append(_native.disable_profiling()["dv_u8_to_f32"][0])
    _native.PROFILE_ONLY = None
    fl.sort()
    floor_us = fl[len(fl) // 2] * 1e3
    vbytes = 4 * Bk * Bk * Dk + 12 * Bk * Dk + 16 * Bk
    ach = vbytes / (t_med / 1e3) / 1e9
    ent = traffic_table.get("dv_btcvae_fwd[B=1024,D=10]") or {}
    res["roofline_logdensity"] = {"kernel": "dv_btcvae_fwd (one launch: parameters + B x B x D sweep + means)", "bound": "hbm", "B": Bk, "D": Dk,
                                  "achieved": round(ach, 1), "peak": pk["hbm"], "unit": "GB/s (virtual bytes of the "
                                  "reference's B*B*D matrix)", "frac": round(ach / pk["hbm"], 4), "us": round(t_med * 1e3, 2),
                                  "virtual_bytes": vbytes, "compulsory_bytes": 12 * Bk * Dk + 16 * Bk,
                                  "traffic": ent.get("dram_bytes"), "traffic_source": ent.get("source"),
                                  "l2": "256 MB flush before every timed launch",
                                  "event_floor_us": round(floor_us, 2),
                                  "frac_net_of_event_floor": round(vbytes / max((t_med * 1e3 - floor_us), 1e-3) / 1e3 / pk["hbm"], 4),
                                  "note": "us = CUDA events around ONE launch after an L2 flush; event_floor_us = the same "
                                          "measurement around a kernel that does nothing (what the method itself costs); frac uses us"}
    return res


def _cos_min(ours, ref):
    c = 1.0
    for k, b in ref.items():
        a = ours[k].detach().double().cpu().flatten()
        b = b.detach().double().cpu().flatten()
        c = min(c, (torch.dot(a, b) / (a.norm() * b.norm()).clamp_min(1e-30)).item())
    return c


def parity_check(trainer, workload, B, device, rank, world):
    """Full-size check of the timed model on one seeded batch per rank: forward, loss and EVERY parameter gradient
    (after the rank average for N>1) of the CUDA path against the CPU oracle -- same weights, input and injected
    noise/permutations.
      * loss and reconstruction: against the fp32 oracle, 1e-4 (north_star);
      * gradients: against the fp64 oracle evaluated ON THE SAME BRANCH of the network (oracle/same_branch.py): at these
        batch sizes two correct fp32 evaluations round a few of the 10^7..10^8 ReLU pre-activations to opposite sides
        of zero and then differ by 1e-3..1e-1 of a gradient's scale (reported as grad_rel_err_vs_oracle_fp32_own_branch,
        informational); with the CUDA path's on/off pattern imposed on the fp64 oracle the comparison is of arithmetic
        again and held to 1e-4, and every flipped unit must be numerically ambiguous (flip_max_rel_preact).
    N>1 ("ddp_parity"): rank r's loss against the oracle on shard r; the rank-AVERAGED gradients against the mean over
    ranks of the oracle's shard gradients (SURVEY.md 8e); FactorVAE covers Trainer._factor_grads_distributed and the
    discriminator."""
    from collections import OrderedDict
    import torch.distributed as dist
    from disvae import ops
    from oracle import disvae_oracle as O
    from oracle import same_branch as SB
    loss_name, img, _, z, n_data, lkw, lr, _ = WORKLOADS[workload]
    g = torch.Generator().manual_seed(4321 + rank)
    x = torch.rand(B, *img, generator=g)
    model, lf = trainer.model, trainer.loss_f
    model.train()
    kw = loss_kwargs(workload, device)
    p32 = OrderedDict((k, v.detach().cpu().clone()) for k, v in model.state_dict().items())
    factor = loss_name == "factor"
    d32 = None
    steps_before = lf.n_train_steps
    ops.start_trace()
    if factor:
        h = B // 2
        e1, e2 = torch.randn(h, z, generator=g), torch.randn(h, z, generator=g)
        perms = torch.stack([torch.randperm(h, generator=g) for _ in range(z)])
        d32 = OrderedDict((k, v.detach().cpu().clone()) for k, v in lf.discriminator.state_dict().items())
        loss = trainer._grads_only(x.to(device), None, eps1=e1.to(device), eps2=e2.to(device), perms=perms).item()
    else:
        eps = torch.randn(B, z, generator=g)
        model.inject_noise([eps])
        loss = trainer._grads_only(x.to(device), None).item()
    trace = ops.stop_trace()
    lf.n_train_steps = steps_before
    ours = {k: p.grad for k, p in model.named_parameters()}
    if factor:
        ours.update({"disc." + k: p.grad for k, p in lf.discriminator.named_parameters()})
    with torch.no_grad():
        if factor:
            recon = model(x[:h].to(device), eps=e1.to(device))[0].cpu()
        else:
            recon = model(x.to(device), eps=eps.to(device))[0].cpu()

    def oracle(p, dp, dtype):
        xx = x.to(dtype)
        if factor:
            cfg = dict(rec_dist="bernoulli", reg_anneal=0, factor_G=kw["factor_G"])
            l, _, ro = O.factor_step(p, dp, O.make_adam(p, 0.0), O.make_adam(dp, 0.0, betas=(0.5, 0.9)), xx, cfg, step=1,
                                     eps1=e1.to(dtype), eps2=e2.to(dtype), perms=perms)
            return l.item(), ro
        ro, (mo, lo), zo = O.vae_forward(p, xx, eps.to(dtype))
        if loss_name == "btcvae":
            l, _ = O.loss_btcvae(xx, ro, mo, lo, zo, n_data, kw["btcvae_A"], kw["btcvae_B"], kw["btcvae_G"], "bernoulli", 1, 0)
        else:
            l, _ = O.loss_betaH(xx, ro, mo, lo, kw["betaH_B"] if loss_name == "betaH" else 1, "bernoulli", 1, 0)
        l.backward()
        return l.item(), ro.detach()

    # fp32 oracle on its own branch: loss / reconstruction referee, gradients informational
    p = O.make_leaf_params(p32)
    dp = O.make_leaf_params(d32) if factor else None
    l32, r32 = oracle(p, dp, torch.float32)
    g32 = {k: v.grad for k, v in p.items()}
    if factor:
        g32.update({"disc." + k: v.grad for k, v in dp.items()})
    # fp64 oracle on the CUDA path's branch: gradient referee
    ref = SB.same_branch_reference(trace, p32, lambda pp, dd: oracle(pp, dd, torch.float64)[0], disc32=d32,
                                   run_oracle32=lambda pp, dd: oracle(pp, dd, torch.float32)[0])
    g64 = ref["grads"]
    if world > 1:                                              # mean of the shard gradients over ranks, like ours
        for gd in (g32, g64):
            for k in gd:
                t = gd[k].to(device)
                dist.all_reduce(t, op=dist.ReduceOp.SUM)
                gd[k] = (t / world).cpu()
    rel = abs(loss - l32) / abs(l32)
    rerr = (recon - r32).abs().max().item()
    e_same, key = SB.grad_errors(ours, g64)
    e_own, _ = SB.grad_errors(ours, g32)
    e_cpu = ref["cpu_fp32_same_branch_err"]
    # Gradients, relative to the largest gradient entry of the tensor's layer, on the same ReLU branch: 3e-4.  Every
    # tensor-core kernel is within 5e-6 of fp64 at these sizes (tests/test_fullsize_gpu.py); composed over the 16-kernel
    # backward chain -- the tensor core accumulates the exact 3xTF32 products with truncation -- the worst tensor lands at
    # 1-2e-4 where the CPU's fp32 FMA chains land at 1-2e-5 (both reported).  Where the CPU oracle itself is worse than
    # 3e-4/8 (long cancelling sums), 8x its error, capped at 1e-3.
    grad_tol = min(max(3e-4, 8.0 * e_cpu), 1e-3)
    ok = bool(rel < 1e-4 and rerr < 1e-4 and e_same <= grad_tol and ref["flip_max_rel"] <= 1e-3)
    res = {"loss_cuda": loss, "loss_oracle": l32, "loss_rel_err": rel, "loss_rel_err_vs_fp64": abs(loss - ref["loss"]) / abs(ref["loss"]),
           "recon_max_abs_err": rerr, "grad_rel_err_vs_fp64_same_branch": e_same, "grad_worst_tensor": key,
           "cpu_fp32_oracle_grad_rel_err_vs_fp64_same_branch": e_cpu, "grad_tol": grad_tol,
           "relu_units": ref["units"], "relu_flips_vs_fp64": ref["flips"], "flip_max_rel_preact": ref["flip_max_rel"],
           "grad_rel_err_vs_oracle_fp32_own_branch": e_own, "grad_cos_min_vs_oracle_fp32": _cos_min(ours, g32),
           "n_grad_tensors": len(ours), "batch": B, "ok": ok}
    if world > 1:
        flags = torch.tensor([float(ok), rel, e_same, ref["flip_max_rel"]], device=device, dtype=torch.float64)
        allf = [torch.zeros_like(flags) for _ in range(world)]
        dist.all_gather(allf, flags)
        res = {"world": world, "ok": bool(all(f[0].item() > 0.5 for f in allf)),
               "loss_rel_err_max": max(f[1].item() for f in allf),
               "avg_grad_rel_err_vs_fp64_same_branch": max(f[2].item() for f in allf),
               "flip_max_rel_preact": max(f[3].item() for f in allf),
               "rank0": res,
               "what": "rank r loss vs oracle on shard r (max over ranks); rank-averaged gradients of every parameter "
                       "vs the mean over ranks of the fp64 oracle's shard gradients on the CUDA path's ReLU branch"}
    return res


# =====================================================================================================
# reference arms
# =====================================================================================================
def oracle_job(workload, batch):
    from oracle import disvae_oracle as O
    loss_name, img, _, z, n_data, lkw, lr, _ = WORKLOADS[workload]
    torch.manual_seed(1234)
    p = O.make_leaf_params(O.init_vae_params(img, z))
    opt = O.make_adam(p, lr)
    cfg = dict(rec_dist="bernoulli", reg_anneal=0, n_data=n_data, betaH_B=4, btcvae_A=1, btcvae_B=6, btcvae_G=1)
    cfg.update(lkw)
    xs = [torch.rand(batch, *img) for _ in range(N_ROTATE)]
    state = dict(step=0)
    if loss_name == "factor":
        dp = O.make_leaf_params(O.init_disc_params(z))
        opt_d = O.make_adam(dp, cfg["lr_disc"], betas=(0.5, 0.9))

    def step():
        x = xs[state["step"] % N_ROTATE]
        state["step"] += 1
        if loss_name == "factor":
            O.factor_step(p, dp, opt, opt_d, x, cfg, state["step"])
        else:
            O.train_step(p, opt, x, loss_name, cfg, state["step"])
    return step


def reference_job(workload, batch, device):
    """The unmodified reference's own training step: disvae.Trainer._train_iteration (training.py:137-164) of
    oracle/_ref.  None if the copy is not there."""
    from oracle import reference_env
    ref = reference_env.find_reference()
    if ref is None:
        return None
    reference_env.activate(ref)
    import logging
    import tempfile
    from collections import defaultdict
    import disvae
    from disvae.models.losses import get_loss_f
    from disvae.training import Trainer
    assert os.path.realpath(disvae.__file__).startswith(os.path.realpath(ref)), disvae.__file__
    loss_name, img, _, z, n_data, lkw, lr, _ = WORKLOADS[workload]
    torch.manual_seed(1234)
    model = disvae.init_specific_model("Burgess", img, z)
    opt = torch.optim.Adam(model.parameters(), lr=lr)
    model = model.to(device)
    loss_f = get_loss_f(loss_name, **loss_kwargs(workload, device))
    trainer = Trainer(model, opt, loss_f, device=device, logger=logging.getLogger("refbench"),
                      save_dir=tempfile.mkdtemp(prefix="dvref"), is_progress_bar=False)
    model.train()
    xs = [torch.rand(batch, *img) for _ in range(N_ROTATE)]
    if device.type == "cuda":
        xs = [x.to(device) for x in xs]                      # resident, like our `value`
    state = dict(step=0)
    storer = defaultdict(list)

    def step():
        x = xs[state["step"] % N_ROTATE]
        state["step"] += 1
        return trainer._train_iteration(x, storer)
    return step


def pick_threads(step):
    """The reference's CPU path is PyTorch intra-op parallelism; on many-core hosts the default (all cores) is not
    the fastest for these small convolutions, so time one step at a few thread counts and keep the best."""
    cores = os.cpu_count() or 1
    best, best_t = cores, None
    for n in sorted({cores, min(cores, 64), min(cores, 32), min(cores, 16)}, reverse=True):
        torch.set_num_threads(n)
        step()
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best


def run_reference(args):
    """CPU arm (rank 0 only): the reference's own implementation of the path on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    B = per_gpu_batch(args, world)
    Bs = B
    step = reference_job(args.workload, Bs, torch.device("cpu"))
    kind = "reference" if step is not None else "port"
    if step is None:
        step = oracle_job(args.workload, Bs)
    cores = pick_threads(step)
    t0 = time.perf_counter()
    step()
    t_one = time.perf_counter() - t0
    sample = "full per-GPU batch of %d images per step" % Bs
    if t_one * (args.steps + args.warmup) > 240.0:                     # keep the arm within a few minutes
        Bs = max(64, B // 4)
        step = reference_job(args.workload, Bs, torch.device("cpu")) or oracle_job(args.workload, Bs)
        sample = "bounded sample: batch %d per step (of %d) -- the B^2 term of the loss is 1/16 per step" % (Bs, B)
    if world > 1:
        sample += "; rank 0 only: %d of the %d images of the global batch per step on ONE host process" % (Bs, B * world)
    for _ in range(max(args.warmup - 1, 1)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    v = round(Bs * args.steps / dt, 1)
    what = ("unmodified reference (oracle/_ref) disvae.Trainer._train_iteration on CPU" if kind == "reference"
            else "oracle port (oracle/disvae_oracle.py) on CPU")
    out = {"impl": "reference", "metric": "images/sec", "value": v, "unit": "img/s", "n_gpus": world, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 3), "higher_is_better": True,
           "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
           "data": "synthetic (torch.rand); random-init weights (seed 1234)",
           "config": config_block(args, world, B), "sample_images_per_step": Bs, "what": what,
           "cpu_baseline": {"value": v, "unit": "img/s", "cores": cores, "kind": kind, "sample": sample,
                            "host_logical_cores": os.cpu_count(), "torch": torch.__version__},
           "e2e": {"value": v, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


def run_reference_cuda(args):
    """The unmodified reference on the B200 through stock PyTorch eager (cuDNN / cuBLAS), TF32 disabled so that it
    computes in the same fp32 as the CPU path -- SURVEY.md 8d's "existing Blackwell kernels" bar."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    if not torch.cuda.is_available():
        print(json.dumps({"impl": "reference-cuda", "unavailable": "no CUDA device"}), flush=True)
        return
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cudnn.benchmark = True
    device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(device)
    B = per_gpu_batch(args, world)
    step = reference_job(args.workload, B, device)
    if step is None:
        print(json.dumps({"impl": "reference-cuda", "unavailable": "oracle/_ref not shipped"}), flush=True)
        return
    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    v = round(B * args.steps / (ms / 1e3), 1)
    out = {"impl": "reference-cuda", "metric": "images/sec", "value": v, "unit": "img/s", "n_gpus": 1, "steps": args.steps,
           "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 4), "higher_is_better": True,
           "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic (torch.rand); random-init weights",
           "config": config_block(args, 1, B),
           "what": "unmodified reference (oracle/_ref) disvae.Trainer._train_iteration, device=cuda, stock PyTorch %s eager "
                   "(cuDNN %s), allow_tf32=False, cudnn.benchmark=True, batches resident" % (
                       torch.__version__, torch.backends.cudnn.version())}
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-cuda"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--batch", type=int, default=0, help="override the per-GPU batch (experiments)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--detail", action="store_true", help="per-entry-point table on stderr")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss, parameters and gradients of the last timed step to DIR/<name>.npy "
                         "(--impl ours only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "reference-cuda":
        run_reference_cuda(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
