#!/usr/bin/env python
"""Child process of tests/test_main_gpu.py: the reference's UNMODIFIED `main.py` (oracle/_ref) drives THIS
repository's `disvae` package on cuda:0 -- the proof of the drop-in boundary (SURVEY.md 8b, reference
main.py:165-247).  Only the data loader is replaced (there are no datasets on the box): `main.get_dataloaders` is
looked up in main's globals (main.py:197,233), so assigning it is an injection, not a source edit.

    python tests/run_reference_main.py <loss> <workdir>

Prints one JSON line with what the parent asserts on.
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "disentangling-vae_b200")
sys.path.insert(0, ROOT)
from oracle import reference_env  # noqa: E402

# DISVAE_DRIVER_SELFTEST=1: drive the reference's OWN disvae on the CPU instead (validates this driver + the synthetic
# loader in the GPU-less build container; tests/test_reference_shipping.py)
SELFTEST = os.environ.get("DISVAE_DRIVER_SELFTEST") == "1"
REF = reference_env.activate(package_first=None if SELFTEST else PKG)

import numpy as np  # noqa: E402
import torch  # noqa: E402
from torch.utils.data import DataLoader, Dataset  # noqa: E402


class SyntheticShapes(Dataset):
    """dSprites-like: img = f(factors), known `lat_sizes`/`lat_names` like utils/datasets.py:148-160."""
    lat_names = ('shape', 'posX')
    lat_sizes = np.array([2, 96])

    def __init__(self, img_size):
        self.img_size = img_size
        C, H, W = img_size
        n = int(self.lat_sizes.prod())
        g = torch.Generator().manual_seed(7)
        imgs = torch.zeros(n, C, H, W)
        k = 0
        for s in range(2):
            for px in range(96):
                x0 = int(px * (W - 12) / 95)
                if s == 0:
                    imgs[k, :, H // 3:H // 3 + 10, x0:x0 + 10] = 1.0
                else:
                    imgs[k, :, H // 2:H // 2 + 6, x0:x0 + 12] = 1.0
                k += 1
        self.imgs = (imgs + 0.02 * torch.rand(imgs.shape, generator=g)).clamp_(0, 1)

    def __len__(self):
        return self.imgs.size(0)

    def __getitem__(self, i):
        return self.imgs[i], 0


def main():
    loss, work = sys.argv[1], sys.argv[2]
    os.makedirs(work, exist_ok=True)
    os.chdir(work)                                         # main.py reads ./hyperparam.ini and writes ./results/<name>
    with open(os.path.join(REF, "hyperparam.ini")) as fh, open("hyperparam.ini", "w") as out:
        out.write(fh.read())
    import disvae
    assert os.path.realpath(disvae.__file__).startswith(os.path.realpath(REF if SELFTEST else PKG)), disvae.__file__
    import main as ref_main
    assert os.path.realpath(ref_main.__file__).startswith(os.path.realpath(REF)), ref_main.__file__
    import utils.datasets as ref_datasets

    dataset = "dsprites" if loss == "btcvae" else "celeba"
    img_size = ref_datasets.get_img_size(dataset)

    def get_dataloaders(name, root=None, shuffle=True, pin_memory=True, batch_size=128, logger=None, **kw):
        return DataLoader(SyntheticShapes(img_size), batch_size=batch_size, shuffle=shuffle, pin_memory=pin_memory)
    ref_main.get_dataloaders = get_dataloaders

    name = "dropin_" + loss
    argv = [name, "-d", dataset, "-l", loss, "-b", "64", "-e", "2", "--checkpoint-every", "1", "--no-progress-bar",
            "-s", "1234", "--eval-batchsize", "64", "--lr", "0.001"] + (["--no-cuda"] if SELFTEST else [])
    args = ref_main.parse_arguments(argv)
    ref_main.main(args)                                    # train -> save_model -> load_model -> Evaluator (losses)

    exp_dir = os.path.join("results", name)
    from disvae.utils.modelIO import load_metadata, load_model
    model = load_model(exp_dir, is_gpu=not SELFTEST)
    meta = load_metadata(exp_dir)
    log = open(os.path.join(exp_dir, "train_losses.log")).read().splitlines()
    test_losses = json.load(open(os.path.join(exp_dir, "test_losses.log")))
    # one traversal through the reference's visualiser (utils/visualize.py:121-123,217-222): decoder on the model's device
    from utils.visualize import Visualizer
    model.eval()
    viz = Visualizer(model=model, model_dir=exp_dir, dataset=meta["dataset"], save_images=False)
    grid = viz.traversals(data=None, n_per_latent=4, n_latents=3)
    samples = torch.stack([SyntheticShapes(img_size)[i][0] for i in (0, 100)])
    rec = viz.reconstruct(samples, size=(2, 2), is_original=True)
    print(json.dumps({
        "loss": loss, "files": sorted(os.listdir(exp_dir)), "log_head": log[0], "log_lines": len(log),
        "logged": sorted({l.split(",")[1] for l in log[1:]}), "test_losses": test_losses,
        "param_device": str(next(model.parameters()).device), "model_class": type(model).__module__,
        "meta_loss": meta["loss"], "img_size": list(meta["img_size"]),
        "traversal_shape": list(np.asarray(grid).shape), "reconstruct_shape": list(np.asarray(rec).shape),
        "native_launches": 0 if SELFTEST else int(__import__("disvae")._native.launch_count()),
    }))


if __name__ == "__main__":
    main()
