"""SURVEY 8(b) / north star: "keeps the ibl.models ... and ibl.evaluators ... API so it drops into examples/test.py
unchanged".  This test RUNS the reference's own `examples/test.py` -- the byte-identical text, stored as golden data
in tests/golden/reference_examples_test.py.txt (its sha256 is pinned below) -- under torch.distributed.run against
this repository's `ibl` package:

    init_dist('pytorch') -> datasets.create('pitts', ...) x2 -> Preprocessor/DistributedSliceSampler loaders ->
    models.create('vgg16') + 'netvlad' + 'embednet' -> DistributedDataParallel -> load_checkpoint/copy_state_dict ->
    --reduction: extract_features(train) -> PCA.train -> Evaluator.evaluate(..., pca=pca)

on a Pittsburgh-shaped synthetic tree (dbStruct .mat files + JPEGs).  The recalls it prints must equal the recalls of
the CPU oracle run on the same JPEGs, checkpoint and PCA fit."""
import hashlib
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

pytestmark = pytest.mark.gpu

FIXTURE = os.path.join(ROOT, "tests", "golden", "reference_examples_test.py.txt")
SHA256 = "23a3d57dc1af659c8b9aab1acb6d75c2b4d75b8312e4c52f3d91b8de342e70c0"
H, W, FEATURES = 96, 128, 32


def test_fixture_is_the_unmodified_reference_script():
    data = open(FIXTURE, "rb").read()
    assert hashlib.sha256(data).hexdigest() == SHA256


def _checkpoint(path):
    from ibl import models
    from ibl.utils.serialization import save_checkpoint
    from openibl_b200 import synth
    torch.manual_seed(3)
    base = models.create("vgg16", pretrained=False)
    pool = models.create("netvlad", dim=base.feature_dim)
    p = synth.make_netvlad_params(seed=3, sharp=True)
    pool.centroids.data.copy_(p["centroids"])
    pool.conv.weight.data.copy_(p["conv_weight"])
    model = models.create("embednet", base, pool)
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    # the training scripts save the DDP-wrapped model: keys carry 'module.' (examples/test.py:97-99)
    save_checkpoint({"state_dict": {"module." + k: v for k, v in sd.items()}, "epoch": 3, "best_recall5": 0.5},
                    False, fpath=path)
    return sd


def _oracle_recalls(data_dir, sd):
    from ibl import datasets
    from ibl.utils.data import get_transformer_test
    from ibl.utils.data.preprocessor import Preprocessor
    from oracle import ibl_oracle as O
    ds = datasets.create("pitts", os.path.join(data_dir, "pitts"), scale="30k", verbose=False)
    tf = get_transformer_test(H, W)

    def feats(items):
        pre = Preprocessor(items, root=ds.images_dir, transform=tf)
        x = torch.stack([pre[i][0] for i in range(len(items))])
        with torch.no_grad():
            return O.extract_descriptor(x, sd, vlad=True)

    train = sorted(list(set(ds.q_train) | set(ds.db_train)))
    U, lams, mu, _ = O.pca_train(feats(train), n_components=FEATURES)
    w, b = O.pca_load(U, lams, mu, n_components=FEATURES)
    q = O.pca_whiten(feats(ds.q_test), w, b)
    db = O.pca_whiten(feats(ds.db_test), w, b)
    d = O.pairwise_distance(q, db).numpy()
    return O.evaluate_all(d, ds.test_pos, [g[1] for g in ds.db_test])


def test_reference_examples_test_py_runs_unmodified_and_matches_oracle(tmp_path):
    from ibl import datasets
    data_dir, logs = str(tmp_path / "data"), str(tmp_path / "logs")
    datasets.write_synthetic_pitts_tree(os.path.join(data_dir, "pitts"), scale="30k")
    ckpt = os.path.join(logs, "model_best.pth.tar")
    sd = _checkpoint(ckpt)
    script = str(tmp_path / "test.py")
    with open(script, "wb") as f:
        f.write(open(FIXTURE, "rb").read())
    # models.create('vgg16') defaults to pretrained=True (a download); PYTHONPATH = this repository's `ibl` + the empty
    # h5py stand-in (inherited by the spawned DataLoader workers, which re-import the script)
    env = dict(os.environ, IBL_VGG16_RANDOM_INIT_OK="1",
               PYTHONPATH=os.pathsep.join([ROOT, os.path.join(ROOT, "tests", "fixtures", "stubs"),
                                           os.environ.get("PYTHONPATH", "")]))
    nproc = 2 if torch.cuda.device_count() >= 2 else 1
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
           "--master-addr", "127.0.0.1", "--master-port", "29741",
           script, "--launcher", "pytorch", "-d", "pitts", "--scale", "30k", "--data-dir", data_dir, "--resume", ckpt,
           "--vlad", "--reduction", "--features", str(FEATURES), "--height", str(H), "--width", str(W),
           "--test-batch-size", "8", "-j", "2"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=str(tmp_path), env=env)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    log = open(os.path.join(logs, "log_test_pitts.txt")).read()
    assert "=> Loaded checkpoint" in out.stdout + log and "calculating PCA parameters" in out.stdout + log
    got = [float(v) for v in re.findall(r"top-(?:1|5|10)\s+([0-9.]+)%", log)[-3:]]
    assert len(got) == 3, log[-2000:]
    want = _oracle_recalls(data_dir, sd)
    assert np.allclose(got, np.round(100 * want, 1), atol=0.051), (got, want)
    assert 0 < want[0] <= 1
    assert os.path.isfile(os.path.join(logs, "pca_params_model_best.h5"))
