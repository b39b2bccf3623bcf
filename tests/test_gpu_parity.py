"""GPU parity tests: the CUDA path, called through the C ABI, against (a) the golden vectors produced by
the unmodified reference, (b) the CPU oracle on seeded inputs, (c) size-independent properties at
BASELINE sizes.  Tolerances are stated next to each check.

    descriptor tolerance (north star): rel-L2 <= 1e-4 vs the reference's fp32 forward
"""
import numpy as np
import pytest
import torch

from conftest import load_golden, rel_l2
from openibl_b200 import synth

pytestmark = pytest.mark.gpu

DESC_TOL = 1e-4        # north-star descriptor tolerance (relative L2, fp32 reference)
# conv5_3 map through 12 bf16x3 tensor-core layers.  Measured 7.7e-5..9.4e-5, almost all of it one
# uniform scale factor (1 - 9e-5): the tcgen05 fp32 accumulator truncates toward zero (bias ~ -2^-26
# per MMA, tools/diag_tc_error.py), which the L2 normalisations downstream cancel exactly.  With the
# best-fit scalar removed the residual is the bf16x3 representation error (FEAT_TOL_TC_DESCALED).
FEAT_TOL_TC = 1.5e-4
FEAT_TOL_TC_DESCALED = 5e-5
FEAT_TOL_SIMT = 5e-6   # fp32 CUDA cores: summation-order differences only


@pytest.fixture(scope="module")
def eng():
    from openibl_b200.engine import Engine
    return Engine.get(0)


@pytest.fixture(scope="module")
def O():
    from oracle import ibl_oracle
    return ibl_oracle


def descaled_rel_l2(a, b):
    """rel-L2 after removing the best-fit scalar between a and b."""
    a = np.asarray(a, dtype=np.float64).ravel()
    b = np.asarray(b, dtype=np.float64).ravel()
    s = float(a @ b) / float(a @ a)
    return float(np.linalg.norm(a * s - b) / np.linalg.norm(b))


def _modes():
    from openibl_b200.engine import CONV_SIMT_FP32, CONV_TC_BF16X3
    return [("simt", CONV_SIMT_FP32, FEAT_TOL_SIMT), ("tc", CONV_TC_BF16X3, FEAT_TOL_TC)]


def _bind(eng, sd, dev="cuda"):
    sdd = {k: v.to(dev) for k, v in sd.items()}
    slots = synth.VGG16_CONV_SLOTS
    eng.set_vgg16([sdd[f"base_model.base.{s}.weight"] for s in slots],
                  [sdd[f"base_model.base.{s}.bias"] for s in slots])
    eng.set_netvlad(sdd["net_vlad.conv.weight"], sdd["net_vlad.centroids"])
    if "pca_layer.weight" in sdd:
        eng.set_pca(sdd["pca_layer.weight"], sdd["pca_layer.bias"])
    return sdd


# ---------------------------------------------------------------------------------------------
# stage (i): one conv layer, both math modes, all epilogues
# ---------------------------------------------------------------------------------------------
CONV_CASES = [
    # N, H, W, cin, cout, relu, pool
    (1, 16, 32, 64, 64, True, False),
    (2, 30, 40, 128, 256, True, False),      # TW=8 patch, partial rows
    (1, 24, 48, 64, 128, True, True),        # fused 2x2 pool
    (1, 35, 45, 64, 64, True, True),         # odd sizes: floor pooling, partial patches
    (2, 17, 23, 256, 512, False, False),     # no ReLU (conv5_3-like), two N tiles
    (1, 60, 80, 512, 512, True, True),
    (1, 16, 24, 256, 256, True, False),      # 3 patches: the SM-pair kernel's last pair has an idle peer
    (3, 30, 40, 512, 512, False, False),     # conv5-like, 30 patches, pair tiles + per-pixel sum of squares path
    (1, 33, 17, 128, 128, True, True),       # halo staging with ragged borders on both axes + fused pool
]


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv3x3_layer_vs_oracle(eng, case):
    N, H, W, cin, cout, relu, pool = case
    g = torch.Generator().manual_seed(hash(case) % 1000)
    x = torch.randn(N, cin, H, W, generator=g)
    w = torch.randn(cout, cin, 3, 3, generator=g) * (2.0 / (cin * 9)) ** 0.5
    b = torch.randn(cout, generator=g) * 0.1
    ref = torch.nn.functional.conv2d(x.double(), w.double(), b.double(), padding=1)
    if relu:
        ref = ref.relu()
    if pool:
        ref = torch.nn.functional.max_pool2d(ref, 2, 2)
    ref = ref.permute(0, 2, 3, 1).contiguous()
    xd = x.permute(0, 2, 3, 1).contiguous().cuda()
    variants = [("simt", 0, 0, 3e-6), ("tc-f32", 1, 0, 2e-5), ("tc-planes", 2, 0, 2e-5)]
    if cout % 256 == 0:
        variants.append(("tc-bn256", 1, 256, 2e-5))
    if cout % 128 == 0:
        variants.append(("tc-bn64", 1, 64, 2e-5))
    for name, mode, bn, tol in variants:
        y = eng.debug_conv3x3(xd, w.cuda(), b.cuda(), relu=relu, pool=pool, mode=mode, bn=bn).cpu()
        assert y.shape == ref.shape, name
        assert rel_l2(y, ref) < tol, (name, rel_l2(y, ref))


# ---------------------------------------------------------------------------------------------
# whole path vs reference golden vectors
# ---------------------------------------------------------------------------------------------
def test_small_96x128_every_stage_vs_reference(eng):
    g = load_golden("small_96x128")
    sd = synth.make_state_dict(seed=5, with_pca=True, pca_dim=128, bias_scale=0.05)
    sdd = _bind(eng, sd)
    x = synth.make_images(seed=6, batch=2, height=96, width=128).cuda()
    for name, mode, ftol in _modes():
        eng.conv_mode = mode
        nhwc, nchw, pool = eng.vgg16_forward(x, want_nchw=True, want_pool=True, want_nhwc=True)
        assert rel_l2(nchw.cpu(), g["feat"]) < ftol, name
        assert descaled_rel_l2(nchw.cpu(), g["feat"]) < min(ftol, FEAT_TOL_TC_DESCALED), name
        assert rel_l2(nhwc.permute(0, 3, 1, 2).cpu(), g["feat"]) < ftol, name
        assert rel_l2(pool.cpu(), g["pool"]) < ftol * 2, name
        raw, nrm = eng.netvlad_forward(nchw, sdd["net_vlad.conv.weight"], sdd["net_vlad.centroids"],
                                       want_raw=True, want_norm=True)
        assert rel_l2(raw.cpu(), g["raw_vlad"]) < DESC_TOL / 4, name
        assert rel_l2(nrm.cpu(), g["vlad"]) < DESC_TOL / 4, name
        vlad, pool2 = eng.extract(x, pca=False, want_pool=True)
        assert rel_l2(vlad.cpu(), g["vlad"]) < DESC_TOL / 4, name
        assert rel_l2(pool2.cpu(), pool.cpu()) < 2e-5   # fused path pools the bf16 hi+lo planes
        desc, _ = eng.extract(x, pca=True)
        assert rel_l2(desc.cpu(), g["desc"]) < DESC_TOL, name


def test_odd_70x90_floor_pooling_vs_reference(eng):
    g = load_golden("odd_70x90")
    sd = synth.make_state_dict(seed=7, with_pca=False, bias_scale=0.05)
    _bind(eng, sd)
    x = synth.make_images(seed=8, batch=1, height=70, width=90).cuda()
    for name, mode, ftol in _modes():
        eng.conv_mode = mode
        _, nchw, pool = eng.vgg16_forward(x)
        assert tuple(nchw.shape) == (1, 512, 4, 5)
        assert rel_l2(nchw.cpu(), g["feat"]) < ftol, name
        vlad, _ = eng.extract(x, pca=False)
        assert rel_l2(vlad.cpu(), g["vlad"]) < DESC_TOL / 4, name


def test_hub_480x640_config_vs_reference(eng):
    """BASELINE configs[0]/[1] shape: full 480x640 image, K=64, PCA 4096, reference-run golden."""
    g = load_golden("hub_480x640")
    sd = synth.make_state_dict(seed=0, with_pca=True)
    _bind(eng, sd)
    x = synth.make_images(seed=1, batch=1).cuda()
    for name, mode, ftol in _modes():
        eng.conv_mode = mode
        _, nchw, pool = eng.vgg16_forward(x)
        assert rel_l2(nchw[:, ::8, ::3, ::4].cpu(), g["feat_sub"]) < ftol, name
        assert descaled_rel_l2(nchw[:, ::8, ::3, ::4].cpu(), g["feat_sub"]) < min(ftol, FEAT_TOL_TC_DESCALED), name
        assert abs(nchw.double().abs().sum().item() - g["feat_abs_sum"]) < 2 * ftol * g["feat_abs_sum"]
        assert rel_l2(pool.cpu(), g["pool"]) < 2 * ftol, name
        vlad, _ = eng.extract(x, pca=False)
        assert rel_l2(vlad.cpu(), g["vlad"]) < DESC_TOL / 4, name
        desc, _ = eng.extract(x, pca=True)
        assert desc.shape == (1, 4096)
        assert abs(float(desc.norm()) - 1.0) < 1e-5
        assert rel_l2(desc.cpu(), g["desc"]) < DESC_TOL, name


def test_sharp_netvlad_full_chain_vs_oracle(eng, O):
    """Random-init NetVLAD parameters make a weak test (descriptors are dominated by the centroid term and
    differ by ~1e-6 between images, SURVEY 7).  With _init_params-style parameters (unit-norm centroids,
    alpha ~ 280) the descriptor depends sharply on the feature map; this is the realistic case and the one
    where the bf16x3 error is largest (measured 7e-5).  Tolerance: the north-star 1e-4."""
    sd = synth.make_state_dict(seed=11, sharp=True, with_pca=False, bias_scale=0.02)
    _bind(eng, sd)
    x = synth.make_images(seed=12, batch=6, height=64, width=96)
    with torch.no_grad():
        _, want = O.embednet_forward(x, sd)
    for name, mode, _ in _modes():
        eng.conv_mode = mode
        got, _ = eng.extract(x.cuda(), pca=False)
        per_image = ((got.cpu().double() - want.double()).norm(dim=1) / want.double().norm(dim=1)).max().item()
        assert per_image < DESC_TOL, (name, per_image)
    # and the images really are distinguishable: pairwise distances are O(1e-2), not O(1e-6)
    d = O.self_distance(want)
    assert float(d[~torch.eye(6, dtype=torch.bool)].min()) > 1e-3


def test_shapes_tokyo_like_and_microbatching(eng, O):
    """Tokyo 24/7 queries arrive one at a time with arbitrary sizes (examples/test.py:44-48: batch 1,
    Resize(max(h,w))); large batches are split into micro-batches of 32 inside ibl_extract; the host entry
    point splits a batch >= 16 into two parts to overlap the copy.  All against the oracle."""
    sd = synth.make_state_dict(seed=17, sharp=True, with_pca=True, pca_dim=256, bias_scale=0.02)
    _bind(eng, sd)
    for (n, h, w) in ((1, 112, 80), (1, 83, 131), (3, 48, 208)):
        x = synth.make_images(seed=31 + h, batch=n, height=h, width=w)
        with torch.no_grad():
            want = O.embednetpca_forward(x, sd)
        got, _ = eng.extract(x.cuda(), pca=True)
        assert got.shape == want.shape
        assert rel_l2(got.cpu(), want) < DESC_TOL, (n, h, w, rel_l2(got.cpu(), want))
    x = synth.make_images(seed=40, batch=37, height=32, width=48)          # 32 + 5 micro-batches
    with torch.no_grad():
        want = O.embednetpca_forward(x, sd)
    got, pool = eng.extract(x.cuda(), pca=True, want_pool=True)
    assert rel_l2(got.cpu(), want) < DESC_TOL and tuple(pool.shape) == (37, 512)
    out_host = torch.empty(37, 256).pin_memory()
    eng.extract_host(x.pin_memory(), out_host, pca=True)                    # 9 + 28 split with overlapped copy
    assert torch.equal(out_host, got.cpu())
    out_host2 = torch.empty(37, 256)                                        # pageable host memory also works
    eng.extract_host(x, out_host2, pca=True)
    assert torch.equal(out_host2, got.cpu())
    # two-slot pipelined entry point: five batches in flight two at a time, same bits as the blocking call
    xs = [synth.make_images(seed=60 + i, batch=3 + i, height=32, width=48).pin_memory() for i in range(5)]
    outs = [torch.empty(3 + i, 256).pin_memory() for i in range(5)]
    done = list(eng.extract_host_stream(zip(xs, outs), pca=True))
    assert len(done) == 5
    for xh, oh in zip(xs, outs):
        want_i, _ = eng.extract(xh.cuda(), pca=True)
        assert torch.equal(oh, want_i.cpu())


def test_u8_preprocess_bit_exact_and_host_u8_path(eng):
    """SURVEY 8(f) rank 4 (input side): ToTensor + Normalize of get_transformer_test
    (ibl/utils/data/__init__.py:37-42) on the device, bit-identical to the CPU transform, and the uint8 host
    entry point giving exactly the descriptors of the fp32 host entry point."""
    from openibl_b200.utils.data import _MEAN, _STD
    sd = synth.make_state_dict(seed=0, sharp=True, with_pca=True, pca_dim=128)
    _bind(eng, sd)
    gen = torch.Generator().manual_seed(77)
    u8 = torch.randint(0, 256, (18, 48, 64, 3), dtype=torch.uint8, generator=gen)
    # torchvision semantics: ToTensor = HWC uint8 -> CHW float / 255; Normalize = (t - mean) / std
    ref = u8.permute(0, 3, 1, 2).float().div(255)
    ref = (ref - torch.tensor(_MEAN).view(1, 3, 1, 1)) / torch.tensor(_STD).view(1, 3, 1, 1)
    got = eng.preprocess_u8(u8.cuda(), _MEAN, _STD).cpu()
    assert torch.equal(got, ref.contiguous())
    out_f = torch.empty(18, 128).pin_memory()
    out_u = torch.empty(18, 128).pin_memory()
    eng.extract_host(ref.contiguous().pin_memory(), out_f, pca=True)
    eng.extract_host_u8(u8.pin_memory(), out_u, _MEAN, _STD, pca=True)
    assert torch.equal(out_f, out_u)


def test_models_api_drop_in(eng):
    """The nn.Module mirror (what examples/test.py builds, :58-70) gives the golden outputs."""
    from ibl import models
    g = load_golden("small_96x128")
    sd = synth.make_state_dict(seed=5, with_pca=True, pca_dim=128, bias_scale=0.05)
    base = models.create("vgg16", pretrained=False)
    pool_layer = models.create("netvlad", dim=base.feature_dim)
    model = models.create("embednetpca", base, pool_layer, dim=128)
    model.load_state_dict(sd)
    model = model.cuda().eval()
    x = synth.make_images(seed=6, batch=2, height=96, width=128).cuda()
    from openibl_b200.engine import CONV_TC_BF16X3
    eng.conv_mode = CONV_TC_BF16X3
    with torch.no_grad():
        assert rel_l2(model(x).cpu(), g["desc"]) < DESC_TOL
        emb = models.create("embednet", model.base_model, model.net_vlad).cuda().eval()
        pool_x, vlad_x = emb(x)
        assert rel_l2(vlad_x.cpu(), g["vlad"]) < DESC_TOL / 4 and rel_l2(pool_x.cpu(), g["pool"]) < DESC_TOL
        p2, feat = model.base_model(x)
        assert rel_l2(feat.cpu(), g["feat"]) < FEAT_TOL_TC
        raw = model.net_vlad(feat)
        assert rel_l2(raw.cpu(), g["raw_vlad"]) < DESC_TOL / 4
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        model(x.cpu())


# ---------------------------------------------------------------------------------------------
# stage (ii): NetVLAD alone, soft and sharp (alpha ~ 280) softmax, both layouts
# ---------------------------------------------------------------------------------------------
def test_netvlad_unit_soft_and_sharp_vs_reference(eng):
    g = load_golden("netvlad_unit")
    gen = torch.Generator().manual_seed(11)
    feat = (torch.randn(2, 512, 30, 40, generator=gen) * 3.0 + 0.5).cuda()
    for tag, sharp in (("soft", False), ("sharp", True)):
        p = synth.make_netvlad_params(seed=3, sharp=sharp)
        w, c = p["conv_weight"].cuda(), p["centroids"].cuda()
        raw, nrm = eng.netvlad_forward(feat, w, c, nhwc=False, want_raw=True, want_norm=True)
        assert rel_l2(raw.cpu(), g[f"{tag}_raw"]) < 2e-5, tag
        assert rel_l2(nrm.cpu(), g[f"{tag}_vlad"]) < 2e-5, tag
        raw2, nrm2 = eng.netvlad_forward(feat.permute(0, 2, 3, 1).contiguous(), w, c, nhwc=True,
                                         want_raw=True, want_norm=True)
        assert rel_l2(raw2.cpu(), g[f"{tag}_raw"]) < 2e-5, tag
        assert rel_l2(eng.vlad_normalize(raw).cpu(), g[f"{tag}_vlad"]) < 2e-5


def test_netvlad_ragged_sizes_vs_oracle(eng, O):
    gen = torch.Generator().manual_seed(5)
    p = synth.make_netvlad_params(seed=8, sharp=True)
    for (N, h, w) in ((1, 1, 1), (3, 7, 9), (1, 15, 20), (2, 33, 31)):
        feat = torch.randn(N, 512, h, w, generator=gen)
        want = O.netvlad(feat, p["conv_weight"], p["centroids"])
        raw, nrm = eng.netvlad_forward(feat.cuda(), p["conv_weight"].cuda(), p["centroids"].cuda(),
                                       want_raw=True, want_norm=True)
        assert rel_l2(raw.cpu(), want) < 2e-5, (N, h, w)
        assert rel_l2(nrm.cpu(), O.vlad_normalize(want)) < 2e-5
        # NHWC input takes the fused tcgen05 kernel (partial last tile, S < 128, several units per image)
        for mode in (1, 0):
            eng.set_gemm_mode(mode)
            raw2, nrm2 = eng.netvlad_forward(feat.permute(0, 2, 3, 1).contiguous().cuda(), p["conv_weight"].cuda(),
                                             p["centroids"].cuda(), nhwc=True, want_raw=True, want_norm=True)
            assert rel_l2(raw2.cpu(), want) < 3e-5, (N, h, w, mode)
            assert rel_l2(nrm2.cpu(), O.vlad_normalize(want)) < 3e-5, (N, h, w, mode)
    # a full batch: 32 images x 1200 pixels -> 4 units per image on 128 CTAs
    feat = torch.randn(32, 30, 40, 512, generator=gen)
    want = O.netvlad(feat.permute(0, 3, 1, 2), p["conv_weight"], p["centroids"])
    eng.set_gemm_mode(1)
    _, nrm = eng.netvlad_forward(feat.cuda(), p["conv_weight"].cuda(), p["centroids"].cuda(), nhwc=True,
                                 want_raw=False, want_norm=True)
    assert rel_l2(nrm.cpu(), O.vlad_normalize(want)) < 3e-5


def test_netvlad_backward_vs_autograd_oracle(eng, O):
    """SURVEY 8 row a11: gradients of NetVLAD.forward w.r.t. the feature map, the assignment weights and the
    centroids, against torch autograd through the fp64 oracle (quarter-region sizes of the SFRS step: 15x20)."""
    from ibl import models
    gen = torch.Generator().manual_seed(21)
    for sharp, (N, h, w) in ((False, (2, 7, 9)), (True, (3, 15, 20)), (True, (1, 5, 5))):
        p = synth.make_netvlad_params(seed=4, sharp=sharp)
        x = torch.randn(N, 512, h, w, generator=gen) * 2.0 + 0.3
        G = torch.randn(N, 64, 512, generator=gen)
        xd = x.double().requires_grad_(True)
        wd = p["conv_weight"].double().requires_grad_(True)
        cd = p["centroids"].double().requires_grad_(True)
        (O.netvlad(xd, wd, cd) * G.double()).sum().backward()
        layer = models.create("netvlad", dim=512).cuda().train()
        layer.centroids.data.copy_(p["centroids"])
        layer.conv.weight.data.copy_(p["conv_weight"])
        xg = x.cuda().requires_grad_(True)
        out = layer(xg)
        assert out.requires_grad and rel_l2(out.detach().cpu(), O.netvlad(x, p["conv_weight"], p["centroids"])) < 3e-5
        (out * G.cuda()).sum().backward()
        tol = 3e-4 if sharp else 5e-5      # sharp softmax (alpha ~ 280) amplifies fp32 rounding in dz
        assert rel_l2(xg.grad.cpu(), xd.grad) < tol, (sharp, N, h, w, rel_l2(xg.grad.cpu(), xd.grad))
        assert rel_l2(layer.conv.weight.grad.cpu(), wd.grad) < tol, (sharp, rel_l2(layer.conv.weight.grad.cpu(), wd.grad))
        assert rel_l2(layer.centroids.grad.cpu(), cd.grad) < tol, (sharp, rel_l2(layer.centroids.grad.cpu(), cd.grad))


def test_embedregionnet_train_branch_vs_reference(eng):
    """SFRS region branch (netvlad.py:123-207) in train mode against the unmodified reference run on CPU
    (tests/golden/region_train.npz): 9x9 region similarities, region descriptors, and the gradients of a scalar
    loss w.r.t. the NetVLAD parameters (the VGG trunk is frozen here, so only those are compared)."""
    from ibl import models
    g = load_golden("region_train")
    sd = synth.make_state_dict(seed=13, sharp=True, with_pca=False, bias_scale=0.02)
    base = models.create("vgg16", pretrained=False)
    pool = models.create("netvlad", dim=512)
    model = models.create("embedregionnet", base, pool, tuple_size=1)
    model.load_state_dict(sd)
    model = model.cuda().train()
    x = synth.make_images(seed=14, batch=5, height=64, width=96).cuda()
    score, va, vb = model(x)
    assert tuple(score.shape) == (1, 4, 9, 9) and tuple(va.shape) == (1, 1, 9, 32768) and tuple(vb.shape) == (1, 4, 9, 32768)
    assert np.abs(score.detach().cpu().numpy() - g["score"]).max() < 2e-4          # cosine similarities in [-1,1]
    assert rel_l2(va.detach().cpu()[..., ::16], g["vlad_a"]) < DESC_TOL
    assert rel_l2(vb.detach().cpu()[..., ::16], g["vlad_b"]) < DESC_TOL
    loss = (score * torch.from_numpy(g["loss_weights"]).cuda()).sum()
    assert abs(loss.item() - float(g["loss"])) < 2e-3 * max(1.0, abs(float(g["loss"])))
    loss.backward()
    assert rel_l2(model.net_vlad.centroids.grad.cpu(), g["grad_centroids"]) < 2e-3
    assert rel_l2(model.net_vlad.conv.weight.grad.cpu(), g["grad_conv_w"]) < 2e-3
    # eval branch unchanged: (pool, vlad)
    model.eval()
    with torch.no_grad():
        pool_x, vlad_x = model(x)
    assert tuple(pool_x.shape) == (5, 512) and tuple(vlad_x.shape) == (5, 32768)


# ---------------------------------------------------------------------------------------------
# stage (iii-a): PCA-whiten + L2
# ---------------------------------------------------------------------------------------------
GEMM_MODES = [("simt", 0, 1e-5), ("tc", 1, 3e-5)]   # (name, ibl gemm mode, rel-L2 tolerance)


@pytest.fixture(autouse=True)
def _default_modes(eng):
    yield
    eng.set_gemm_mode(1)
    eng.conv_mode = 1


def test_pca_unit_vs_reference(eng):
    g = load_golden("pca_unit")
    p = synth.make_pca_params(seed=9, in_dim=32768, out_dim=64)
    gen = torch.Generator().manual_seed(12)
    v = torch.nn.functional.normalize(torch.randn(5, 32768, generator=gen), dim=1)
    w, b = p["weight"].cuda(), p["bias"].cuda()
    for name, mode, tol in GEMM_MODES:
        eng.set_gemm_mode(mode)
        eng._pca_key = None
        eng.set_pca(w, b)                       # registers (and, for tcgen05, re-lays-out) W
        out = eng.pca_l2(v.cuda(), w, b)
        assert rel_l2(out.cpu(), g["out"]) < tol, name


def test_pca_fit_load_infer_roundtrip_vs_oracle(eng, O, tmp_path):
    """SURVEY 8(f) rank 2: PCA.train on the GPU (pca.py:28-84), PCA.load (pca.py:86-106), PCA.infer
    (pca.py:108-123) end to end.  Eigenvector signs are arbitrary, so the whitened outputs are compared
    through sign-invariant quantities: |y| per component and all pairwise distances."""
    from openibl_b200.pca import PCA
    gen = torch.Generator().manual_seed(31)
    # covariance branch (n_dims <= n_pts) and dual branch (n_dims > n_pts, what examples/test.py:108-121 hits with
    # 10k x 32768 descriptors); both on the engine's fp32 GEMM (ibl_gemm_nt) + torch.linalg.eigh
    for n_pts, n_dims, P in ((700, 512, 64), (150, 1024, 32)):
        basis = torch.randn(n_dims, n_dims, generator=gen)
        x = (torch.randn(n_pts, n_dims, generator=gen) * torch.logspace(0, -2, n_dims)) @ basis
        x = torch.nn.functional.normalize(x + 0.1 * torch.randn(n_dims, generator=gen), dim=1)
        pca = PCA(pca_n_components=P, pca_whitening=True, pca_parameters_path=str(tmp_path / f"pca{n_pts}.h5"))
        pca.train(x.cuda())
        pca.load(gpu=0)
        assert tuple(pca.weight.shape) == (P, n_dims, 1, 1) and tuple(pca.bias.shape) == (P,)
        q = x[:50].cuda()
        got = pca.infer(q).cpu()
        U, lams, mu, _ = O.pca_train(x.clone(), n_components=P)
        w, b = O.pca_load(U, lams, mu, n_components=P)
        want = O.pca_whiten(x[:50], w, b)
        assert rel_l2(got.abs(), want.abs()) < 2e-3, (n_pts, rel_l2(got.abs(), want.abs()))
        dg, dw = torch.cdist(got.double(), got.double()), torch.cdist(want.double(), want.double())
        assert float((dg - dw).abs().max()) < 2e-3
    # the GEMM entry point itself, both math modes, ragged inner dimension (zero-padded to 64)
    a, bm = torch.randn(70, 333, generator=gen), torch.randn(45, 333, generator=gen)
    for mode, tol in ((0, 2e-6), (1, 2e-5)):
        c = eng.gemm_nt(a.cuda(), bm.cuda(), alpha=0.5, mode=mode).cpu()
        assert rel_l2(c, 0.5 * (a.double() @ bm.double().t())) < tol, mode


def test_pca_full_size_vs_oracle(eng, O):
    p = synth.make_pca_params(seed=1, in_dim=32768, out_dim=4096)
    gen = torch.Generator().manual_seed(13)
    w, b = p["weight"].cuda(), p["bias"].cuda()
    eng._pca_key = None
    eng.set_pca(w, b)
    for n in (1, 33):
        v = torch.nn.functional.normalize(torch.randn(n, 32768, generator=gen), dim=1)
        want = O.pca_whiten(v, p["weight"], p["bias"])
        for name, mode, tol in GEMM_MODES:
            eng.set_gemm_mode(mode)
            got = eng.pca_l2(v.cuda(), w, b)
            assert rel_l2(got.cpu(), want) < tol, (name, n)
    from openibl_b200.pca import PCA
    pca = PCA(4096)
    pca.weight, pca.bias = w, b
    assert rel_l2(pca.infer(v.cuda()).cpu(), want) < 3e-5


# ---------------------------------------------------------------------------------------------
# stage (iii-b): distance, top-k, merge, recall
# ---------------------------------------------------------------------------------------------
def test_retrieval_vs_reference_golden(eng):
    from openibl_b200.evaluators import evaluate_all, pairwise_distance, recalls_from_topk
    g = load_golden("retrieval")
    q, db, gt = synth.make_gallery(n_db=1500, n_q=300, dim=512, sigma=0.28)
    for name, mode, _ in GEMM_MODES:
        eng.set_gemm_mode(mode)
        d = eng.l2dist_dense(q.cuda(), db.cuda())
        # dense matrix: fp32 CUDA cores 2e-5 abs; tcgen05 bf16x3 (no re-scoring on this path) 1e-4 abs
        assert np.abs(d[:32].cpu().numpy() - g["dist_sub"]).max() < (2e-5 if mode == 0 else 1e-4), name
        dk, ik = eng.l2dist_topk(q.cuda(), db.cuda(), 10)     # top-k is re-scored in exact fp32
        assert np.array_equal(ik.cpu().numpy(), g["top10"]), name
        assert np.abs(dk.cpu().numpy() - g["top10_dist"]).max() < 2e-5, name
    gallery = [("d%05d" % i, i // 3, 0.0, 0.0) for i in range(1500)]
    query = [("q%05d" % i, i, 0.0, 0.0) for i in range(300)]
    gt_list = [np.array([int(t)]) for t in gt]
    assert np.array_equal(recalls_from_topk(ik.cpu().numpy(), gt_list, gallery), g["recalls"])
    _, i120 = eng.l2dist_topk(q.cuda(), db.cuda(), 120)
    assert np.array_equal(recalls_from_topk(i120.cpu().numpy(), gt_list, gallery, nms=True), g["recalls_nms"])
    # reference-shaped API: features dict -> dense matrix -> recalls
    feats = {f: r for (f, _, _, _), r in zip(query, q)}
    feats.update({f: r for (f, _, _, _), r in zip(gallery, db)})
    dm, xq, yg = pairwise_distance(feats, query, gallery)
    assert dm.shape == (300, 1500) and not dm.is_cuda and xq.shape == (300, 512)
    assert np.array_equal(evaluate_all(dm, gt_list, gallery), g["recalls"])
    sub = {k: feats[k] for k in list(feats)[:64]}
    sd_, _, _ = pairwise_distance(sub)
    assert np.abs(sd_.numpy() - g["self_dist"]).max() < 2e-5


def test_rerank_on_gpu_distances_vs_reference_golden(eng):
    """Evaluator.evaluate(rerank=True) path (evaluators.py:194-199): dense q-g / q-q / g-g distances from the
    tcgen05 dense kernel, k-reciprocal re-ranking on the device; against the unmodified reference function run on
    the reference's own fp32 distances (tests/golden/rerank.npz)."""
    from openibl_b200.utils.rerank import re_ranking
    g = load_golden("rerank")
    for name in "abc":
        k1, k2, lam = g[f"{name}_params"]
        q, db = torch.from_numpy(g[f"{name}_q"]).cuda(), torch.from_numpy(g[f"{name}_db"]).cuda()
        pad = (-q.shape[1]) % 64                     # the tensor-core distance path wants dim % 64 == 0
        if pad:
            q, db = torch.nn.functional.pad(q, (0, pad)), torch.nn.functional.pad(db, (0, pad))
        qg, qq, gg = eng.l2dist_dense(q, db), eng.l2dist_dense(q, q), eng.l2dist_dense(db, db)
        # |x|^2 + |y|^2 - 2xy on values of 2-3: a few fp32 ulps between two evaluation orders
        assert float((qg.cpu() - torch.from_numpy(g[f"{name}_qg"])).abs().max()) < 3e-5
        out = re_ranking(qg, qq, gg, k1=int(k1), k2=int(k2), lambda_value=float(lam))
        assert out.is_cuda
        ref = torch.from_numpy(g[f"{name}_final"])
        # a near-tie in a neighbour list may flip under 1e-6 distance noise and move a few entries; the bulk agrees
        close = ((out.cpu() - ref).abs() < 1e-4).float().mean()
        assert close > 0.995, (name, float(close))


def test_topk_edge_cases(eng, O):
    q, db, _ = synth.make_gallery(n_db=700, n_q=9, dim=64, sigma=0.5)
    qd, dbd = q.cuda(), db.cuda()
    d = O.pairwise_distance(q, db).numpy()
    for name, mode, _ in GEMM_MODES:
        eng.set_gemm_mode(mode)
        _topk_edge_cases(eng, O, q, db, qd, dbd, d)


def test_topk_raw_vlad_dim_32768(eng, O):
    """--vlad without --reduction ranks the 32768-d descriptors directly (examples/test.py:127-131)."""
    q, db, _ = synth.make_gallery(n_db=300, n_q=9, dim=32768, sigma=0.02)
    d = O.pairwise_distance(q, db).numpy()
    wd, wi = O.topk_from_distmat(d, 10)
    for name, mode, _ in GEMM_MODES:
        eng.set_gemm_mode(mode)
        dk, ik = eng.l2dist_topk(q.cuda(), db.cuda(), 10)
        assert np.array_equal(ik.cpu().numpy(), wi), name
        assert np.allclose(dk.cpu().numpy(), wd, atol=2e-5), name


def _topk_edge_cases(eng, O, q, db, qd, dbd, d):
    # k = 1, k = 12/13 (register top-16 vs dense path), k = 128, padded shard, idx_base, duplicates
    for k in (1, 12, 13, 128):
        dk, ik = eng.l2dist_topk(qd, dbd, k)
        wd, wi = O.topk_from_distmat(d, k)
        assert np.array_equal(ik.cpu().numpy(), wi) and np.allclose(dk.cpu().numpy(), wd, atol=1e-5), k
    dk, ik = eng.l2dist_topk(qd, dbd, 10, idx_base=5000, n_valid=333)
    wd, wi = O.topk_from_distmat(d[:, :333], 10)
    assert np.array_equal(ik.cpu().numpy(), wi + 5000)
    dup = torch.cat([db[:50], db[:50]]).cuda()
    _, ik = eng.l2dist_topk(qd, dup, 4)
    ik = ik.cpu().numpy()
    assert (ik[:, 0] < 50).all() and (ik[:, 1] == ik[:, 0] + 50).all()
    # fewer valid rows than k: padded with (inf, -1)
    dk, ik = eng.l2dist_topk(qd, dbd, 10, n_valid=3)
    assert (ik[:, 3:] == -1).all() and torch.isinf(dk[:, 3:]).all() and (ik[:, :3] >= 0).all()
    # merge of shard candidates == ranking of the whole
    parts = [eng.l2dist_topk(qd, dbd[lo:lo + 175].contiguous(), 10, idx_base=lo) for lo in range(0, 700, 175)]
    md, mi = eng.topk_merge(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]), 10)
    wd, wi = O.topk_from_distmat(d, 10)
    assert np.array_equal(mi.cpu().numpy(), wi)


def test_retrieval_pitts30k_shape_properties(eng):
    """configs[2] size: 6.8k x 10k x 4096.  Size-independent properties + a subset against torch fp64."""
    q, db, gt = synth.make_gallery(10000, 6800, 4096)
    qd, dbd = q.cuda(), db.cuda()
    eng.set_gemm_mode(0)
    dk0, ik0 = eng.l2dist_topk(qd, dbd, 10)                           # fp32 CUDA cores
    eng.set_gemm_mode(1)
    dk, ik = eng.l2dist_topk(qd, dbd, 10)                             # tcgen05 + exact re-scoring
    assert eng.dist_flagged() <= 6800 // 200                           # the guard's exact fallback stays rare
    assert float((ik == ik0).float().mean()) > 0.999
    assert float((dk - dk0).abs().max()) < 5e-6
    dk120, ik120 = eng.l2dist_topk(qd[:512].contiguous(), dbd, 120)    # dense-tile path (Tokyo nms, k=120)
    assert bool((ik120[:, :10] == ik[:512]).float().mean() > 0.999)
    assert bool((dk[:, 1:] >= dk[:, :-1]).all())                       # sorted ascending
    assert int(ik.min()) >= 0 and int(ik.max()) < 10000
    assert bool((ik.sort(dim=1).values[:, 1:] != ik.sort(dim=1).values[:, :-1]).all())   # no duplicates
    sel = torch.arange(0, 6800, 97, device="cuda")
    exact = (2 - 2 * (qd[sel].double() @ dbd.double().t()))
    wd, wi = exact.topk(10, largest=False)
    got_d = dk[sel].double()
    assert float((got_d - wd).abs().max()) < 5e-6
    agree = float((ik[sel] == wi).float().mean())
    assert agree > 0.99, agree                                          # near-ties may swap at 1e-7
    # recall on the planted positives is identical to the exact ranking's
    from openibl_b200.evaluators import recalls_from_topk
    gallery = [("d%06d" % i, i, 0, 0) for i in range(10000)]
    gl = [np.array([int(t)]) for t in gt[sel.cpu()]]
    assert np.array_equal(recalls_from_topk(ik[sel].cpu().numpy(), gl, gallery),
                          recalls_from_topk(wi.cpu().numpy(), gl, gallery))


def test_retrieval_pitts250k_shard_shape(eng):
    """configs[3] per-GPU shape: 6.8k queries x one 31,250-row shard (250k / 8) x 4096, with the
    DistributedSliceSampler padding masked out (n_valid < n) and a non-zero index base.  Checked against
    an exact fp64 ranking of a query subset and by merging two half-shards."""
    n, n_valid, base = 31250, 31000, 3 * 31250
    q, db, gt = synth.make_gallery(n, 6800, 4096, seed_db=7, seed_q=8)
    qd, dbd = q.cuda(), db.cuda()
    dk, ik = eng.l2dist_topk(qd, dbd, 10, idx_base=base, n_valid=n_valid)
    assert eng.dist_flagged() <= 6800 // 200                           # the guard's exact fallback stays rare
    assert bool((dk[:, 1:] >= dk[:, :-1]).all())
    assert int(ik.min()) >= base and int(ik.max()) < base + n_valid
    sel = torch.arange(0, 6800, 211, device="cuda")
    exact = 2 - 2 * (qd[sel].double() @ dbd[:n_valid].double().t())
    wd, wi = exact.topk(10, largest=False)
    assert float((dk[sel].double() - wd).abs().max()) < 5e-6
    assert float((ik[sel] == wi + base).float().mean()) > 0.99
    h = n_valid // 2
    a = eng.l2dist_topk(qd, dbd[:h].contiguous(), 10, idx_base=base)
    b = eng.l2dist_topk(qd, dbd[h:n_valid].contiguous(), 10, idx_base=base + h)
    md, mi = eng.topk_merge(torch.stack([a[0], b[0]]), torch.stack([a[1], b[1]]), 10)
    assert float((mi == ik).float().mean()) > 0.9995 and float((md - dk).abs().max()) < 5e-6


# ---------------------------------------------------------------------------------------------
# batch-32 480x640 (configs[1]): size-independent properties
# ---------------------------------------------------------------------------------------------
def test_batch_480x640_properties(eng):
    from openibl_b200.engine import CONV_SIMT_FP32, CONV_TC_BF16X3
    sd = synth.make_state_dict(seed=0, with_pca=True)
    _bind(eng, sd)
    x = synth.make_images(seed=21, batch=5)
    xd = x.cuda()
    eng.conv_mode = CONV_TC_BF16X3
    desc, _ = eng.extract(xd, pca=True)
    assert float((desc.norm(dim=1) - 1).abs().max()) < 1e-5
    # batch independence: image i alone gives the same row (bitwise: same kernels, same tiles)
    one, _ = eng.extract(xd[3:4].contiguous(), pca=True)
    assert rel_l2(one.cpu(), desc[3:4].cpu()) < 1e-6
    # tensor-core path vs the fp32 CUDA-core path on the device, full size
    eng.conv_mode = CONV_SIMT_FP32
    desc32, _ = eng.extract(xd, pca=True)
    eng.conv_mode = CONV_TC_BF16X3
    assert rel_l2(desc.cpu(), desc32.cpu()) < DESC_TOL
    # host-buffer entry point == device entry point
    out_host = torch.empty(5, 4096).pin_memory()
    eng.extract_host(x.pin_memory(), out_host, pca=True)
    assert torch.equal(out_host, desc.cpu())
    assert eng.launch_count > 0


# ---------------------------------------------------------------------------------------------
# configs[1] at its real size against the ORACLE (not only self-consistency)
# ---------------------------------------------------------------------------------------------
def test_batch32_480x640_vs_oracle_both_conv_modes(eng, O):
    """The benchmarked shape -- 32 images of 3x480x640 through ibl_extract (VGG16 + NetVLAD + PCA 4096) -- in both
    conv math modes against oracle.extract_descriptor (reference forward, evaluators.py:22-34 + netvlad.py:95-110)
    on the host cores.  Per-image relative L2 <= 1e-4 (north star)."""
    sd = synth.make_state_dict(seed=0, with_pca=True)
    _bind(eng, sd)
    x = synth.make_images(seed=1, batch=32)
    torch.set_num_threads(max(1, min(64, (torch.get_num_threads() or 1))))
    with torch.no_grad():
        want = O.extract_descriptor(x, sd).double()
    xd = x.cuda()
    for name, mode, _ in _modes():
        eng.conv_mode = mode
        got, _ = eng.extract(xd, pca=True)
        per_image = ((got.cpu().double() - want).norm(dim=1) / want.norm(dim=1))
        assert float(per_image.max()) < DESC_TOL, (name, float(per_image.max()))
    # the golden (unmodified reference, batch 1) is image 0 of this batch
    g = load_golden("hub_480x640")
    assert rel_l2(got[:1].cpu(), g["desc"]) < DESC_TOL


def test_sharp_full_chain_480x640_vs_oracle(eng, O):
    """_init_params-style NetVLAD parameters (alpha ~ 280) at the REAL size (S = 1200 locations): the case where
    the bf16x3 representation error of the feature map is amplified most (7e-5 at 64x96).  Raw 32768-d VLAD and
    PCA'd descriptors, per image, <= 1e-4."""
    sd = synth.make_state_dict(seed=11, sharp=True, with_pca=True, bias_scale=0.02)
    _bind(eng, sd)
    x = synth.make_images(seed=12, batch=4)
    with torch.no_grad():
        _, want_v = O.embednet_forward(x, sd)
        want_p = O.pca_whiten(want_v, sd["pca_layer.weight"], sd["pca_layer.bias"])
    worst = {}
    for name, mode, _ in _modes():
        eng.conv_mode = mode
        got_v, _ = eng.extract(x.cuda(), pca=False)
        got_p, _ = eng.extract(x.cuda(), pca=True)
        ev = ((got_v.cpu().double() - want_v.double()).norm(dim=1) / want_v.double().norm(dim=1)).max().item()
        ep = ((got_p.cpu().double() - want_p.double()).norm(dim=1) / want_p.double().norm(dim=1)).max().item()
        worst[name] = (ev, ep)
        assert ev < DESC_TOL and ep < DESC_TOL, worst
    print("sharp 480x640 per-image rel-L2 (vlad, pca):", worst)
    d = O.self_distance(want_v)
    assert float(d[~torch.eye(4, dtype=torch.bool)].min()) > 1e-3     # the images are distinguishable


def test_evaluate_all_large_k_and_engine_cache_invalidation(eng, O):
    """evaluate_all with recall_topk beyond 128 ranks (advisor finding: used to return zeros silently) and the
    explicit cache invalidation for `.data` writes that do not bump Tensor._version."""
    from openibl_b200.evaluators import evaluate_all
    from openibl_b200.engine import invalidate_caches
    q, db, gt = synth.make_gallery(n_db=3000, n_q=40, dim=64, sigma=1.5)
    d = O.pairwise_distance(q, db).numpy()
    gallery = [("d%05d" % i, i // 2, 0.0, 0.0) for i in range(3000)]
    gt_list = [np.array([int(t)]) for t in gt]
    for topk, nms in (([1, 5, 10, 20], True), ([1, 100, 500], False)):
        want = O.evaluate_all(d, gt_list, [g[1] for g in gallery], recall_topk=tuple(topk), nms=nms)
        got = evaluate_all(torch.from_numpy(d), gt_list, gallery, recall_topk=topk, nms=nms)
        assert np.array_equal(got, want), (topk, nms, got, want)
    dk, ik = eng.topk_rows(torch.from_numpy(d).cuda(), 1000)
    wd, wi = O.topk_from_distmat(d, 1000)
    assert np.array_equal(ik.cpu().numpy(), wi)
    with pytest.raises(NotImplementedError):
        evaluate_all(torch.from_numpy(d), gt_list, gallery, recall_topk=[2000])
    # cache invalidation
    sd = synth.make_state_dict(seed=5, with_pca=True, pca_dim=128, bias_scale=0.05)
    sdd = _bind(eng, sd)
    x = synth.make_images(seed=6, batch=1, height=64, width=96).cuda()
    a, _ = eng.extract(x, pca=True)
    w0 = sdd["base_model.base.0.weight"]
    w0.data.mul_(1.5)                                  # no version bump
    slots = synth.VGG16_CONV_SLOTS
    ws, bs = [sdd[f"base_model.base.{s}.weight"] for s in slots], [sdd[f"base_model.base.{s}.bias"] for s in slots]
    invalidate_caches()
    eng.set_vgg16(ws, bs)
    b, _ = eng.extract(x, pca=True)
    assert rel_l2(a.cpu(), b.cpu()) > 1e-4             # the new weights are in effect
    sd2 = dict(sd)
    sd2["base_model.base.0.weight"] = sd["base_model.base.0.weight"] * 1.5
    with torch.no_grad():
        want = O.embednetpca_forward(x.cpu(), sd2)
    assert rel_l2(b.cpu(), want) < DESC_TOL


def test_descriptor_is_bit_identical_across_batch_compositions(eng):
    """An image's descriptor must not depend on the batch it travels in (tile shapes, NetVLAD units per image and
    PCA split-K are functions of the image size only): that is what makes the 250k gallery rank identically on 1 and
    8 GPUs, whose slices end in different tail batches."""
    sd = synth.make_state_dict(seed=2, sharp=True, with_pca=True, pca_dim=256, bias_scale=0.02)
    _bind(eng, sd)
    for (h, w) in ((64, 96), (480, 640)):
        n = 37 if h == 64 else 33
        x = synth.make_images(seed=50, batch=n, height=h, width=w).cuda()
        full, _ = eng.extract(x, pca=True)
        full_v, _ = eng.extract(x, pca=False)
        for lo, hi in ((0, 1), (3, 10), (n - 18, n)):
            part, _ = eng.extract(x[lo:hi].contiguous(), pca=True)
            part_v, _ = eng.extract(x[lo:hi].contiguous(), pca=False)
            assert torch.equal(part_v, full_v[lo:hi]), (h, lo, hi, "vlad")
            assert torch.equal(part, full[lo:hi]), (h, lo, hi, "pca")


def test_single_pass_screening_guard_and_exact_fallback(eng, O):
    """The distance/top-k path screens with ONE fp16 tensor-core pass and decides in exact fp32.  (a) On descriptor-like
    data the guard never fires and the ranking equals the oracle's.  (b) On an adversarial database -- 40 near-copies
    of every query's positive, 1e-6 apart, far more than the 16 survivors a query keeps -- the guard must fire, and
    the exact brute-force fallback must give the oracle's ranking (fp32 distances, ties to the lowest index)."""
    q, db, gt = synth.make_gallery(n_db=5000, n_q=300, dim=512, sigma=0.28)
    d = O.pairwise_distance(q, db).numpy()
    wd, wi = O.topk_from_distmat(d, 10)
    dk, ik = eng.l2dist_topk(q.cuda(), db.cuda(), 10)
    assert eng.dist_flagged() == 0
    assert np.array_equal(ik.cpu().numpy(), wi) and np.allclose(dk.cpu().numpy(), wd, atol=2e-5)
    # adversarial: clusters of near-duplicates
    gen = torch.Generator().manual_seed(3)
    centers = torch.nn.functional.normalize(torch.randn(60, 256, generator=gen), dim=1)
    db2 = (centers.repeat_interleave(40, dim=0) + 1e-6 * torch.randn(2400, 256, generator=gen)).contiguous()
    q2 = torch.nn.functional.normalize(centers.repeat(3, 1) + 0.05 * torch.randn(180, 256, generator=gen), dim=1).contiguous()
    d2 = O.pairwise_distance(q2, db2).numpy()
    dk2, ik2 = eng.l2dist_topk(q2.cuda(), db2.cuda(), 10, idx_base=7)
    flagged = eng.dist_flagged()
    assert flagged > 0, "the guard must notice that 16 survivors cannot cover 40 near-ties"
    got_d, got_i = dk2.cpu().numpy(), ik2.cpu().numpy() - 7
    # distances are exact fp32 either way; indices may differ from the fp32-GEMM oracle only inside exact ties
    wd2, wi2 = O.topk_from_distmat(d2, 10)
    assert np.allclose(got_d, wd2, atol=3e-6)
    eng.set_gemm_mode(0)                                       # fp32 CUDA-core path: same arithmetic family as the fallback
    dk3, ik3 = eng.l2dist_topk(q2.cuda(), db2.cuda(), 10, idx_base=7)
    eng.set_gemm_mode(1)
    assert np.allclose(got_d, dk3.cpu().numpy(), atol=3e-6)
    # every returned neighbour really has the distance it claims (exact fp64 check) and belongs to the right cluster
    exact = ((q2.double().unsqueeze(1) - db2.double()[torch.from_numpy(got_i)]) ** 2).sum(-1).numpy()
    assert np.abs(exact - got_d).max() < 5e-6
    assert (got_i // 40 == (np.arange(180) % 60)[:, None]).all()


def test_gpu_resize_matches_pillow_bit_exact(eng):
    """SURVEY 8 f4: T.Resize((H, W)) of the reference's test transform (utils/data/__init__.py:37-42) on the GPU,
    bit-identical to PIL.Image.resize(..., BILINEAR): down- and up-scaling, odd sizes, one-axis-only, identity, and
    then ToTensor + Normalize on the device equal to the torchvision pipeline on the CPU."""
    from PIL import Image
    import torchvision.transforms as T
    from openibl_b200.utils.data import _MEAN, _STD, get_transformer_test
    rng = np.random.RandomState(0)
    for (h, w, oh, ow) in ((120, 160, 96, 128), (37, 53, 64, 96), (480, 640, 480, 640), (300, 451, 480, 640),
                           (768, 1024, 480, 640), (50, 50, 17, 200), (90, 128, 96, 128), (96, 130, 96, 128)):
        imgs = rng.randint(0, 256, size=(3, h, w, 3)).astype(np.uint8)
        want = np.stack([np.asarray(Image.fromarray(im).resize((ow, oh), Image.BILINEAR)) for im in imgs])
        got = eng.resize_u8(torch.from_numpy(imgs).cuda(), oh, ow)
        assert torch.equal(got.cpu(), torch.from_numpy(want)), (h, w, oh, ow)
    tf = get_transformer_test(96, 128)
    ref = torch.stack([tf(Image.fromarray(im)) for im in imgs])
    dev = eng.preprocess_u8(eng.resize_u8(torch.from_numpy(imgs).cuda(), 96, 128), _MEAN, _STD)
    assert torch.equal(dev.cpu(), ref)


def test_device_argsort_rows_and_sampler_refresh(eng):
    """SURVEY 8 f3: the samplers' `torch.argsort(distmat, dim=1)` (sampler.py:49,129) on the device -- short rows
    (shared-memory bitonic), long rows (chunk sort + merge passes), exact ties -- and the tuple samplers refreshed
    through it yield the reference's tuples (tests/golden/sampler.npz)."""
    import random
    from ibl.utils.data.sampler import DistributedRandomTupleSampler, DistributedRandomDiffTupleSampler
    gen = torch.Generator().manual_seed(1)
    for (m, n) in ((5, 1), (7, 150), (3, 10000), (2, 16384), (3, 16385), (2, 70001)):
        d = torch.rand(m, n, generator=gen)
        d[:, n // 3] = d[:, n // 2]                                   # a tie per row
        want = torch.argsort(d, dim=1, stable=True)
        got = eng.argsort_rows(d.cuda()).cpu()
        assert torch.equal(got, want), (m, n)
    g = load_golden("sampler")
    NQ, NG = g["dist"].shape
    q = [("q%03d" % i, i, 0.0, 0.0) for i in range(NQ)]
    gal = [("g%03d" % i, 1000 + i, 0.0, 0.0) for i in range(NG)]
    pos_l, neg_l = [p.tolist() for p in g["pos"]], [sorted(set(n.tolist())) for n in g["neg"]]
    sub = list(range(3, NQ, 2))
    for name, cls, kw in (("tuple", DistributedRandomTupleSampler, dict(neg_num=4, neg_pool=30)),
                          ("diff", DistributedRandomDiffTupleSampler, dict(pos_num=3, pos_pool=5, neg_num=4, neg_pool=30))):
        s = cls(q, gal, pos_l, neg_l, num_replicas=2, rank=1, **kw)
        random.seed(12)
        if name == "tuple":
            s.sort_gallery(torch.from_numpy(g["dist"]), sub)
        else:
            s.sort_gallery(torch.from_numpy(g["dist"]).cuda(), torch.from_numpy(g["jac"]), sub)
        assert torch.equal(s.sort_idx, torch.from_numpy(g["sort_idx"]))
        for ep in (0, 1):
            got = np.asarray([r + [-1] * (9 - len(r)) for r in iter(s)], dtype=np.int64)
            assert np.array_equal(got, g[f"{name}_r1_e{ep}"]), (name, ep)
