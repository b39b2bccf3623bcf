"""Kernel variants that are selected by environment variables (read once per process) are exercised in child
processes, each running the relevant subset of the parity tests: every staging / pairing mode of the tcgen05
conv and the one-SM distance kernel must give the same answers as the defaults.  Also pins the hardware property the halo-staged conv relies on."""
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

VARIANTS = [
    # env, -k expression[, test file (default test_gpu_parity.py)]
    ({"IBL_CONV_HALO": "2"}, "conv3x3 or small or odd"),                    # halo staging on every N tile
    ({"IBL_CONV_HALO": "0", "IBL_CONV_2SM": "0"}, "conv3x3 or small or odd"),   # im2col boxes, one SM per tile
    ({"IBL_CONV_2SM": "2", "IBL_CONV_HALO": "0"}, "conv3x3 or odd"),        # SM pairs on the 128-wide tiles too
    ({"IBL_CONV1_FUSED": "0"}, "small or odd or hub or tokyo"),             # separate conv1_1 / conv1_2 kernels
    ({"IBL_CONV1_FUSED": "0", "IBL_CONV1_SIMT": "1"}, "small or odd"),      # ... with the CUDA-core conv1_1
    ({"IBL_DIST_BN": "512"}, "retrieval or topk or single_pass"),            # 256 x 512 screening tiles, one accumulator
    ({"IBL_DIST_SCREEN": "3"}, "retrieval or topk"),                         # round-1 bf16x3 screening on SM pairs
    ({"IBL_DIST_SCREEN": "3", "IBL_DIST_2SM": "0"}, "retrieval_vs_reference or topk"),   # ... on one SM
    ({"IBL_DIST_SCREEN": "3", "IBL_DIST_2SM": "0", "IBL_DIST_BN": "128", "IBL_GEMM_MC": "1"}, "retrieval_vs_reference or topk"),
    # the crafted rankings of test_gpu_rank_rounding.py on every screening variant
    ({"IBL_DIST_BN": "512"}, "topk or dist_flagged", "test_gpu_rank_rounding.py"),
    ({"IBL_DIST_SCREEN": "3"}, "topk or dist_flagged", "test_gpu_rank_rounding.py"),
    ({"IBL_DIST_SCREEN": "3", "IBL_DIST_2SM": "0"}, "topk or dist_flagged", "test_gpu_rank_rounding.py"),
]


def _variant_id(v):
    ident = ",".join(f"{k}={val}" for k, val in v[0].items())
    return ident if len(v) == 2 else ident + ":" + v[2].replace("test_gpu_", "").replace(".py", "")


@pytest.mark.gpu
@pytest.mark.parametrize("variant", VARIANTS, ids=[_variant_id(v) for v in VARIANTS])
def test_variant_matches_references(variant):
    env, expr = variant[:2]
    test_file = variant[2] if len(variant) > 2 else "test_gpu_parity.py"
    child_env = dict(os.environ)
    child_env.update(env)
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(ROOT, "tests", test_file), "-q", "-x",
                        "-k", expr, "-p", "no:cacheprovider"], cwd=ROOT, env=child_env, capture_output=True, text=True,
                       timeout=600)
    tail = (r.stdout + r.stderr)[-2000:]
    assert r.returncode == 0, tail
    assert " passed" in r.stdout and "failed" not in r.stdout, tail


@pytest.mark.gpu
def test_umma_sw128_operand_accepts_unaligned_start_and_odd_group_stride():
    """tc_conv.cu's halo staging reads nine tap views out of one TMA-written tile: starts that are 128-byte but
    not 1024-byte aligned, 8-row groups 10 rows apart, descriptor base_offset = 0."""
    from openibl_b200.engine import Engine, _ptr, _stream
    from openibl_b200._cabi import check
    eng = Engine.get(0)
    g = torch.Generator(device="cuda").manual_seed(5)
    rows = 200
    A = torch.randint(-8, 9, (rows, 64), device="cuda", generator=g).to(torch.bfloat16)
    B = torch.randint(-8, 9, (64, 64), device="cuda", generator=g).to(torch.bfloat16)
    D = torch.empty(128, 64, device="cuda")
    m = torch.arange(128, device="cuda")
    for group_rows, s0 in ((8, 0), (10, 0), (10, 1), (10, 11), (10, 22), (12, 3)):
        idx = s0 + (m // 8) * group_rows + (m % 8)
        want = A[idx].float() @ B.float().t()
        check(eng.lib.ibl_debug_umma_strided(eng.h, _ptr(A), rows, _ptr(B), s0, group_rows, 0, _ptr(D), _stream(0)), "probe")
        torch.cuda.synchronize()
        assert torch.equal(D, want), (group_rows, s0)
