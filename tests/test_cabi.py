"""The C-ABI shared library loads and exports every symbol include/pgmuvi_b200.h declares;
argument validation works without a GPU (no compute launches here)."""
import ctypes
import os
import re

import pytest

from conftest import ROOT
from pgmuvi_b200 import _lib

HEADER = os.path.join(ROOT, "include", "pgmuvi_b200.h")


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(pgm_[a-z0-9_]+)\s*\(", src)))


def test_header_and_binding_agree():
    assert set(declared_symbols()) == set(_lib.EXPORTS)


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    for sym in declared_symbols():
        assert hasattr(lib, sym), f"{sym} missing from {_lib.LIB_PATH}"
    assert lib.pgm_version() >= 100


def test_constants_match_header():
    src = open(HEADER).read()
    consts = dict(re.findall(r"#define\s+(PGM_[A-Z0-9_]+)\s+(\d+)", src))
    assert int(consts["PGM_KIND_SM1D"]) == _lib.KIND_SM1D
    assert int(consts["PGM_KIND_SM_ARD_PRODSUM"]) == _lib.KIND_SM_ARD_PRODSUM
    assert int(consts["PGM_KIND_SM_ARD_SUMPROD"]) == _lib.KIND_SM_ARD_SUMPROD
    assert int(consts["PGM_CON_SOFTPLUS"]) == _lib.CON_SOFTPLUS
    assert int(consts["PGM_CON_INTERVAL"]) == _lib.CON_INTERVAL
    assert int(consts["PGM_FLAG_GRAD"]) == _lib.FLAG_GRAD
    assert int(consts["PGM_FLAG_LEARN_NOISE"]) == _lib.FLAG_LEARN_NOISE
    assert int(consts["PGM_FLAG_BOUNDS_PER_LC"]) == _lib.FLAG_BOUNDS_PER_LC
    assert int(consts["PGM_OPT_ADAMW"]) == _lib.OPT_ADAMW


def test_bad_arguments_are_rejected_before_any_launch():
    lib = _lib.load()
    one = 8  # any non-null fake pointer: validation fails before it is dereferenced
    rc = lib.pgm_sm_mll_grad_f64(one, None, one, None, one, one, one, one, 1, 64, 1, 9, 0, 0,
                                 one, None, one, one, 1 << 30, None)
    assert rc == -1 and b"Q" in lib.pgm_last_error()
    rc = lib.pgm_sm_mll_grad_f64(one, None, one, None, one, one, one, one, 1, 64, 2, 4, 0, 0,
                                 one, None, one, one, 1 << 30, None)
    assert rc == -1 and b"d == 1" in lib.pgm_last_error()
    rc = lib.pgm_sm_mll_grad_f64(None, None, one, None, one, one, one, one, 1, 64, 1, 4, 0, 0,
                                 one, None, one, one, 1 << 30, None)
    assert rc == -1 and b"null" in lib.pgm_last_error()
    rc = lib.pgm_optim_step_f64(one, one, None, None, None, 1, 4, 1, 0.1, 0.9, 0.999, 1e-8, 0.0,
                                1, None)
    assert rc == -1 and b"exp_avg" in lib.pgm_last_error()
    # B == 0 is a no-op (empty batch)
    assert lib.pgm_sm_mll_grad_f64(None, None, None, None, None, None, None, None, 0, 64, 1, 4,
                                   0, 0, None, None, None, None, 0, None) == 0


def test_model_validation_matches_the_compiled_configurations():
    """A (kind, d, Q) model is accepted exactly when build.CONFIGS has a row of its kind and d with
    QT >= max(Q, 1) (stationary kinds take Q == 0, the others 1 <= Q <= 8); no launch happens here
    (workspace_bytes = 0)."""
    from pgmuvi_b200.build import CONFIGS
    rejections = (b"stationary kinds have no mixtures", b"time kernels 3..5", b"stationary kind / d",
                  b"Q (num_mixtures)", b"d == 1", b"d == 2", b"unknown kernel_kind")
    lib = _lib.load()
    one = 8
    for kind in range(-1, 41):
        for d in range(0, 4):
            for Q in range(-1, 10):
                q_ok = Q == 0 if _lib.is_stat(kind) else 1 <= Q <= 8
                accepted = q_ok and any(c[0] == kind and c[2] == d and c[1] >= max(Q, 1)
                                        for c in CONFIGS)
                rc = lib.pgm_sm_mll_grad_f64(one, None, one, None, one, one, one, one, 1, 64, d, Q,
                                             kind, 0, one, None, one, one, 0, None)
                err = lib.pgm_last_error()
                case = (kind, d, Q, err)
                assert rc == -1, case
                if accepted:
                    assert b"workspace" in err, case
                else:
                    assert any(r in err for r in rejections), case
                assert (lib.pgm_fisher_workspace_bytes(64, 1, d, Q, kind, 0) == 0) != accepted, case


def test_workspace_is_per_block_not_per_lightcurve():
    lib = _lib.load()
    w512 = lib.pgm_workspace_bytes(8, 512, 1, 4, -1)
    w1024 = lib.pgm_workspace_bytes(8, 1024, 1, 4, -1)
    assert 0 < w512 < w1024 < (8 << 30)


def test_f32_staging_size_and_validation():
    lib = _lib.load()
    # mll+grad: x, y, noise [B,n] + raw, grad [B,P] + lb, ub [P] + mll [B], each 256-aligned
    s1 = lib.pgm_f32_staging_bytes(4096, 512, 1, 4, 0, 0, 0, 0)
    assert s1 >= 8 * (3 * 4096 * 512 + 2 * 4096 * 13 + 2 * 13 + 4096)
    assert s1 < 8 * (3 * 4096 * 512 + 2 * 4096 * 13 + 2 * 13 + 4096) + 12 * 256
    # the fit entry adds the loss and raw histories
    s2 = lib.pgm_f32_staging_bytes(4096, 512, 1, 4, 0, 0, 300, 1)
    assert s2 - s1 >= 8 * (300 * 4096 + 301 * 4096 * 13)
    one = 8
    rc = lib.pgm_sm_mll_grad_f32(one, None, one, None, one, one, one, one, 1, 64, 1, 4, 0, 0,
                                 one, None, one, one, 1024, None)
    assert rc == -1 and b"workspace" in lib.pgm_last_error()
    rc = lib.pgm_sm_fit_f32(one, None, one, None, one, one, one, one, 1, 64, 1, 4, 0, 0, 2, 0.1,
                            0.9, 0.999, 1e-8, 0.01, 0, 0, 0.0, 9, one, None, one, one, one,
                            1 << 30, None)
    assert rc == -1 and b"maxiter" in lib.pgm_last_error()


def test_ops_refuse_cpu_tensors():
    import torch
    from pgmuvi_b200 import ops
    x = torch.zeros(1, 8, 1, dtype=torch.float64)
    y = torch.zeros(1, 8, dtype=torch.float64)
    raw = torch.zeros(1, 13, dtype=torch.float64)
    k = torch.ones(13, dtype=torch.int32)
    b = torch.zeros(13, dtype=torch.float64)
    with pytest.raises((RuntimeError, NotImplementedError)):
        ops.sm_mll_grad(x, y, None, raw, k, b, b, None, 0, 4, False, True)
