"""CPU: the C-ABI library loads and exports every symbol include/yagre_b200.h declares.
No compute call is made (there is no GPU here)."""
import ctypes as C
import os
import re

import pytest

from yagre_mcmc_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "yagre_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(yg_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    names = header_symbols()
    assert len(names) >= 17
    for n in names:
        assert hasattr(lib, n), f"{n} declared in yagre_b200.h but not exported"
    assert set(names) == set(_lib.SYMBOLS), set(names) ^ set(_lib.SYMBOLS)


def test_abi_version_and_struct_sizes():
    lib = _lib.load()
    assert lib.yg_abi_version() == _lib.YG_ABI_VERSION
    assert lib.yg_pooled_len(2) == 3 + 2 + 4 + 4 + 2
    # POD layouts the binding mirrors (sizes from the C compiler's rules)
    assert C.sizeof(_lib.YgLevel) == 8 * 2 + 8 + 8 + 8 * 7 + 8 * 3 + 8 + 8          # ABI 4: + tempering
    assert C.sizeof(_lib.YgProblem) == 8 + _lib.YG_MAX_LEVELS * C.sizeof(_lib.YgLevel) + 8 + 8 + 8
    assert C.sizeof(_lib.YgConfig) % 8 == 0


def test_create_rejects_bad_config_without_touching_the_gpu():
    lib = _lib.load()
    cfg = _lib.YgConfig()
    cfg.abi_version = 999
    h = C.c_void_p()
    assert lib.yg_create(C.byref(cfg), C.byref(h)) == _lib.YG_ERR_ABI
    cfg.abi_version = _lib.YG_ABI_VERSION
    cfg.n_chains, cfg.dim, cfg.n_levels = 4, 99, 1
    assert lib.yg_create(C.byref(cfg), C.byref(h)) == _lib.YG_ERR_UNSUPPORTED      # beyond every kernel's size
    cfg.dim = 0
    assert lib.yg_create(C.byref(cfg), C.byref(h)) == _lib.YG_ERR_INVALID
    assert b"dim" in lib.yg_last_error()
    cfg.dim, cfg.n_levels = 2, 4            # three surrogates crash in the reference itself (mlda.py:23-33)
    with pytest.raises(NotImplementedError):
        _lib.check(lib.yg_create(C.byref(cfg), C.byref(h)))
    cfg.n_levels, cfg.model, cfg.sub_chain_length = 3, _lib.MODEL_LV, 2      # two surrogates: not on the LV kernel
    with pytest.raises(NotImplementedError):
        _lib.check(lib.yg_create(C.byref(cfg), C.byref(h)))
    cfg.n_levels, cfg.model, cfg.dim, cfg.adaptive = 1, _lib.MODEL_GAUSS, 1, 1
    with pytest.raises(NotImplementedError, match="scalar chains"):        # chain/adaptive.py:41-43
        _lib.check(lib.yg_create(C.byref(cfg), C.byref(h)))


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from yagre_mcmc_b200.ensemble import ChainEnsemble, LoweredProblem
    import numpy as np
    pb = LoweredProblem(dict(model='gauss', dim=1, levels=1, J=1), dict(
        prop_L=[[1.0]], L0_g_mean=[0.0], L0_g_prec=[[1.0]], L0_g_logconst=0.0))
    with pytest.raises(_lib.BackendUnavailable):
        ChainEnsemble(pb, 4)


def test_state_layout_names_every_yg_state_field():
    from yagre_mcmc_b200.ensemble import state_layout
    lay = state_layout(6, 3, 2, True, 4)
    assert [k + "_dev" for k in lay] == [f for f, _ in _lib.YgState._fields_]


def test_check_state_accepts_exactly_the_layout():
    """What load_state checks before a pointer reaches yg_load_state, which copies the layout's byte count from each."""
    import torch
    from yagre_mcmc_b200.ensemble import check_state, state_layout
    n, d = 6, 3
    for lay in (state_layout(n, d, 2, True, 4), state_layout(n, 12, 1, False, 0)):
        good = {k: torch.zeros(shape, dtype=dtype) for k, (shape, dtype) in lay.items()}
        check_state(good, lay)
        check_state(dict(theta=good["theta"], logpost=good["logpost"], step_index=3), lay)
        for k in ("theta", "logpost"):
            with pytest.raises(ValueError):
                check_state({j: v for j, v in good.items() if j != k}, lay)
        for k, v in good.items():
            bad = [torch.zeros((v.shape[0] + 1,) + tuple(v.shape[1:]), dtype=v.dtype),      # oversized
                   v.to(torch.float32), v.to(torch.float64 if v.dtype == torch.int64 else torch.int64), v.numpy()]
            if v.dim() > 1:
                bad.append(v.transpose(0, -1))
            for b in bad:
                with pytest.raises(ValueError, match=k):
                    check_state(dict(good, **{k: b}), lay)
