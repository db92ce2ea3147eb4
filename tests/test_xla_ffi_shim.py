"""bpl_next_b200/csrc/xla_ffi_shim.cc (the jax.ffi handlers a bpl-next maintainer registers, INTEGRATION.md B) compiled
against a stand-in for XLA's FFI C++ API (tests/xla_ffi_mock/ -- the real headers ship with jaxlib, which is not installable
here) and its three implementations called the way XLA's executor would: typed buffers with [batch..., D] dimensions,
result buffers, the stream.  The numbers must be those of the C ABI called directly."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from tests import helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIBDIR = os.path.join(ROOT, "bpl_next_b200", "lib")


def _cuda_include():
    """include/ of the CUDA toolkit whose nvcc builds the library (NVCC, else nvcc on PATH)."""
    nvcc = shutil.which(os.environ.get("NVCC", "nvcc"))
    assert nvcc, "nvcc not found"
    return os.path.join(os.path.dirname(os.path.dirname(os.path.realpath(nvcc))), "include")


def _build(tmp_path):
    so = str(tmp_path / "libmockxla.so")
    cmd = ["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-Wall", "-Wno-comment", "-Werror",
           "-I", os.path.join(ROOT, "tests", "xla_ffi_mock"), "-I", os.path.join(ROOT, "include"), "-I", _cuda_include(),
           os.path.join(ROOT, "tests", "xla_ffi_mock", "drive.cc"), "-L", LIBDIR, "-lbplx", f"-Wl,-rpath,{LIBDIR}", "-o", so]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return so


def test_shim_compiles_against_the_stand_in_api(tmp_path):
    so = _build(tmp_path)
    lib = C.CDLL(so)
    assert lib.mock_xla_call_density and lib.mock_xla_call_grid


@pytest.mark.gpu
def test_handlers_give_the_c_abi_numbers(tmp_path):
    import torch
    from bpl_next_b200 import Problem, score_grid
    from oracle import datasets

    lib = C.CDLL(_build(tmp_path))
    vp, i64 = C.c_void_p, C.c_int64
    lib.mock_xla_call_density.argtypes = [C.c_int, i64, vp, i64, i64, i64, vp, vp, vp, vp, i64, vp, C.c_char_p, C.c_int]
    arr = H.small_problem("neutral_wc", seed=4, multi_conf=True, T=13, M=400)
    p = Problem(arr)
    st = torch.cuda.current_stream().cuda_stream
    err = C.create_string_buffer(256)
    for lik, D in ((0, p.D), (1, sum(c for _, c, _ in p.loglik_layout.values()))):
        x = torch.rand((3, 5, D), device="cuda") - 0.5  # two leading batch axes, like a vmapped call
        if lik:
            x[..., -1] = torch.rand((3, 5), device="cuda") * 0.9 + 0.05
        lp = torch.empty((3, 5), device="cuda"); g = torch.empty_like(x); cc = torch.empty((3, 5), device="cuda")
        ws = p.workspace(15)
        rc = lib.mock_xla_call_density(lik, p._h.value, x.data_ptr(), 3, 5, D, lp.data_ptr(), g.data_ptr(), cc.data_ptr(),
                                       ws.data_ptr(), ws.numel(), st, err, 256)
        assert rc == 0, err.value
        want = (p.loglik if lik else p.logdensity)(x.reshape(15, D).contiguous())
        torch.cuda.synchronize()
        assert torch.equal(lp.reshape(15), want[0]) and torch.equal(g.reshape(15, D), want[1]) and torch.equal(cc.reshape(15), want[2])
    # a wrong trailing axis is refused with a message, not executed
    x = torch.zeros((1, 2, p.D + 1), device="cuda")
    rc = lib.mock_xla_call_density(0, p._h.value, x.data_ptr(), 1, 2, p.D + 1, lp.data_ptr(), g.data_ptr(), cc.data_ptr(),
                                   ws.data_ptr(), ws.numel(), st, err, 256)
    assert rc == -1 and b"parameter count" in err.value
    # grid
    s, fx = datasets.config_5(S=96, F=40)
    ds = {k: torch.from_numpy(v).cuda() for k, v in s.items()}
    dfx = {k: torch.from_numpy(v).cuda() for k, v in fx.items()}
    grid_w, out_w = score_grid("neutral_wc", ds, dfx, 10)
    S, T = s["attack"].shape
    Cf, F = s["confederation_strength"].shape[1], len(fx["home_team"])
    grid = torch.empty((F, 11, 11), device="cuda"); out = torch.empty((F, 3), device="cuda")
    ws2 = torch.empty(64 << 20, dtype=torch.uint8, device="cuda")
    lib.mock_xla_call_grid.argtypes = [i64, i64, C.c_float, i64, i64, i64, i64] + [vp] * 13 + [i64, vp, vp, vp, i64, vp, C.c_char_p, C.c_int]
    rc = lib.mock_xla_call_grid(3, 10, 1.0 / S, S, T, Cf, F, ds["attack"].data_ptr(), ds["defence"].data_ptr(),
                                ds["home_attack"].data_ptr(), ds["away_attack"].data_ptr(), ds["home_defence"].data_ptr(),
                                ds["away_defence"].data_ptr(), ds["confederation_strength"].data_ptr(), ds["corr_coef"].data_ptr(),
                                dfx["home_team"].data_ptr(), dfx["away_team"].data_ptr(), dfx["home_conf"].data_ptr(),
                                dfx["away_conf"].data_ptr(), dfx["neutral_venue"].data_ptr(), T, grid.data_ptr(), out.data_ptr(),
                                ws2.data_ptr(), ws2.numel(), st, err, 256)
    assert rc == 0, err.value
    torch.cuda.synchronize()
    assert torch.equal(grid, grid_w) and torch.equal(out, out_w)
