"""CPU: the C-ABI library loads and exports every symbol include/asyncrl_b200.h declares; the
host-only entry points work; the product fails loudly without a GPU (no CPU fallback)."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "asyncrl_b200.h")).read()
    return sorted(set(re.findall(r"ARL_API[^;(]*?\b(arl_\w+)\s*\(", src)))


def test_header_declares_the_expected_surface():
    syms = header_symbols()
    assert len(syms) == 59, syms
    for must in ("arl_preprocess_push", "arl_forward", "arl_backward", "arl_sample_actions",
                 "arl_returns_lossgrad", "arl_clip_rmsprop", "arl_param_layout", "arl_last_error",
                 "arl_comm_init", "arl_allreduce_grads"):      # SURVEY §8b minimum export set
        assert must in syms
    assert "arl_forward_egreedy" in syms and "arl_nstep_q_lossgrad" in syms    # n-step Q: one header


def test_library_exports_every_declared_symbol(pkg):
    lib = pkg._cabi.load()
    for s in header_symbols():
        assert getattr(lib, s) is not None, s
    assert set(header_symbols()) == set(pkg._cabi.EXPORTS)      # ctypes table == header


def test_param_layout_is_the_reference_order(pkg):
    off = pkg._cabi.param_layout(6)
    assert off == [0, 4096, 4112, 12304, 12336, 675888, 676144, 677680, 677686, 677942, 677943]
    assert pkg._cabi.param_layout(18)[-1] == 681027
    lib = pkg._cabi.load()
    buf = (ctypes.c_int64 * 11)()
    assert lib.arl_param_layout(0, buf) == -1                  # ARL_ERR_INVALID, message set
    assert b"action_size" in lib.arl_last_error()
    assert lib.arl_param_layout(6, None) == -1


def test_a2_block_rows_is_a_pure_host_function(pkg):
    """Rows of one a2 block = envs one forward launch handles (api.cu): the whole batch up to 16 384
    envs, above that the largest divisor <= 16 384 that is a multiple of 128 (>= 2048), else one
    launch again -- the value arl_fc_backward needs to walk a2."""
    f = pkg._cabi.a2_block_rows
    assert [f(n) for n in (1, 4096, 16384)] == [1, 4096, 16384]
    assert f(32768) == 16384 and f(65536) == 16384 and f(18432) == 9216 and f(20480) == 10240
    assert f(16385) == 16385 and f(3 * 16384 + 1) == 3 * 16384 + 1      # no divisor: one launch
    for n in (24576, 40960, 49152, 61440):
        c = f(n)
        assert n % c == 0 and 2048 <= c <= 16384 and c % 128 == 0


def test_no_cpu_fallback(pkg):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(pkg._cabi.ArlError):
        pkg._cabi.init("cuda:0")
    with pytest.raises(pkg._cabi.ArlError):
        pkg.History(pkg.config.M1, num_envs=2)
    with pytest.raises(pkg._cabi.ArlError):
        pkg._cabi.ptr(torch.zeros(4))                          # CPU tensors are refused


def test_product_never_imports_the_oracle():
    pkg_dir = os.path.join(ROOT, "async-rl-tensorflow_b200")
    for base, _, files in os.walk(pkg_dir):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".sh")):
                txt = open(os.path.join(base, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, re.M), f
                assert "/root/reference" not in txt, f


def test_ctypes_prototypes_match_the_header(pkg):
    """Every prototype in _cabi.SIGNATURES has the argument count and the pointer / integer /
    float kinds of its declaration in include/asyncrl_b200.h (a drifted ctypes table corrupts
    the call frame silently)."""
    src = open(os.path.join(ROOT, "include", "asyncrl_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    decls = dict((m.group(1), m.group(2)) for m in
                 re.finditer(r"ARL_API\s+int\s+(arl_\w+)\s*\(([^;]*?)\)\s*;", src, re.S))
    kind = {ctypes.c_void_p: "ptr", ctypes.c_int: "int", ctypes.c_int64: "i64",
            ctypes.c_uint64: "u64", ctypes.c_float: "f32", ctypes.c_double: "f64"}

    def ckind(param):
        p = " ".join(param.split())
        if "*" in p:
            return "ptr"
        if p.startswith("float"):
            return "f32"
        if p.startswith("double"):
            return "f64"
        if p.startswith("int64_t"):
            return "i64"
        if p.startswith("uint64_t"):
            return "u64"
        assert p.startswith("int "), p
        return "int"

    for name, argtypes in pkg._cabi.SIGNATURES.items():
        params = [p for p in decls[name].split(",") if p.strip() and p.strip() != "void"]
        got = ["ptr" if isinstance(a, type) and issubclass(a, ctypes._Pointer) else kind[a]
               for a in argtypes]
        assert got == [ckind(p) for p in params], (name, got, params)
