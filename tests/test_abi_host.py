"""CPU suite: the C-ABI library loads, exports every symbol include/qgemm.h declares, and its
host-only logic (argument validation, sharding arithmetic, error strings) behaves.  No kernel
is launched here."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "llama.cpp-quant-gemm_b200", "lib", "libqgemm_sm100.so")


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(LIB):
        import __graft_entry__
        __graft_entry__.build()
    from quant_gemm import _lib
    return _lib.lib()


def test_header_symbols_are_exported(lib):
    hdr = open(os.path.join(ROOT, "include", "qgemm.h")).read()
    declared = set(re.findall(r"QGEMM_API[^;(]*?\b(qgemm_\w+)\s*\(", hdr))
    assert len(declared) >= 14
    from quant_gemm import _lib
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    for name in declared:
        assert hasattr(lib, name), name


def test_peers_struct_layout_matches_header(tmp_path):
    """The ctypes mirror of struct qgemm_peers has the size and field offsets a C compiler gives the header."""
    import subprocess
    from quant_gemm import _lib
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "qgemm.h"\n'
                   'int main(void){printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(qgemm_peers), offsetof(qgemm_peers, C),'
                   ' offsetof(qgemm_peers, flag), offsetof(qgemm_peers, done), offsetof(qgemm_peers, wait_index),'
                   ' offsetof(qgemm_peers, C_multicast)); return 0;}\n')
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    P = _lib.QgemmPeers
    assert got == [C.sizeof(P), P.C.offset, P.flag.offset, P.done.offset, P.wait_index.offset, P.C_multicast.offset]


def test_version_and_strings(lib):
    assert lib.qgemm_version() == 100
    for code in range(-5, 1):
        assert len(lib.qgemm_strerror(code)) > 1
    assert [lib.qgemm_block_bytes(t) for t in (2, 3, 6, 7, 8, 9)] == [18, 20, 22, 24, 34, 36]
    assert lib.qgemm_block_bytes(5) == 0


def test_argument_validation_without_gpu(lib):
    # validation happens before any CUDA call, so these hold with or without a device
    BAD, ALIGN = -1, -2
    p = C.c_void_p(0x1000)
    assert lib.qgemm_gemm(2, p, p, p, 1, 1, 31, 1, 1, 0, None, 0, None) == BAD       # K % 32
    assert lib.qgemm_gemm(4, p, p, p, 1, 1, 32, 1, 1, 0, None, 0, None) == BAD       # unknown type
    assert lib.qgemm_gemm(2, None, p, p, 1, 1, 32, 1, 1, 0, None, 0, None) == BAD    # null
    assert lib.qgemm_gemm(2, p, p, p, -1, 1, 32, 1, 1, 0, None, 0, None) == BAD
    assert lib.qgemm_gemm(2, C.c_void_p(0x1002), p, p, 1, 1, 32, 1, 1, 0, None, 0, None) == ALIGN
    assert lib.qgemm_gemm(2, p, C.c_void_p(0x1001), p, 1, 1, 32, 1, 1, 0, None, 0, None) == ALIGN
    assert lib.qgemm_gemm(2, p, p, p, 0, 5, 32, 1, 1, 0, None, 0, None) == 0          # empty T: no-op
    assert lib.qgemm_quantize_q8_1(p, p, 0, 64, 0, None) == 0
    assert lib.qgemm_quantize_q8_1(p, p, 1, 33, 0, None) == BAD
    assert lib.qgemm_quantize_weight(9, p, p, 1, 32, 0, None) == BAD
    assert lib.qgemm_dequantize(2, p, C.c_void_p(0x1004), 1, 32, None) == ALIGN


def test_chain_step_struct_layout_matches_header(tmp_path):
    """ctypes mirror of struct qgemm_chain_step == the header's layout."""
    import subprocess
    from quant_gemm import _lib
    src = tmp_path / "layout_chain.c"
    fields = ["act_q8_1", "act_f32", "gate_f32", "nmat", "weights", "C", "F", "K", "ldc_f", "flags"]
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "qgemm.h"\nint main(void){printf("%zu", sizeof(qgemm_chain_step));'
                   + "".join(f'printf(" %zu", offsetof(qgemm_chain_step, {f}));' for f in fields) + 'printf("\\n"); return 0;}\n')
    exe = tmp_path / "layout_chain"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    S = _lib.QgemmChainStep
    assert got == [C.sizeof(S)] + [getattr(S, f).offset for f in fields]


def test_chain_argument_validation_without_gpu(lib):
    from quant_gemm import _lib
    BAD, ALIGN, WS = -1, -2, -5
    S = _lib.QgemmChainStep
    arr = (S * 2)()
    for d in arr:
        d.act_q8_1, d.nmat, d.K, d.ldc_f = 0x1000, 1, 4096, 1
        d.weights[0], d.C[0], d.F[0] = 0x2000, 0x3000, 512
    sync = C.c_void_p(0x4000)
    need = lib.qgemm_gemv_chain_sync_bytes(2)     # counters + the scratch of the in-kernel quantizer
    assert need >= 20 and lib.qgemm_gemv_chain_sync_bytes(0) == 0
    assert lib.qgemm_gemv_chain_max_steps() >= 128
    assert lib.qgemm_gemv_chain(2, arr, 0, 0, sync, need, None) == BAD
    assert lib.qgemm_gemv_chain(4, arr, 2, 0, sync, need, None) == BAD        # unknown type
    assert lib.qgemm_gemv_chain(2, arr, 2, 0, None, 0, None) == WS
    assert lib.qgemm_gemv_chain(2, arr, 2, 0, sync, need - 1, None) == WS
    arr[1].nmat = 4
    assert lib.qgemm_gemv_chain(2, arr, 2, 0, sync, need, None) == BAD
    arr[1].nmat = 1
    arr[1].act_f32 = 0x5000                                                     # both kinds of activations
    assert lib.qgemm_gemv_chain(2, arr, 2, 0, sync, need, None) == BAD
    arr[1].act_f32 = None
    arr[1].K = 100
    assert lib.qgemm_gemv_chain(2, arr, 2, 0, sync, need, None) == BAD
    arr[1].K = 4096
    arr[1].weights[0] = 0x2001
    assert lib.qgemm_gemv_chain(2, arr, 2, 0, sync, need, None) == ALIGN
    arr[1].weights[0] = 0x2000
    arr[1].flags = 0x8
    assert lib.qgemm_gemv_chain(2, arr, 2, 0, sync, need, None) == BAD          # only QGEMM_INPUTS_READY is a step flag
    arr[1].flags = 0x20
    import torch
    if not torch.cuda.is_available():
        assert lib.qgemm_gemv_chain(2, arr, 2, 0, sync, need, None) in (-3, -4)   # no device: fails loudly, computes nothing


def test_new_entries_validate_before_any_cuda_call(lib):
    """fp16-activation entries and the explicit-hint forms: argument errors are reported with or without a device."""
    BAD, ALIGN = -1, -2
    p = C.c_void_p(0x1000)
    odd = C.c_void_p(0x1001)
    assert lib.qgemm_quantize_q8_1_f16(p, p, 1, 33, 0, None) == BAD            # K % 32
    assert lib.qgemm_quantize_q8_1_f16(None, p, 1, 32, 0, None) == BAD
    assert lib.qgemm_quantize_q8_1_f16(odd, p, 1, 32, 0, None) == ALIGN        # halves: 2-byte alignment
    assert lib.qgemm_quantize_q8_1_f16(C.c_void_p(0x1002), p, 0, 32, 0, None) == 0   # empty: no-op
    assert lib.qgemm_gemm_f16act(2, p, p, p, 1, 1, 31, 1, 1, 0, None, 0, None) == BAD
    assert lib.qgemm_gemm_f16act(4, p, p, p, 1, 1, 32, 1, 1, 0, None, 0, None) == BAD
    assert lib.qgemm_gemm_f16act(2, odd, p, p, 1, 1, 32, 1, 1, 0, None, 0, None) == ALIGN
    assert lib.qgemm_gemm_f16act(2, C.c_void_p(0x1002), p, p, 0, 5, 32, 1, 1, 0, None, 0, None) == 0   # 2-byte aligned halves are fine
    assert lib.qgemm_gemm_hinted(2, p, p, p, 1, 1, 31, 1, 1, 0, None, 0, None, p, 64) == BAD
    assert lib.qgemm_gemm_hinted(2, p, p, p, 0, 5, 32, 1, 1, 0, None, 0, None, p, 64) == 0
    wp, cp, fs = (C.c_void_p * 1)(0x2000), (C.c_void_p * 1)(0x3000), (C.c_int * 1)(8)
    assert lib.qgemm_gemm_group_hinted(2, p, 0, wp, cp, fs, 1, 32, 1, 1, 0, None, p, 64) == BAD   # nmat = 0
    assert lib.qgemm_gemm_group_hinted(2, p, 1, wp, cp, fs, 1, 31, 1, 1, 0, None, p, 64) == BAD


def check_no_cpu_fallback(lib):
    p = C.c_void_p(0x1000)
    assert lib.qgemm_gemm(2, p, p, p, 1, 1, 32, 1, 1, 0, None, 0, None) in (-3, -4)
    assert lib.qgemm_quantize_q8_1(p, p, 1, 32, 0, None) in (-3, -4)


def test_no_cpu_fallback(lib):
    """Without a B200 the compute entries must fail loudly, never compute on the host.  Where a GPU is present, the
    check runs in a child process that is shown no device."""
    import subprocess
    import sys
    import torch
    if not torch.cuda.is_available():
        check_no_cpu_fallback(lib)
        return
    path = os.pathsep.join([os.path.join(ROOT, "tests"), os.path.join(ROOT, "llama.cpp-quant-gemm_b200")])
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", PYTHONPATH=path + os.pathsep + os.environ.get("PYTHONPATH", ""))
    code = "import test_abi_host as t; from quant_gemm import _lib; t.check_no_cpu_fallback(_lib.lib())"
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]


def test_shard_range(lib):
    from quant_gemm import _lib
    for F, world, align in [(28672, 8, 256), (28672, 4, 256), (4096, 2, 128), (1000, 3, 64), (7, 4, 1), (5, 8, 4)]:
        ranges = [_lib.shard_range(F, world, r, align) for r in range(world)]
        assert ranges[0][0] == 0 and ranges[-1][1] == F
        for (a0, a1), (b0, b1) in zip(ranges, ranges[1:]):
            assert a1 == b0 and a0 <= a1
        for a0, a1 in ranges[:-1]:
            assert (a0 % align == 0 or a0 == F) and (a1 % align == 0 or a1 == F)
        sizes = [b - a for a, b in ranges]
        assert max(sizes) - min(sizes) < 2 * align  # last unit may be partial
    assert _lib.shard_range(28672, 8, 3, 256) == (3 * 3584, 4 * 3584)
    with pytest.raises(RuntimeError):
        _lib.shard_range(10, 2, 2, 1)


def test_python_surface_matches_reference_names():
    import quant_gemm
    # python/quant_gemm/__init__.py:92-101 __all__ of the reference
    for name in ["quantize_q4_0", "quantize_q8_1", "gemm_q4_0_q8_1", "dequantize_q4_0", "QK4_0", "QK8_1",
                 "BLOCK_Q4_0_BYTES", "BLOCK_Q8_1_BYTES"]:
        assert name in quant_gemm.__all__ and hasattr(quant_gemm, name)
    assert (quant_gemm.QK4_0, quant_gemm.QK8_1, quant_gemm.BLOCK_Q4_0_BYTES, quant_gemm.BLOCK_Q8_1_BYTES) == (32, 32, 18, 36)


def test_python_checks_raise_like_torch_check():
    import torch
    import quant_gemm
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        quant_gemm.quantize_q8_1(torch.zeros(2, 32))
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        quant_gemm.gemm_q4_0_q8_1(torch.zeros(18, dtype=torch.uint8), torch.zeros(36, dtype=torch.uint8), 1, 1, 32)
