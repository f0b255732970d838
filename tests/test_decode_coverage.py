"""Decode path coverage: every output of every GEMV plan cell, of the grouped and PDL launch forms, and of the benchmarked
decode step, against an independent float64 reference with a per-output error bound.

ref64() recomputes C = A . B^T from the raw block bytes in numpy (nibbles, q5 high bits, int8 values, fp16 scales read with
.view(np.float16), subnormals included): sumi is an exact float64 batched matmul per block, each block is folded with the
formulas of include/qgemm.h (q4_0: d_w*(d_a*sumi - 8*s_a), q4_1 / q5_1: + m_w*s_a/4 or m_w*s_a under QGEMM_MS_EXACT, ...) and
summed in float64.  It also returns S = sum_b (|d_w*d_a*sumi| + |s_a term|).  Any fp32 evaluation of the same sum -- whatever
its order: lane-sequential, butterfly, split over warps or K segments -- is within (nb + 4) * 2^-24 * S of the exact value, so
that bound is checked for EVERY output.  The max|dC|/max|C| <= 1e-5 gate of the rest of the suite only sees errors as large
as the largest row; rows with small per-row scales (subnormal fp16 d) are invisible to it, and the negative controls below
show it passing results the per-output gate rejects.

GEMV plan cells (gemv_plan, csrc/gemv.cu; grid = min(F, 296) CTAs on a B200, skewed row spans when F >= 8 * grid = 2368).
Passes as (TT tokens, PPL register pairs per lane or 0 = activations in smem, WPR warps per row, RT rows per tile, F = kFull /
r = ragged).  The same for all five formats unless noted:
    T=1  K=1024  (1,1,1,8,r)   K=2048 (1,1,1,8,F)   K=3072 (1,2,1,8,r)   K=4096 (1,2,1,8,F)   K=5120 (1,3,1,8,r)
         K=6144  (1,3,1,8,F)   K=8192 (1,2,2,4,F)   K=11008 (1,3,2,4,r)  K=14336 (1,2,4,2,r)  K=16384 (1,2,4,2,F)
         K=28672 (1,2,8,1,r)
         largest K with a plan (1,3,8,1): q4_0 49152 (F), q4_1 46976, q5_0 44544, q5_1 42496, q8_0 34304 (r);
         the next K with bulk-copyable rows (49408, 47104, 44800, 42560, 34560) has none: forced GEMV -> QGEMM_E_ALIGN
    T=2  K=4096 (2,1,2,8,F) [q8_0 RT 4]   K=11008 (2,1,8,2,r)   K=16384 (2,1,8,2,F) [q8_0 RT 1]
         K=28672 q4_0/q4_1/q5_0 (2,0,8,1,r); q5_1/q8_0 (1,2,8,1,r) x 2
    T=3  K=4096 (3,1,2,8,F) [q8_0 RT 4]   K=11008 (3,1,8,2,r)   K=16384 (3,1,8,2,F) [q8_0 RT 1]
         K=28672 q4_0/q4_1/q5_0 (2,0,8,1,r) + (1,2,8,1,r); q5_1/q8_0 (1,2,8,1,r) x 3
    T=4..8 K=4096 (T,0,1,8)   K=8192 (T,0,2,4|2|1)
    K=14336 T=4 (4,0,4,2|1)   T=5 (5,0,4,1) [q8_0 (4,0,4,1) + (1,2,4,2,r)]   T=6 (5,0,4,1) + (1,2,4,2,r) [q8_0 + (2,1,8,1,r)]
            T=7 (5,0,4,1) + (2,1,8,2,r) [q8_0 + (3,1,8,1,r)]   T=8 (5,0,4,1) + (3,1,8,2,r) [q8_0 (4,0,4,1) x 2]
    T=9  K=4096 (8,0,1,8) + (1,2,1,8,F)   K=14336 (5,0,4,1) + (4,0,4,2|1) [q8_0 (4,0,4,1) x 2 + (1,2,4,2,r)]
    T=13 K=4096 (8,0,1,8) + (5,0,1,8)     K=14336 (5,0,4,1) x 2 + (3,1,8,2,r) [q8_0 (4,0,4,1) x 3 + (1,2,4,2,r)]
Every cell runs at F = 290 (one row per CTA), 1000 and 2371 (skew on; not at the largest K, to keep F * K <= 64M), and
each call's launch count must equal its number of passes in gemv_pass_tokens(); activations are staged by one bulk copy
(act_bulk = 1) when 16-byte aligned, word by word (act_bulk = 0) at byte offsets +4 / +8 / +12.
"""
import functools
import os

import numpy as np
import pytest

import datagen
import qgemm_oracle as qo

TOL_MAXNORM = 1e-5
U32 = 2.0 ** -24
WTS = qo.WEIGHT_TYPES
PATH_AUTO, PATH_GEMV, PATH_MMA = 0x000, 0x200, 0x300
STATIC, READY = 0x10, 0x20
E_ALIGN = -2
G = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_vectors.npz"))


@pytest.fixture(scope="module")
def O():
    return qo.Oracle()


# ------------------------------------------------------------------------------------------
# ref64: independent float64 reference straight from the block bytes
# ------------------------------------------------------------------------------------------
def _f16(b):
    """uint8 [..., 2] (little-endian fp16 bits) -> float64 [...]"""
    return np.ascontiguousarray(b).view(np.float16)[..., 0].astype(np.float64)


def _unpack_weights(wt, w):
    """uint8 [F, nb, bs] -> q float64 [nb, F, 32] (un-offset integers: 0..15, 0..31 or int8), d [nb, F], m [nb, F] | None"""
    w = np.ascontiguousarray(w.transpose(1, 0, 2))
    d = _f16(w[..., 0:2])
    m = _f16(w[..., 2:4]) if wt in (qo.Q4_1, qo.Q5_1) else None
    if wt == qo.Q8_0:
        return w[..., 2:34].view(np.int8).astype(np.float64), d, m
    off = {qo.Q4_0: 2, qo.Q4_1: 4, qo.Q5_0: 6, qo.Q5_1: 8}[wt]
    qs = w[..., off:off + 16]
    q = np.concatenate([qs & 0x0F, qs >> 4], axis=-1)          # element i: low nibble of byte i, i + 16: high nibble
    if wt in (qo.Q5_0, qo.Q5_1):
        qh = np.ascontiguousarray(w[..., off - 4:off]).view("<u4")  # [nb, F, 1], bit i = 5th bit of element i
        q = q | (((qh >> np.arange(32, dtype=np.uint32)) & 1) << 4).astype(np.uint8)
    return q.astype(np.float64), d, m


def ref64(wt, act, weight, flags=0, chunk_elems=1 << 22):
    """act uint8 [T, nb, 36], weight uint8 [F, nb, bs] -> (C64 [F, T], S [F, T]) in float64."""
    T, nb, _ = act.shape
    F = weight.shape[0]
    assert weight.shape[1] == nb and weight.shape[2] == qo.BLOCK_BYTES[wt]
    a = np.ascontiguousarray(act.transpose(1, 0, 2))             # [nb, T, 36]
    d_a, s_a = _f16(a[..., 0:2])[:, None, :], _f16(a[..., 2:4])[:, None, :]
    q_a = a[..., 4:36].view(np.int8).astype(np.float64).transpose(0, 2, 1)   # [nb, 32, T]
    C64, S = np.empty((F, T)), np.empty((F, T))
    rows = max(1, chunk_elems // (nb * 32))
    for f0 in range(0, F, rows):
        q_w, d_w, m_w = _unpack_weights(wt, weight[f0:f0 + rows])
        d_w = d_w[:, :, None]
        # |q_w| <= 255 (127 signed), |q_a| <= 128, 32 products: every partial sum is an integer far below 2^53 -> exact
        sumi = np.matmul(q_w, q_a)                                   # [nb, rows, T]
        t1 = d_w * d_a * sumi                                        # products of fp16 values and sumi: exact in float64
        if wt in (qo.Q4_0, qo.Q5_0):
            t2 = -(8.0 if wt == qo.Q4_0 else 16.0) * d_w * s_a
        elif wt in (qo.Q4_1, qo.Q5_1):
            t2 = m_w[:, :, None] * s_a * (1.0 if flags & qo.GEMM_MS_EXACT else 0.25)
        else:
            t2 = np.zeros_like(t1)
        C64[f0:f0 + rows] = (t1 + t2).sum(axis=0)
        S[f0:f0 + rows] = (np.abs(t1) + np.abs(t2)).sum(axis=0)
    return C64, S


def _ratios(c, C64, S, nb):
    """|c - C64| / ((nb + 4) 2^-24 S) per output; an output with S = 0 must be exactly zero (ratio 0, else inf)."""
    err = np.abs(np.asarray(c, np.float64) - C64)
    lim = (nb + 4) * U32 * S
    return np.where(lim > 0, err / np.where(lim > 0, lim, 1.0), np.where(err > 0, np.inf, 0.0))


def bound_ratio(c, C64, S, nb):
    """max over outputs of the ratio above; > 1 fails"""
    r = _ratios(c, C64, S, nb)
    return float(r.max()) if r.size else 0.0


def check_ref64(c, ref, nb, what, oracle=None):
    """c [F, T] (fp32) against ref = (C64, S): the per-output bound, the 1e-5 max-norm gate against C64 and, if
    given, against the oracle's fp32 result."""
    C64, S = ref
    c = np.asarray(c)
    assert c.shape == C64.shape, what
    assert np.isfinite(c).all(), f"{what}: non-finite outputs"
    r = _ratios(c, C64, S, nb)
    if r.size and r.max() > 1.0:
        i = np.unravel_index(np.argmax(r), c.shape)
        raise AssertionError(f"{what}: {int((r > 1).sum())} outputs over the bound; worst (f={i[0]}, t={i[1]}) = {c[i]!r}, "
                             f"exact {C64[i]!r}, S {S[i]:.3e}, {r[i]:.2f}x the bound")
    e = qo.max_norm_err(c, C64)
    assert e <= TOL_MAXNORM, f"{what}: max-norm {e:.3e} vs ref64"
    if oracle is not None:
        e = qo.max_norm_err(c, oracle)
        assert e <= TOL_MAXNORM, f"{what}: max-norm {e:.3e} vs oracle"


# ------------------------------------------------------------------------------------------
# data
# ------------------------------------------------------------------------------------------
def scaled_rows(T, F, K, seed=0):
    """Model-like operands whose rows span decades, like real weights: per-row scale 10^U(-4, 0), ~1.5 % of the rows at
    1e-5 (fp16 d subnormal or zero), ~1 % all-zero rows, per-token activation scales 10^U(-1, 1), and one all-zero
    activation block.  Returns fp32 x [T, K], w [F, K]."""
    rng = np.random.default_rng(seed)
    w = rng.standard_normal((F, K), dtype=np.float32)
    w *= np.float32(0.02)
    w.reshape(-1)[::128] *= 8.0
    scale = 10.0 ** rng.uniform(-4, 0, F)
    scale[rng.choice(F, max(1, F // 64), replace=False)] = 1e-5
    scale[rng.choice(F, max(1, F // 100), replace=False)] = 0.0
    w *= scale.astype(np.float32)[:, None]
    x = rng.standard_normal((T, K), dtype=np.float32) * (10.0 ** rng.uniform(-1, 1, (T, 1))).astype(np.float32)
    x[0, 32 * rng.integers(K // 32):][:32] = 0.0
    return x, w


@functools.lru_cache(maxsize=3)
def _weights_f32(F, K):
    return scaled_rows(1, F, K, seed=F * 7 + K)[1]


@functools.lru_cache(maxsize=2)
def _acts_f32(T, K):
    return scaled_rows(T, 1, K, seed=K + 1)[0]


# ------------------------------------------------------------------------------------------
# CPU self-tests of the reference and of the gate
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("wt", WTS)
@pytest.mark.parametrize("K", [4096, 11008])
def test_ref64_vs_oracle_within_bound(O, wt, K):
    T, F = 3, 96
    cases = []
    x, w = datagen.model_like(T, F, K, seed=K + wt)
    cases.append(("model-like", O.quantize_q8_1(x), O.quantize_weight(wt, w)))
    x, w = scaled_rows(T, F, K, seed=K + wt)
    cases.append(("scaled rows", O.quantize_q8_1(x), O.quantize_weight(wt, w)))
    cases.append(("fuzz", datagen.fuzz_act_blocks(T, K // 32, seed=wt, const_ds=False),
                  datagen.fuzz_weight_blocks(wt, F, K // 32, seed=wt)))
    cases.append(("extreme", *datagen.extreme_blocks(wt)))
    for name, aq, wq in cases:
        for fl in ((0, qo.GEMM_MS_EXACT) if wt in (qo.Q4_1, qo.Q5_1) else (0,)):
            ref = ref64(wt, aq, wq, fl)
            check_ref64(O.gemm(wt, aq, wq, layout="FT", flags=fl), ref, aq.shape[1], f"oracle {name} flags {fl}")
            check_ref64(O.gemm(wt, aq, wq, layout="FT", flags=fl | qo.GEMM_FMA), ref, aq.shape[1], f"oracle FMA order {name}")


def test_ref64_exact_on_extreme_blocks(O):
    """|sumi| at its bound: the float64 sum is exact there, so ref64 equals the integer arithmetic."""
    for wt in WTS:
        a, w = datagen.extreme_blocks(wt)
        C64, _ = ref64(wt, a, w)
        sumi = O.gemm_sumi(wt, a, w).astype(np.float64)     # [T, F, nb]
        d_w = _f16(w[..., 0:2])                               # [F, nb]
        d_a, s_a = _f16(a[..., 0:2]), _f16(a[..., 2:4])       # [T, nb]
        t1 = d_w[None] * d_a[:, None] * sumi
        if wt in (qo.Q4_0, qo.Q5_0):
            t2 = -(8.0 if wt == qo.Q4_0 else 16.0) * d_w[None] * s_a[:, None]
        elif wt in (qo.Q4_1, qo.Q5_1):
            t2 = 0.25 * _f16(w[..., 2:4])[None] * s_a[:, None]
        else:
            t2 = 0.0
        assert (C64 == (t1 + t2).sum(-1).T).all()


@pytest.mark.parametrize("wt", WTS)
def test_ref64_vs_golden_vectors(wt):
    n = qo.TYPE_NAMES[wt]
    for a, w, c in ((f"fuzz_a_{n}", f"fuzz_w_{n}", f"fuzz_c_{n}_FT"),
                    ("g1_a_q8_1_ref", f"g1_w_{n}_fw", f"g1_c_{n}_FT"), ("g3_a_q8_1_ref", f"g3_w_{n}_fw", f"g3_c_{n}_FT")):
        ref = ref64(wt, G[a], G[w])
        check_ref64(G[c], ref, G[a].shape[1], f"golden {c}")


def test_scaled_rows_reach_small_and_zero_rows(O):
    T, F, K = 4, 1000, 4096
    x, w = scaled_rows(T, F, K, seed=5)
    wq = O.quantize_weight(qo.Q4_0, w)
    d = _f16(wq[..., 0:2])
    assert ((d > 0) & (d < 2.0 ** -14)).mean() > 0.3           # subnormal fp16 scales
    assert (np.abs(w).max(axis=1) == 0).sum() >= 10            # all-zero rows
    assert ((np.abs(w).max(axis=1) > 0) & (np.abs(w).max(axis=1) < 1e-5)).any()
    assert (np.abs(x.reshape(T, -1, 32)).max(axis=2) == 0).sum() == 1   # one all-zero activation block
    sc = np.abs(x).max(axis=1)
    assert sc.max() / sc.min() > 2                             # per-token scales differ


@pytest.mark.parametrize("wt", WTS)
def test_negative_controls_per_output_gate_sees_small_rows(O, wt):
    """One dropped block and one flipped weight nibble in a row whose |C| is <= 1e-4 of max|C|: the max-norm gate passes
    both results, the per-output gate rejects both."""
    T, F, K = 2, 512, 4096
    nb = K // 32
    x, w = scaled_rows(T, F, K, seed=11 + wt)
    aq, wq = O.quantize_q8_1(x), O.quantize_weight(wt, w)
    ref = ref64(wt, aq, wq)
    C64 = ref[0]
    check_ref64(O.gemm(wt, aq, wq, layout="FT"), ref, nb, "unmutated")
    rowmax = np.abs(C64).max(axis=1)
    d = _f16(wq[..., 0:2])
    cand = np.nonzero((rowmax > 0) & (rowmax <= 1e-4 * rowmax.max()) & (d > 0).any(axis=1))[0]
    assert cand.size, "no small row with nonzero fp16 d in the data"
    f = int(cand[np.argmin(rowmax[cand])])
    b = int(np.argmax(np.abs(d[f])))                          # the row's largest block
    dropped = wq.copy()
    dropped[f, b, :] = 0                                      # d = m = 0 and all quants 0: the block contributes nothing
    flipped = wq.copy()
    qa = aq[..., 4:].view(np.int8)[0, b].astype(np.int32)
    j = int(np.argmax(np.abs(qa[:16])))                       # a low-nibble element of a large activation
    qs_off = {qo.Q4_0: 2, qo.Q4_1: 4, qo.Q5_0: 6, qo.Q5_1: 8, qo.Q8_0: 2}[wt]
    flipped[f, b, qs_off + j] ^= 0x08 if wt != qo.Q8_0 else 0x80
    for name, bad in (("dropped block", dropped), ("flipped nibble", flipped)):
        c = O.gemm(wt, aq, bad, layout="FT")
        assert qo.max_norm_err(c, C64) <= TOL_MAXNORM, name    # the max-norm gate cannot see it ...
        assert bound_ratio(c, *ref, nb) > 1.0, name            # ... the per-output gate does
        with pytest.raises(AssertionError):
            check_ref64(c, ref, nb, name)


def test_ref64_chunking_is_invisible(O):
    x, w = scaled_rows(2, 300, 2048, seed=3)
    aq, wq = O.quantize_q8_1(x), O.quantize_weight(qo.Q5_1, w)
    a, b = ref64(qo.Q5_1, aq, wq), ref64(qo.Q5_1, aq, wq, chunk_elems=64 * 1024 * 7)
    assert (a[0] == b[0]).all() and (a[1] == b[1]).all()


# ------------------------------------------------------------------------------------------
# GPU helpers (raw C ABI, device memory from torch)
# ------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def L():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from quant_gemm import _lib
    return _lib.lib()   # raises if the CUDA library is missing: no silent fallback


def _torch():
    import torch
    return torch


def _stream():
    return _torch().cuda.current_stream().cuda_stream


def _dev(a):
    return _torch().from_numpy(np.ascontiguousarray(a)).cuda()


def _host(t):
    _torch().cuda.synchronize()
    return t.cpu().numpy()


def _bits(t):
    return t.view(_torch().int32)


SENTINEL = -7.25   # written into the padding of strided outputs: must survive untouched


class DevWeights:
    """A weight matrix at the start of a device buffer with slack behind it (hints may run past the matrix but stay
    inside the allocation), plus a copy at a 2-byte offset."""

    def __init__(self, wq, slack=1 << 20):
        torch = _torch()
        self.nbytes, self.slack = wq.size, slack
        self.buf = torch.zeros(self.nbytes + slack, dtype=torch.uint8, device="cuda")
        self.buf[:self.nbytes] = _dev(wq.reshape(-1))
        self.ptr = self.buf.data_ptr()
        assert self.ptr % 256 == 0

    def misaligned(self):
        torch = _torch()
        b = torch.zeros(self.nbytes + 16, dtype=torch.uint8, device="cuda")
        b[2:2 + self.nbytes] = self.buf[:self.nbytes]
        return b, b.data_ptr() + 2


def _gemm(L, wt, a_ptr, w_ptr, c_ptr, T, F, K, ldc_t, ldc_f, flags, hint=None):
    if hint is None:
        return L.qgemm_gemm(wt, a_ptr, w_ptr, c_ptr, T, F, K, ldc_t, ldc_f, flags, None, 0, _stream())
    return L.qgemm_gemm_hinted(wt, a_ptr, w_ptr, c_ptr, T, F, K, ldc_t, ldc_f, flags, None, 0, _stream(), hint[0], hint[1])


def _run_ft(L, wt, a_ptr, w_ptr, T, F, K, flags, hint=None):
    """C [F, T] (ggml layout) from one call; a launch that the stream may overlap with earlier work (INPUTS_READY)
    starts after a device synchronize, so nothing in flight touches its buffers."""
    torch = _torch()
    c = torch.empty((F, T), dtype=torch.float32, device="cuda")
    if flags & READY:
        torch.cuda.synchronize()
    rc = _gemm(L, wt, a_ptr, w_ptr, c.data_ptr(), T, F, K, 1, T, flags, hint)
    assert rc == 0, f"qgemm_gemm rc {rc} flags {flags:#x}"
    return c


# ------------------------------------------------------------------------------------------
# 3. the GEMV plan matrix (forced PATH_GEMV, all five formats)
# ------------------------------------------------------------------------------------------
CELLS = {1024: [1], 2048: [1], 3072: [1], 4096: [1, 2, 3, 4, 5, 6, 7, 8, 9, 13], 5120: [1], 6144: [1],
         8192: [1, 4, 5, 6, 7, 8], 11008: [1, 2, 3], 14336: [1, 4, 5, 6, 7, 8, 9, 13], 16384: [1, 2, 3], 28672: [1, 2, 3]}
ROWS = (290, 1000, 2371)     # one row per CTA / ~3.4 rows per CTA / skewed spans
TMAX = 13


def gemv_pass_tokens(wt, T, K):
    """Tokens per launch of a forced-GEMV call, restating gemv_plan (csrc/gemv.cu) for the table above: for each pass the
    largest TT <= 8 whose activations (registers when TT * PPL <= 3 with the fewest warps per row, else shared memory) and
    two weight stages of RT rows fit the 110 KB shared-memory budget."""
    nb = K // 32
    np_, rowbytes = nb // 2, nb * qo.BLOCK_BYTES[wt]

    def tt_of(T):
        for tt in range(min(T, 8), 0, -1):
            ppl, wpr = 0, 1
            for w in (1, 2, 4, 8):
                need = -(-np_ // (32 * w))
                if need * tt <= 3:
                    ppl, wpr = need, w
                    break
            if ppl == 0:
                while wpr < 8 and np_ > 64 * wpr:
                    wpr *= 2
            rt = 8 // wpr
            while rt < 8 and 2 * rt * rowbytes <= 24 * 1024:
                rt *= 2
            fixed = 768 + tt * nb * (40 if ppl == 0 else 36) + 128
            stage = lambda r: -(-r * rowbytes // 128) * 128    # noqa: E731
            while rt > 1 and fixed + 2 * stage(rt) > 110 * 1024:
                rt //= 2
            if fixed + 2 * stage(rt) <= 110 * 1024:
                return tt
        return 0

    first, out, t0 = tt_of(T), [], 0
    while first and t0 < T:
        out.append(first if T - t0 >= first else tt_of(T - t0))
        t0 += first
    return out


def test_gemv_pass_table():
    """Spot checks of gemv_pass_tokens() against the table in the module docstring."""
    assert gemv_pass_tokens(qo.Q4_0, 8, 14336) == [5, 3]
    assert gemv_pass_tokens(qo.Q8_0, 8, 14336) == [4, 4]
    assert gemv_pass_tokens(qo.Q8_0, 13, 14336) == [4, 4, 4, 1]
    assert gemv_pass_tokens(qo.Q5_1, 3, 28672) == [1, 1, 1]
    assert gemv_pass_tokens(qo.Q4_0, 3, 28672) == [2, 1]
    assert gemv_pass_tokens(qo.Q4_0, 13, 4096) == [8, 5]
    for wt, (kmax, kover) in K_LIMIT.items():
        assert gemv_pass_tokens(wt, 1, kmax) == [1] and gemv_pass_tokens(wt, 1, kover) == []


def _gemv_variants(L, wt, aq, dw, T, F, K, ref, what, oracle):
    """The plain forced-GEMV call against ref64 and the oracle, then every launch form against it bit for bit."""
    torch = _torch()
    nb = K // 32
    flags = PATH_GEMV
    da = _dev(aq)
    L.qgemm_reset_launch_count()
    c0 = _run_ft(L, wt, da.data_ptr(), dw.ptr, T, F, K, flags)
    assert L.qgemm_last_path() == PATH_GEMV
    assert L.qgemm_launch_count() == len(gemv_pass_tokens(wt, T, K)), f"{what}: passes differ from the plan table"
    check_ref64(_host(c0), ref, nb, what, oracle)
    forms = {
        "WEIGHTS_STATIC": dict(flags=flags | STATIC),
        "WEIGHTS_STATIC|INPUTS_READY": dict(flags=flags | STATIC | READY),
        "hint aligned": dict(flags=flags | STATIC, hint=(dw.ptr, dw.nbytes)),
        "hint misaligned": dict(flags=flags | STATIC, hint=(dw.ptr + 8, dw.nbytes - 8)),
        "hint past the matrix": dict(flags=flags | STATIC, hint=(dw.ptr + max(0, dw.nbytes - 4096) // 16 * 16, dw.slack)),
    }
    for name, kw in forms.items():
        c = _run_ft(L, wt, da.data_ptr(), dw.ptr, T, F, K, **kw)
        assert torch.equal(_bits(c), _bits(c0)), f"{what}: {name} differs from the plain call"
    # include layout, padded rows: C[t * (F + 3) + f]
    out = torch.full((T, F + 3), float(SENTINEL), device="cuda")
    assert _gemm(L, wt, da.data_ptr(), dw.ptr, out.data_ptr(), T, F, K, F + 3, 1, flags) == 0
    assert torch.equal(_bits(out[:, :F].t()), _bits(c0)), f"{what}: ldc_t = F + 3"
    assert (out[:, F:] == SENTINEL).all(), f"{what}: padding overwritten (ldc_t)"
    # ggml layout, padded: C[f * (T + 3) + t]
    out = torch.full((F, T + 3), float(SENTINEL), device="cuda")
    assert _gemm(L, wt, da.data_ptr(), dw.ptr, out.data_ptr(), T, F, K, 1, T + 3, flags) == 0
    assert torch.equal(_bits(out[:, :T]), _bits(c0)), f"{what}: ldc_f = T + 3"
    assert (out[:, T:] == SENTINEL).all(), f"{what}: padding overwritten (ldc_f)"
    # activations 4-byte aligned only: word-by-word staging instead of the bulk copy
    raw = torch.zeros(aq.size + 16, dtype=torch.uint8, device="cuda")
    for off in (4, 8, 12):
        raw[off:off + aq.size] = da.reshape(-1)
        c = _run_ft(L, wt, raw.data_ptr() + off, dw.ptr, T, F, K, flags)
        assert torch.equal(_bits(c), _bits(c0)), f"{what}: activations at +{off}"
    return c0


@pytest.mark.gpu
@pytest.mark.parametrize("wt", WTS)
@pytest.mark.parametrize("K", sorted(CELLS))
def test_gemv_plan_matrix(L, O, K, wt):
    """Every (T, K) cell of the table above at three row counts; ref64 and the oracle are computed once per (F, K) for
    TMAX tokens and sliced (outputs of different tokens are independent)."""
    x = _acts_f32(TMAX, K)
    aq = O.quantize_q8_1(x)
    for F in ROWS:
        wq = O.quantize_weight(wt, _weights_f32(F, K))
        C64, S = ref64(wt, aq, wq)
        oracle = O.gemm(wt, aq, wq, layout="FT")
        dw = DevWeights(wq)
        for T in CELLS[K]:
            _gemv_variants(L, wt, aq[:T], dw, T, F, K, (C64[:, :T], S[:, :T]),
                           f"{qo.TYPE_NAMES[wt]} T={T} F={F} K={K}", oracle[:, :T])
        del dw


K_LIMIT = {qo.Q4_0: (49152, 49408), qo.Q4_1: (46976, 47104), qo.Q5_0: (44544, 44800), qo.Q5_1: (42496, 42560),
           qo.Q8_0: (34304, 34560)}


@pytest.mark.gpu
@pytest.mark.parametrize("wt", WTS)
def test_gemv_longest_rows_and_beyond(L, O, wt):
    """T=1 at the largest K the format's plan accepts (one row per tile, 8 warps per row, 3 pairs per lane) and at the next
    bulk-copyable K, where forced GEMV returns QGEMM_E_ALIGN and AUTO still computes the right product."""
    torch = _torch()
    kmax, kover = K_LIMIT[wt]
    x = _acts_f32(1, kmax)
    aq = O.quantize_q8_1(x)
    for F in ROWS[:2]:    # F * K <= 64M keeps the CPU reference short; skewed spans of long rows: K = 28672 above
        wq = O.quantize_weight(wt, _weights_f32(F, kmax))
        dw = DevWeights(wq)
        _gemv_variants(L, wt, aq, dw, 1, F, kmax, ref64(wt, aq, wq), f"{qo.TYPE_NAMES[wt]} F={F} K={kmax}",
                       O.gemm(wt, aq, wq, layout="FT"))
        del dw
    F = 1000
    x = scaled_rows(1, 1, kover, seed=kover)[0]
    aq = O.quantize_q8_1(x)
    wq = O.quantize_weight(wt, scaled_rows(1, F, kover, seed=kover + 1)[1])
    da, dw = _dev(aq), DevWeights(wq)
    c = torch.empty((F, 1), device="cuda")
    assert _gemm(L, wt, da.data_ptr(), dw.ptr, c.data_ptr(), 1, F, kover, 1, 1, PATH_GEMV) == E_ALIGN
    c = _run_ft(L, wt, da.data_ptr(), dw.ptr, 1, F, kover, PATH_AUTO)
    assert L.qgemm_last_path() != PATH_GEMV
    check_ref64(_host(c), ref64(wt, aq, wq), kover // 32, f"AUTO above the GEMV limit K={kover}", O.gemm(wt, aq, wq, layout="FT"))


@pytest.mark.gpu
@pytest.mark.parametrize("wt", [qo.Q4_0, qo.Q8_0])
def test_gemv_lm_head(L, O, wt):
    """The Llama-3 LM head, F = 128256 rows at K = 4096, one token: 433 rows per CTA on skewed spans."""
    F, K = 128256, 4096
    aq = O.quantize_q8_1(_acts_f32(TMAX, K))[:1]
    step = 16384
    wq = np.concatenate([O.quantize_weight(wt, scaled_rows(1, min(step, F - f0), K, seed=900 + f0)[1])
                         for f0 in range(0, F, step)])
    dw = DevWeights(wq)
    _gemv_variants(L, wt, aq, dw, 1, F, K, ref64(wt, aq, wq), f"LM head {qo.TYPE_NAMES[wt]}", O.gemm(wt, aq, wq, layout="FT"))


@pytest.mark.gpu
@pytest.mark.parametrize("wt", WTS)
def test_gemv_weights_2byte_aligned(L, O, wt):
    """Weights at a 2-byte offset (the ABI minimum) cannot be bulk-copied: forced GEMV says QGEMM_E_ALIGN, AUTO computes
    the product on another path."""
    torch = _torch()
    F, K = 1000, 4096
    x = _acts_f32(TMAX, K)
    aq = O.quantize_q8_1(x)
    wq = O.quantize_weight(wt, _weights_f32(F, K))
    C64, S = ref64(wt, aq, wq)
    dw = DevWeights(wq)
    buf, ptr = dw.misaligned()
    for T in (1, 4):
        da = _dev(aq[:T])
        c = torch.empty((F, T), device="cuda")
        assert _gemm(L, wt, da.data_ptr(), ptr, c.data_ptr(), T, F, K, 1, T, PATH_GEMV) == E_ALIGN
        c = _run_ft(L, wt, da.data_ptr(), ptr, T, F, K, PATH_AUTO)
        check_ref64(_host(c), (C64[:, :T], S[:, :T]), K // 32, f"AUTO, weights at +2, T={T}")


# ------------------------------------------------------------------------------------------
# 4. groups, the benchmarked launch sequence, real dependencies
# ------------------------------------------------------------------------------------------
def _group(L, wt, a_ptr, w_ptrs, c_ptrs, Fs, T, K, ldc_t, ldc_f, flags, hint=None):
    import ctypes as C
    n = len(w_ptrs)
    wp, cp, fs = (C.c_void_p * n)(*w_ptrs), (C.c_void_p * n)(*c_ptrs), (C.c_int * n)(*Fs)
    if hint is None:
        return L.qgemm_gemm_group(wt, a_ptr, n, wp, cp, fs, T, K, ldc_t, ldc_f, flags, _stream())
    return L.qgemm_gemm_group_hinted(wt, a_ptr, n, wp, cp, fs, T, K, ldc_t, ldc_f, flags, _stream(), hint[0], hint[1])


@pytest.mark.gpu
@pytest.mark.parametrize("wt", WTS)
@pytest.mark.parametrize("Fs", [(4096, 4096, 4096), (11008, 11008), (4099, 37, 2500)], ids=["qkv", "gate_up", "ragged"])
def test_group_vs_separate_gemv(L, O, wt, Fs):
    """One grouped launch (matrix boundaries inside a CTA's span, skewed spans) for T = 1..8: every output against ref64
    and bit for bit against separate forced-GEMV calls."""
    torch = _torch()
    K = 4096
    aq8 = O.quantize_q8_1(_acts_f32(TMAX, K))[:8]
    wqs = [O.quantize_weight(wt, scaled_rows(1, F, K, seed=F + 31 * m)[1]) for m, F in enumerate(Fs)]
    refs = [ref64(wt, aq8, w) for w in wqs]
    dws = [DevWeights(w, slack=0) for w in wqs]
    for T in range(1, 9):
        da = _dev(aq8[:T])
        for flags in (PATH_GEMV, STATIC):
            outs = [torch.empty((F, T), device="cuda") for F in Fs]
            assert _group(L, wt, da.data_ptr(), [d.ptr for d in dws], [o.data_ptr() for o in outs], Fs, T, K, 1, T, flags) == 0
            assert L.qgemm_last_path() == PATH_GEMV
            for m, F in enumerate(Fs):
                sep = _run_ft(L, wt, da.data_ptr(), dws[m].ptr, T, F, K, PATH_GEMV)
                assert torch.equal(_bits(outs[m]), _bits(sep)), f"group {Fs} T={T} matrix {m} flags {flags:#x}"
                if flags == PATH_GEMV:
                    check_ref64(_host(outs[m]), (refs[m][0][:, :T], refs[m][1][:, :T]), K // 32,
                                f"group {Fs} {qo.TYPE_NAMES[wt]} T={T} matrix {m}")


LLAMA7B = [("wq", 4096, 4096), ("wk", 4096, 4096), ("wv", 4096, 4096), ("wo", 4096, 4096),
           ("w_gate", 11008, 4096), ("w_up", 11008, 4096), ("w_down", 4096, 11008)]
HINT_WINDOW = 12 << 20


@pytest.mark.gpu
def test_benchmarked_decode_step_in_a_graph(L, O):
    """The single-GPU decode step of the benchmark, rebuilt for two layers (Q4_0): 14 matrices back to back in one arena
    (256-byte padding), both activation vectors quantized by one launch at the front, then the grouped form (q/k/v and
    gate/up in one launch each, WEIGHTS_STATIC) and the separate form (WEIGHTS_STATIC, plus INPUTS_READY on k, v and up),
    each launch hinting a 12 MB window from the next launch's weights, clamped to the arena's end -- all captured in one
    CUDA graph.  Replayed with two activation vectors into outputs filled with NaN: every output of every matrix against
    ref64 after each replay, and the two forms bit for bit equal."""
    torch = _torch()
    import quant_gemm
    wt, layers = qo.Q4_0, 2
    mats = [(F, K) for _ in range(layers) for _, F, K in LLAMA7B]
    sizes = [F * (K // 32) * 18 for F, K in mats]
    arena = torch.empty(sum((n + 255) // 256 * 256 for n in sizes), dtype=torch.uint8, device="cuda")
    arena_end = arena.data_ptr() + arena.numel()
    wq_host, wdev, off = [], [], 0
    for i, (F, K) in enumerate(mats):
        wq = datagen.fuzz_weight_blocks(wt, F, K // 32, seed=100 + i)
        wq[..., 0:2] = ((np.random.default_rng(i).random((F, K // 32)) * 0.02 + 0.001)
                        .astype(np.float16).view(np.uint8).reshape(F, K // 32, 2))
        arena[off:off + sizes[i]] = _dev(wq.reshape(-1))
        wq_host.append(wq)
        wdev.append(arena[off:off + sizes[i]])
        off += (sizes[i] + 255) // 256 * 256
    KS = (4096, 11008)
    x_host = torch.empty((1, sum(KS)), dtype=torch.float32).pin_memory()
    x_dev = torch.empty((1, sum(KS)), device="cuda")
    aq_all = torch.empty((1, sum(KS) // 32, 36), dtype=torch.uint8, device="cuda")
    aq = {4096: aq_all[:, :128], 11008: aq_all[:, 128:]}
    out_g = torch.empty(sum(F for F, _ in mats), device="cuda")
    out_s = torch.empty_like(out_g)
    starts = [int(v) for v in np.cumsum([0] + [F for F, _ in mats])]
    view = lambda buf, i: buf[starts[i]:starts[i + 1]]        # noqa: E731

    def hint(i):
        p = wdev[i].data_ptr()
        return (p, min(HINT_WINDOW, arena_end - p))

    groups = []
    for l in range(layers):
        b = 7 * l
        groups += [[b, b + 1, b + 2], [b + 3], [b + 4, b + 5], [b + 6]]

    def step():
        x_dev.copy_(x_host, non_blocking=True)
        quant_gemm.quantize_q8_1(x_dev, out=aq_all)
        for gi, g in enumerate(groups):
            K = mats[g[0]][1]
            nxt = groups[(gi + 1) % len(groups)][0]
            a = aq[K].data_ptr()
            if len(g) == 1:
                rc = _gemm(L, wt, a, wdev[g[0]].data_ptr(), view(out_g, g[0]).data_ptr(), 1, mats[g[0]][0], K, 1, 1,
                           STATIC, hint(nxt))
            else:
                rc = _group(L, wt, a, [wdev[i].data_ptr() for i in g], [view(out_g, i).data_ptr() for i in g],
                            [mats[i][0] for i in g], 1, K, 1, 1, STATIC, hint(nxt))
            assert rc == 0
        for i, (F, K) in enumerate(mats):
            rc = _gemm(L, wt, aq[K].data_ptr(), wdev[i].data_ptr(), view(out_s, i).data_ptr(), 1, F, K, 1, 1,
                       STATIC | READY if i % 7 in (1, 2, 5) else STATIC, hint((i + 1) % len(mats)))
            assert rc == 0

    torch.cuda.synchronize()                                   # the arena was filled on the default stream
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        x_host.copy_(torch.randn((1, sum(KS)), generator=torch.Generator().manual_seed(1)))
        step()                                                 # warm: kernel attributes are set outside the capture
        stream.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            step()
    for seed in (7, 8):
        x = torch.randn((1, sum(KS)), generator=torch.Generator().manual_seed(seed))
        torch.cuda.synchronize()
        x_host.copy_(x)
        with torch.cuda.stream(stream):
            out_g.fill_(float("nan"))
            out_s.fill_(float("nan"))
            graph.replay()
        stream.synchronize()
        assert torch.equal(_bits(out_g), _bits(out_s)), "grouped and separate forms differ"
        aqh = _host(aq_all)
        xn = x.numpy()
        assert (aqh[0, :128] == O.quantize_q8_1(xn[:, :4096])[0]).all()
        assert (aqh[0, 128:] == O.quantize_q8_1(xn[:, 4096:])[0]).all()
        og = _host(out_g)
        for i, (F, K) in enumerate(mats):
            a = aqh[:, :128] if K == 4096 else aqh[:, 128:]
            check_ref64(og[starts[i]:starts[i + 1], None], ref64(wt, a, wq_host[i]), K // 32,
                        f"replay seed {seed} matrix {i} ({LLAMA7B[i % 7][0]} layer {i // 7})")


@functools.lru_cache(maxsize=1)
def _layer_weights(wt, layers):
    O = qo.Oracle()
    ws = []
    for l in range(layers):
        for j, (_, F, K) in enumerate(LLAMA7B):
            _, w = scaled_rows(1, F, K, seed=300 + 7 * l + j)
            ws.append(O.quantize_weight(wt, w))
    return ws


@pytest.mark.gpu
@pytest.mark.parametrize("grouped", [True, False], ids=["grouped", "separate"])
def test_dependent_layers_pdl_bit_identical(L, O, grouped):
    """Two Llama layers in which every input is the requantized output of the projection before it:
    x -> [q, k, v];  quantize(v) -> o;  quantize(o) -> [gate, up];  quantize(silu(gate) * up) -> down;  quantize(down) ->
    the next layer.  Every GEMV with WEIGHTS_STATIC (programmatic dependent launch), INPUTS_READY where a launch shares its
    input with the one before it (k, v, up in the separate form); eagerly and from a CUDA graph.  Bit-identical to the same
    sequence with flags 0, and every stage against ref64 on the GPU's own quantized input."""
    torch = _torch()
    import quant_gemm
    wt, layers, T = qo.Q4_0, 2, 1
    wq = _layer_weights(wt, layers)
    wd = [_dev(w) for w in wq]
    x0 = _dev(scaled_rows(T, 1, 4096, seed=77)[0])

    def run(dep):
        """dep: use the PDL flags.  Returns (outputs, quantized inputs) per stage, in fresh buffers."""
        outs, acts = [], []
        st, rd = (STATIC, STATIC | READY) if dep else (0, 0)

        def gemv(a, idx, flags):
            F, K = LLAMA7B[idx % 7][1:]
            c = torch.empty((F, T), device="cuda")
            assert _gemm(L, wt, a.data_ptr(), wd[idx].data_ptr(), c.data_ptr(), T, F, K, 1, T, flags) == 0
            return c

        def group(a, idxs, flags):
            cs = [torch.empty((LLAMA7B[i % 7][1], T), device="cuda") for i in idxs]
            assert _group(L, wt, a.data_ptr(), [wd[i].data_ptr() for i in idxs], [c.data_ptr() for c in cs],
                          [LLAMA7B[i % 7][1] for i in idxs], T, LLAMA7B[idxs[0] % 7][2], 1, T, flags) == 0
            return cs

        x = x0
        for l in range(layers):
            b = 7 * l
            a = quant_gemm.quantize_q8_1(x.reshape(T, -1))
            qkv = group(a, [b, b + 1, b + 2], st) if grouped else [gemv(a, b, st), gemv(a, b + 1, rd), gemv(a, b + 2, rd)]
            acts += [a] * 3
            a = quant_gemm.quantize_q8_1(qkv[2].t().contiguous())
            o = gemv(a, b + 3, st)
            acts.append(a)
            a = quant_gemm.quantize_q8_1(o.t().contiguous())
            gu = group(a, [b + 4, b + 5], st) if grouped else [gemv(a, b + 4, st), gemv(a, b + 5, rd)]
            acts += [a] * 2
            a = quant_gemm.quantize_q8_1_silu_mul(gu[0].t().contiguous(), gu[1].t().contiguous())
            down = gemv(a, b + 6, st)
            acts.append(a)
            outs += qkv + [o] + gu + [down]
            x = down.t().contiguous()
        return outs, acts

    torch.cuda.synchronize()
    plain, plain_acts = run(False)
    eager, _ = run(True)
    torch.cuda.synchronize()
    for i, (p, e) in enumerate(zip(plain, eager)):
        assert torch.equal(_bits(p), _bits(e)), f"eager PDL sequence differs at stage {i}"
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            g_outs, _ = run(True)
        for c in g_outs:
            c.fill_(float("nan"))
        graph.replay()
    stream.synchronize()
    for i, (p, g) in enumerate(zip(plain, g_outs)):
        assert torch.equal(_bits(p), _bits(g)), f"graph replay differs at stage {i}"
    for i, (c, a) in enumerate(zip(plain, plain_acts)):
        ah = _host(a)
        check_ref64(_host(c), ref64(wt, ah, wq[i]), ah.shape[1], f"stage {i} ({LLAMA7B[i % 7][0]} layer {i // 7})")


@pytest.mark.gpu
def test_back_to_back_static_gemvs_same_output(L, O):
    """Write after write: two WEIGHTS_STATIC GEMVs into the same C (the second may start under the first): the second's
    result must be what remains."""
    torch = _torch()
    wt, F, K = qo.Q4_0, 4096, 4096
    aq = O.quantize_q8_1(_acts_f32(TMAX, K))[:1]
    w1 = O.quantize_weight(wt, _weights_f32(F, K))
    w2 = O.quantize_weight(wt, scaled_rows(1, F, K, seed=4242)[1])
    da, d1, d2 = _dev(aq), _dev(w1), _dev(w2)
    want = _run_ft(L, wt, da.data_ptr(), d2.data_ptr(), 1, F, K, PATH_GEMV)
    c = torch.full((F, 1), float("nan"), device="cuda")
    assert _gemm(L, wt, da.data_ptr(), d1.data_ptr(), c.data_ptr(), 1, F, K, 1, 1, STATIC) == 0
    assert _gemm(L, wt, da.data_ptr(), d2.data_ptr(), c.data_ptr(), 1, F, K, 1, 1, STATIC) == 0
    torch.cuda.synchronize()
    assert torch.equal(_bits(c), _bits(want))
    check_ref64(_host(c), ref64(wt, aq, w2), K // 32, "second of two back-to-back GEMVs")


# ------------------------------------------------------------------------------------------
# 5. skinny path (PATH_MMA): the regs, bigk and wide kernels
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("wt", WTS)
@pytest.mark.parametrize("T,F,K", [(3, 4096, 4096),      # regs kernel
                                   (8, 11008, 4096),     # regs; q8_0: wide (F * K >= 2^25)
                                   (5, 4096, 11008),     # bigk (rows too long for register fragments)
                                   (8, 4096, 14336),     # bigk
                                   (16, 11008, 4096),    # wide (T > 8), 16-token pass
                                   (24, 4096, 8192)])    # wide for q4_0 (16 + 8 tokens); the other formats' tiles do not
                                                         # fit it at this K: passes of 8 on the regs kernel
def test_mma_paths_scaled_rows(L, O, wt, T, F, K):
    torch = _torch()
    x, w = scaled_rows(T, F, K, seed=T + F + K + wt)
    aq, wq = O.quantize_q8_1(x), O.quantize_weight(wt, w)
    da, dw = _dev(aq), _dev(wq)
    L.qgemm_reset_launch_count()
    c0 = _run_ft(L, wt, da.data_ptr(), dw.data_ptr(), T, F, K, PATH_MMA)
    assert L.qgemm_last_path() == PATH_MMA
    # the wide kernel takes 32 (K = 4096) or 16 (K = 8192) tokens per launch, the regs and bigk kernels 8
    wide = K == 4096 and (T > 8 or (wt == qo.Q8_0 and F * K >= 1 << 25)) or (K == 8192 and T > 8 and wt == qo.Q4_0)
    per = (32 if K == 4096 else 16) if wide else 8
    assert L.qgemm_launch_count() == -(-T // per), "the shape did not reach the kernel it is listed for"
    check_ref64(_host(c0), ref64(wt, aq, wq), K // 32, f"mma {qo.TYPE_NAMES[wt]} {T}x{F}x{K}", O.gemm(wt, aq, wq, layout="FT"))
    for fl in (STATIC, STATIC | READY):
        c = _run_ft(L, wt, da.data_ptr(), dw.data_ptr(), T, F, K, PATH_MMA | fl)
        assert torch.equal(_bits(c), _bits(c0)), f"flags {fl:#x}"
