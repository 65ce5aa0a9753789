"""The tcgen05 GEMM (csrc/gemm.cuh) and its five epilogues element by element against plain fp64 torch.

Every linear layer of the model runs through this GEMM, yet the engine tests see it only through the logits.  Here both
kernels (gemm_tc_kernel<128> and the CTA-pair gemm_tc_pair_kernel) run stand-alone through
tests/kernels/gemm_harness.cu (the engine's own tensor maps and launches) in both engine modes (bf16, and the fp32 mode's
SPLIT variant with three k segments and (hi, lo) outputs), and every output element is checked:

* lattice inputs (integers, and multiples of 1/256 for low parts and residuals) on which every partial sum is exact in
  fp32, so the output must equal the fp64 result bit for bit whatever the summation order: addressing, tiling, the
  pipeline and every epilogue's arithmetic;
* random trained-like inputs at the engine's shapes: every element within a bound derived from the arithmetic (not
  fitted), the GELU over its whole range, and the residual variants the engine uses, including the fp32 mode's K-chunked
  MLP-down;
* isolation: every output is pre-filled with NaN and nothing outside the written region may change; a document's
  Q/K/V^T does not depend on its slot or its neighbours, and no output depends on the grid size.

bf16 has 8 significand bits, so round-to-nearest errs by at most 2^-8 relative, and a (hi, lo) pair by 2^-16; fp32
round-to-nearest by 2^-24; the tensor core's fp32 accumulation, which truncates, is charged 2^-23 per added term.
"""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest
import torch

import __graft_entry__ as ge

pytestmark = pytest.mark.gpu

HARNESS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "kernels", "gemm_harness.cu")
EPI_BIAS, EPI_GELU, EPI_RESID, EPI_QKV, EPI_PATCH = range(5)         # GemmEpilogue (gemm.cuh)
EPI_NAME = {EPI_BIAS: "BIAS", EPI_GELU: "GELU", EPI_RESID: "RESID", EPI_QKV: "QKV", EPI_PATCH: "PATCH"}
STAGES = {128: 6, 256: 5}                      # GemmSmem<128>::STAGES, GemmPairSmemT::STAGES
U_BF16, U_PAIR, U_ACC, U_FP32 = 2.0 ** -8, 2.0 ** -16, 2.0 ** -23, 2.0 ** -24
GELU_FIT = 4.2e-7                              # |error| of the fitted 0.5 erfc(z) on z in [0, 4.3] (gemm.cuh)
GELU_CLAMP = 4.3
HALF_ERFC_CLAMP = 0.5 * math.erfc(GELU_CLAMP)   # ~6.0e-10: what the clamp leaves beyond z = 4.3
LATTICE_STEP = 1.0 / 256.0
N_PATCH = 196                                  # 224 x 224 pages in 16 x 16 patches
# document lengths: the attention tests' LENS (198 = CLS + 197 visual rows, tile edges, 709 = a full document, 1024)
LENS = [198, 199, 255, 256, 257, 320, 336, 337, 383, 384, 385, 641, 656, 657, 709, 1024]
DEV = torch.device("cuda")


@pytest.fixture(scope="module")
def gemm(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("gemm_harness") / "libgemm_harness.so")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    subprocess.check_call([nvcc] + ge.NVCC_FLAGS + ["-I", ge.CSRC, "--shared", HARNESS, "-o", out])
    lib = C.CDLL(out)
    p, i, q = C.c_void_p, C.c_int, C.c_longlong
    lib.gemm_run.argtypes = ([i] * 4 + [p, p, q, q, p, p, q, p, i, i, i, p, p, p, i] + [p] * 8 +
                             [i, p, p, i, p, p, i, i, p, i, i])
    lib.gemm_run.restype = i
    for rule in (lib.gemm_bn, lib.gemm_bn_qkv, lib.gemm_k_chunk):
        rule.argtypes, rule.restype = [i], i
    global _lib
    _lib = lib
    return lib


_lib = None   # the harness the gemm fixture loaded: its exports are the engine's shape rules (gemm.cuh)


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def pick_bn(n):
    """gemm_block_n: BLOCK_N of a GEMM family with N = n columns."""
    return _lib.gemm_bn(n)


def bn_qkv(H):
    """gemm_block_n_qkv: the QKV GEMM's BLOCK_N."""
    return _lib.gemm_bn_qkv(H)


def kchunk(I):
    """gemm_kchunk: K chunk of the fp32-mode MLP-down."""
    return _lib.gemm_k_chunk(I)


def split_bf16(x):
    hi = x.to(torch.bfloat16)
    return hi, (x - hi.float()).to(torch.bfloat16)


def nan_like(shape, dtype):
    return torch.full(shape, float("nan"), dtype=dtype, device=DEV)


# ------------------------------------------------------------------------------------------------ one GEMM problem
class Gemm:
    """Inputs of one GEMM launch in the engine's layouts, its launch, and its outputs mapped back to a dense [M, N].

    a / a_lo: bf16 [a_rows, K] (rows >= M hold NaN or are absent); w / w_lo: bf16 [N, K]; bias fp32 [N].  Epilogue
    extras (all optional, set by the caller before run()):
      RESID: resid / resid_lo (bf16 [rows, N]), resid_f32 (fp32 [rows, N]), or resid_y (fp32 [y_rows, N]) with
             resid_stats (fp32 [M, 2]), resid_src (int32 [M] or None), resid_w / resid_b (fp32 [N]).
      QKV:   lens (rows per slot, sum = M), kv_pitch; heads = N / 192.
      PATCH: pos (fp32 [n_patch + 1, N]), n_patch."""

    def __init__(self, epi, bn, split, M, N, K, a, w, bias, a_lo=None, w_lo=None):
        self.epi, self.bn, self.split, self.M, self.N, self.K = epi, bn, bool(split), M, N, K
        self.a, self.a_lo, self.w, self.w_lo, self.bias = a, a_lo, w, w_lo, bias
        self.resid = self.resid_lo = self.resid_f32 = self.resid_y = None
        self.resid_stats = self.resid_src = self.resid_w = self.resid_b = None
        self.resid_prefetch = 0
        self.lens, self.kv_pitch, self.pos, self.n_patch = None, 0, None, N_PATCH
        self.m_dev = True

    def name(self):
        return f"{EPI_NAME[self.epi]} bn {self.bn} {'split' if self.split else 'bf16'} M {self.M} N {self.N} K {self.K}"

    # -------------------------------------------------------------- launch
    def alloc_outputs(self):
        M, N, odt = self.M, self.N, torch.bfloat16
        rows = (max(M, 1) + 255) // 256 * 256 + 128          # a stray write past M lands in the buffer
        if self.epi in (EPI_RESID, EPI_PATCH):
            odt = torch.float32
        if self.epi == EPI_QKV:
            self.H = N // 3
            self.heads = self.H // 64
            self.out = nan_like((rows, 2 * self.H), odt)
            lens = self.lens
            self.row0 = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
            assert self.row0[-1] == M and max(lens, default=0) <= self.kv_pitch
            self.vt = nan_like((len(lens) + 2, self.heads, 64, self.kv_pitch), odt)     # two slots past n_slots
            self.vt_lo = nan_like(self.vt.shape, odt)
        elif self.epi == EPI_PATCH:
            self.n_docs = (M + self.n_patch - 1) // self.n_patch
            self.out = nan_like(((self.n_docs + 1) * (self.n_patch + 1), N), odt)   # one document past the last
        else:
            self.out = nan_like((rows, N), odt)
        self.out_lo = nan_like(self.out.shape, torch.bfloat16) if odt == torch.bfloat16 else None

    def run(self, lib, grid=0, a_rows=None, a_view=None, w_view=None, a_pitch=None, w_pitch=None, K=None,
            fresh=True):
        """One launch.  a_view / w_view, a_pitch / w_pitch and K: the K-chunk launches of the fp32-mode MLP-down."""
        if fresh:
            self.alloc_outputs()
        a, a_lo = a_view if a_view is not None else (self.a, self.a_lo)
        w, w_lo = w_view if w_view is not None else (self.w, self.w_lo)
        K = K or self.K
        M, N = self.M, self.N
        m = torch.tensor([M], dtype=torch.int32, device=DEV) if self.m_dev else None
        row0 = n_slots = None
        qk_cols = heads = 0
        if self.epi == EPI_QKV:
            row0 = torch.as_tensor(self.row0, dtype=torch.int32, device=DEV)
            n_slots = torch.tensor([len(self.lens)], dtype=torch.int32, device=DEV)
            qk_cols, heads = 2 * self.H, self.heads
        vt, vt_lo = (self.vt, self.vt_lo) if self.epi == EPI_QKV else (None, None)
        torch.cuda.synchronize()
        rc = lib.gemm_run(self.epi, self.bn, int(self.split), grid, _p(a), _p(a_lo if self.split else None),
                          a_rows if a_rows is not None else a.shape[0], a_pitch or a.shape[1], _p(w),
                          _p(w_lo if self.split else None), w_pitch or w.shape[1], _p(m), M, N, K, _p(self.bias),
                          _p(self.out), _p(self.out_lo), self.out.shape[1], _p(self.resid), _p(self.resid_lo),
                          _p(self.resid_f32), _p(self.resid_y), _p(self.resid_stats), _p(self.resid_src),
                          _p(self.resid_w), _p(self.resid_b), self.resid_prefetch, _p(vt), _p(vt_lo), qk_cols,
                          _p(row0), _p(n_slots), self.kv_pitch, heads, _p(self.pos), self.n_patch, self.n_patch + 1)
        assert rc == 0, f"{self.name()}: gemm_run returned {rc}"

    # -------------------------------------------------------------- outputs -> dense [M, N], untouched regions
    def slot_tok(self):
        """(slot, token) of every row < M."""
        lens = torch.as_tensor(self.lens, dtype=torch.int64, device=DEV)
        slot = torch.repeat_interleave(torch.arange(len(self.lens), device=DEV), lens)
        tok = torch.arange(self.M, device=DEV) - torch.as_tensor(self.row0[:-1], device=DEV)[slot]
        return slot, tok

    def patch_rows(self):
        m = torch.arange(self.M, device=DEV)
        return (m // self.n_patch) * (self.n_patch + 1) + 1 + m % self.n_patch

    def collect(self):
        """-> (hi, lo): the outputs of rows < M as [M, N] (lo None for fp32 outputs and in bf16 mode), after checking
        that nothing outside the written region changed."""
        M, N, what = self.M, self.N, self.name()
        written = torch.zeros(self.out.shape[0], dtype=torch.bool, device=DEV)
        if self.epi == EPI_PATCH:
            written[self.patch_rows()] = True
        else:
            written[:M] = True
        outs = [self.out] + ([self.out_lo] if self.out_lo is not None else [])
        for k, t in enumerate(outs):
            lo_part = k == 1
            if lo_part and not self.split:
                assert torch.isnan(t.float()).all(), f"{what}: out_lo written in bf16 mode"
                continue
            stray = ~torch.isnan(t[~written].float())
            if stray.any():
                rows = torch.nonzero(~written).flatten()
                r = int(rows[int(torch.nonzero(stray.any(1))[0])])
                pytest.fail(f"{what}: {'out_lo' if lo_part else 'out'} row {r} outside the written rows was changed")
        hi = self.out[written][:, :N] if self.epi != EPI_PATCH else self.out[self.patch_rows()]
        lo = (self.out_lo[written] if self.out_lo is not None else None) if self.split else None
        if self.epi == EPI_QKV:
            H, h = self.H, self.heads
            slot, tok = self.slot_tok()
            hd = torch.arange(h, device=DEV)[None, :, None]
            d = torch.arange(64, device=DEV)[None, None, :]
            vmask = torch.zeros(self.vt.shape, dtype=torch.bool, device=DEV)
            vmask[slot[:, None, None], hd, d, tok[:, None, None]] = True
            for k, t in enumerate((self.vt, self.vt_lo)):
                if k == 1 and not self.split:
                    assert torch.isnan(t.float()).all(), f"{what}: vt_lo written in bf16 mode"
                    continue
                stray = ~torch.isnan(t.float()) & ~vmask
                if stray.any():
                    s, hh, dd, tk = [int(x) for x in torch.nonzero(stray)[0]]
                    pytest.fail(f"{what}: {'vt_lo' if k else 'vt'} (slot {s}, head {hh}, d {dd}, token {tk}) outside "
                                f"the documents was changed (n_slots {len(self.lens)}, kv_pitch {self.kv_pitch})")
            v = self.vt[slot[:, None, None], hd, d, tok[:, None, None]].reshape(M, H)
            hi = torch.cat([hi[:, :2 * H], v], 1)
            if self.split:
                vl = self.vt_lo[slot[:, None, None], hd, d, tok[:, None, None]].reshape(M, H)
                lo = torch.cat([lo[:, :2 * H], vl], 1)
        return hi, lo

    def where(self, m, n):
        """A human-readable location of output element (m, n)."""
        bm = 128 if self.bn == 128 else 256
        s = f"(m {m}, n {n}) in tile (m-block {m // bm}, n-block {n // self.bn})"
        if self.epi == EPI_QKV and n >= 2 * self.H:
            slot = int(np.searchsorted(self.row0, m, side="right") - 1)
            nv = n - 2 * self.H
            s += f", V^T (slot {slot}, head {nv // 64}, d {nv % 64}, token {m - int(self.row0[slot])})"
        if self.epi == EPI_PATCH:
            s += f", document {m // self.n_patch} patch {m % self.n_patch}"
        return s

    # -------------------------------------------------------------- fp64 reference
    def reference(self, K_total=None):
        """-> dict: acc (A W^T, the three split products), absacc (sum |a w| over the same terms), dropped (split:
        |A_lo| |W_lo|^T), x (acc + bias), resid (the residual term as the kernel's inputs define it) and its own
        computation error e_resid, y (the epilogue's output before rounding)."""
        M = self.M
        K = K_total or self.K
        A = self.a[:M, :K].double()
        W = self.w[:, :K].double()
        acc = A @ W.T
        absacc = A.abs() @ W.abs().T
        dropped = None
        if self.split:
            Al, Wl = self.a_lo[:M, :K].double(), self.w_lo[:, :K].double()
            acc = acc + Al @ W.T + A @ Wl.T
            absacc = absacc + Al.abs() @ W.abs().T + A.abs() @ Wl.abs().T
            dropped = Al.abs() @ Wl.abs().T
        b = self.bias.double()[None, :]
        r = dict(acc=acc, absacc=absacc, dropped=dropped, x=acc + b, absx=absacc + b.abs())
        e_res = torch.zeros_like(acc)
        res = torch.zeros_like(acc)
        if self.epi == EPI_RESID:
            if self.split and self.resid_f32 is not None:
                res = self.resid_f32[:M].double()
            elif self.resid_y is not None:
                src = (self.resid_src.long() if self.resid_src is not None else torch.arange(M, device=DEV))
                st = self.resid_stats[:M].double()
                t = (self.resid_y[src].double() - st[:, :1]) * st[:, 1:] * self.resid_w.double()[None, :]
                res = t + self.resid_b.double()[None, :]
                e_res = 3 * U_FP32 * t.abs() + U_FP32 * res.abs()     # y - mean, * rstd, * w, + b
            else:
                res = self.resid[:M].double()
                if self.resid_lo is not None:
                    res = res + self.resid_lo[:M].double()
                    e_res = U_FP32 * res.abs()                        # resid + resid_lo
        elif self.epi == EPI_PATCH:
            res = self.pos[1:].double().repeat((M + self.n_patch - 1) // self.n_patch, 1)[:M]
        r["resid"], r["e_resid"] = res, e_res
        if self.epi == EPI_GELU:
            r["y"] = 0.5 * r["x"] * (1.0 + torch.erf(r["x"] / math.sqrt(2.0)))
        else:
            r["y"] = r["x"] + res
        return r


def error_bound(g, ref, n_terms, n_rounds=1):
    """Per-element bound on |kernel output - fp64 output| for Gemm g: [M, N].

    Accumulation: the products are exact in fp32 and every added term costs at most 2^-23 of sum |a w| (truncating
    fp32 accumulation), n_terms = K (3K in the split mode); SPLIT also drops A_lo W_lo^T, at most |A_lo| |W_lo|^T.
    Epilogue: acc + bias is one fp32 rounding (2^-24 |x|).  GELU: the input error times max |gelu'| = 1.13, plus
    |x| |error of Phi|, where Phi = 1 - h or h with h = 0.5 erfc(|x| / sqrt2) = 2^q(z): the fit errs by 4.2e-7 on
    z < 4.3; beyond it the kernel returns the clamped h(4.3) = 0.5 erfc(4.3) (1 +- 0.7 %) while the true h lies in
    (0, 0.5 erfc(4.3)], so by 1.01 * 0.5 erfc(4.3); the fp32 polynomial (|q| <= 31, six FMAs) and ex2.approx (2^-22)
    add 2^-16 h; 1 - h and x * Phi two fp32 roundings, 2^-23 |y|.  RESID / PATCH: the residual or pos-embed add is one
    more fp32 rounding (2^-24 |y|), plus the residual's own computation (resid + resid_lo: 2^-24 |r|; the LayerNorm
    recompute (y - mean) rstd w + b: 3 * 2^-24 |(y - mean) rstd w| + 2^-24 |r|).  n_rounds > 1 (the K-chunked MLP-down)
    charges the bias and residual roundings once per launch, at |acc| + |bias| + |residual|.
    Output: bf16 2^-8 (|y| + e), a (hi, lo) pair 2^-16 (|y| + e); fp32 outputs carry no further rounding.  A factor
    1.01 covers second-order terms."""
    e = n_terms * U_ACC * ref["absacc"]
    if ref["dropped"] is not None:
        e = e + ref["dropped"]
    x, y = ref["x"], ref["y"]
    if n_rounds > 1:
        e = e + 2 * n_rounds * U_FP32 * (ref["absx"] + ref["resid"].abs())
    else:
        e = e + U_FP32 * x.abs()
    if g.epi == EPI_GELU:
        z = x.abs() / math.sqrt(2.0)
        h = 0.5 * torch.special.erfc(z)
        fit = torch.where(z < GELU_CLAMP, GELU_FIT, 1.01 * HALF_ERFC_CLAMP)
        e = 1.13 * e + x.abs() * (fit + U_PAIR * h) + 2 * U_FP32 * y.abs()
    elif g.epi in (EPI_RESID, EPI_PATCH):
        e = e + ref["e_resid"] + (U_FP32 * y.abs() if n_rounds == 1 else 0.0)
    if g.epi in (EPI_BIAS, EPI_GELU, EPI_QKV):
        e = e + (U_PAIR if g.split else U_BF16) * (y.abs() + e)
    return e * 1.01


def check_bound(g, hi, lo, ref, n_terms, n_rounds=1, what=None):
    what = what or g.name()
    got = hi.double() + (lo.double() if lo is not None else 0.0)
    assert torch.isfinite(got).all(), f"{what}: non-finite output"
    bound = error_bound(g, ref, n_terms, n_rounds)
    err = (got - ref["y"]).abs()
    ratio = torch.where(err == 0, torch.zeros_like(err), err / bound)
    worst = float(ratio.max()) if ratio.numel() else 0.0
    if worst > 1.0:
        m, n = [int(v) for v in torch.nonzero(ratio == ratio.max())[0]]
        pytest.fail(f"{what}: {g.where(m, n)}: got {float(got[m, n]):.9g} want {float(ref['y'][m, n]):.9g} "
                    f"bound {float(bound[m, n]):.3g} (ratio {worst:.3g})")
    print(f"{what}: worst |err| / bound = {worst:.4f}")
    return worst


def check_exact(g, hi, lo, ref):
    """Lattice inputs: bf16 outputs equal bf16(y) (SPLIT: hi = bf16(y), lo = bf16(y - hi)); fp32 outputs equal y."""
    y32 = ref["y"].float()
    assert torch.equal(y32.double(), ref["y"]), f"{g.name()}: the lattice result is not exact in fp32"
    if hi.dtype == torch.float32:
        pairs = [("out", hi.view(torch.int32), y32.view(torch.int32))]
    else:
        want_hi = y32.to(torch.bfloat16)
        pairs = [("out", hi.view(torch.int16), want_hi.view(torch.int16))]
        if g.split:
            want_lo = (y32 - want_hi.float()).to(torch.bfloat16)
            pairs.append(("out_lo", lo.view(torch.int16), want_lo.view(torch.int16)))
    for nm, a, b in pairs:
        ne = a != b
        if ne.any():
            m, n = [int(v) for v in torch.nonzero(ne)[0]]
            got = (hi if nm == "out" else lo)[m, n]
            pytest.fail(f"{g.name()}: {int(ne.sum())} {nm} elements differ, first at {g.where(m, n)}: got "
                        f"{float(got):.9g} want {float(ref['y'][m, n]):.9g}")


# ------------------------------------------------------------------------------------------------ lattice inputs
def lattice_ranges(K, split, extra):
    """(amax, jmax): operand integers in [-amax, amax], SPLIT low parts j / 256 with |j| <= jmax, the widest for which
    the largest possible partial sum (K products, the three split segments, plus `extra` for bias and residual) stays
    at or below 2^22 grid steps of 1/256: two bits of margin for the tensor core's internal alignment."""
    for amax in (4, 2, 1):
        for jmax in (8, 4, 2, 1):
            biggest = K * (amax * amax + (2 * amax * jmax * LATTICE_STEP if split else 0.0)) + extra
            if biggest / LATTICE_STEP <= 2 ** 22:
                return amax, jmax, biggest
    raise AssertionError(f"K = {K}: no lattice range keeps the partial sums exact")


def lat_int(g, shape, lim):
    return torch.randint(-lim, lim + 1, shape, generator=g, device=DEV).float()


def lat_frac(g, shape, jmax):
    return torch.randint(-jmax, jmax + 1, shape, generator=g, device=DEV).float() * LATTICE_STEP


def lattice_gemm(epi, bn, split, M, N, K, seed, a_rows=None, resid_kind=None, lens=None, kv_pitch=1024):
    """A Gemm on lattice inputs.  a_rows: rows of the A tensor map (default: M padded with 128 NaN rows)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    BIAS_LIM, RES_LIM = 64, 64
    extra = BIAS_LIM + 1 + (RES_LIM + 1) * 4
    amax, jmax, biggest = lattice_ranges(K, split, extra)
    assert biggest / LATTICE_STEP <= 2 ** 22
    a_rows = a_rows if a_rows is not None else M + 128
    a = lat_int(g, (a_rows, K), amax)
    a[M:] = float("nan")                     # rows past M: NaN (an exact-M map has none; TMA fills zeros)
    w = lat_int(g, (N, K), amax)
    bias = lat_int(g, (N,), BIAS_LIM)
    a_lo = w_lo = None
    if split:
        a_lo = lat_frac(g, (a_rows, K), jmax)
        a_lo[M:] = float("nan")
        w_lo = lat_frac(g, (N, K), jmax)
        bias = bias + lat_frac(g, (N,), 255)
    gm = Gemm(epi, bn, split, M, N, K, a.to(torch.bfloat16), w.to(torch.bfloat16), bias,
              a_lo.to(torch.bfloat16) if split else None, w_lo.to(torch.bfloat16) if split else None)
    rows = M + 128
    if epi == EPI_RESID:
        if split:
            gm.resid_f32 = lat_int(g, (rows, N), RES_LIM) + lat_frac(g, (rows, N), 255)
        elif resid_kind in ("bf16", "lo"):
            gm.resid = lat_int(g, (rows, N), RES_LIM).to(torch.bfloat16)
            if resid_kind == "lo":
                gm.resid_lo = lat_frac(g, (rows, N), 64).to(torch.bfloat16)
        else:                                # "y" / "y_src": (y - mean) rstd w + b exact with rstd = 2^-k
            set_resid_y(gm, g, resid_kind == "y_src", lattice=True)
    if epi == EPI_QKV:
        gm.lens, gm.kv_pitch = lens if lens is not None else ragged_lens(M), kv_pitch
    if epi == EPI_PATCH:
        gm.pos = lat_int(g, (N_PATCH + 1, N), 8) + (lat_frac(g, (N_PATCH + 1, N), 255) if split else 0.0)
        gm.m_dev = False                     # the engine launches the patch GEMM with m_static
    return gm


def set_resid_y(gm, g, with_src, lattice):
    """resid_y rows (fp32) behind output rows < M, through a compaction map into a larger buffer (with_src: as after
    an exit, rows in between left) or row for row.  The source of row M - 1 is the buffer's last row: rows past M read
    row M - 1's source (gemm_resid_rows clamps)."""
    M, N = gm.M, gm.N
    if with_src:
        y_rows = M + 37 + M // 3
        src = torch.sort(torch.randperm(y_rows - 1, generator=torch.Generator().manual_seed(M))[:max(M - 1, 0)])[0]
        src = torch.cat([src, torch.tensor([y_rows - 1])]) if M > 0 else src
        gm.resid_src = src.to(torch.int32).to(DEV)
    else:
        y_rows = M
    y_rows = max(y_rows, 1)
    if lattice:
        gm.resid_y = lat_int(g, (y_rows, N), 64)
        mean = lat_int(g, (max(M, 1), 1), 8)
        rstd = torch.exp2(-torch.randint(0, 4, (max(M, 1), 1), generator=g, device=DEV).float())
        gm.resid_w = lat_int(g, (N,), 3)
        gm.resid_b = lat_frac(g, (N,), 255) * 8.0
    else:
        gm.resid_y = torch.randn(y_rows, N, generator=g, device=DEV) * 3.0 + 0.5
        src = gm.resid_src.long() if with_src else torch.arange(max(M, 1), device=DEV)[:max(M, 1)]
        rows = gm.resid_y[src[:max(M, 1)]] if M > 0 else gm.resid_y[:1]
        mean = rows.mean(1, keepdim=True)
        rstd = torch.rsqrt(rows.var(1, unbiased=False, keepdim=True) + 1e-5)
        gm.resid_w = 1.0 + torch.randn(N, generator=g, device=DEV) * 0.1
        gm.resid_b = torch.randn(N, generator=g, device=DEV) * 0.1
    gm.resid_stats = torch.cat([mean, rstd], 1).contiguous()[:max(M, 1)]


def ragged_lens(M):
    """Documents of the LENS lengths, in turn, covering M rows (the last one shorter)."""
    lens, i = [], 0
    while sum(lens) < M:
        lens.append(min(LENS[i % len(LENS)], M - sum(lens)))
        i += 1
    return lens


def run_lattice(lib, gm, grid=0, a_rows=None):
    gm.run(lib, grid=grid, a_rows=a_rows)
    hi, lo = gm.collect()
    ref = gm.reference()
    if gm.epi == EPI_GELU:                   # addressing only: the GELU arithmetic is held to the derived bound
        check_bound(gm, hi, lo, ref, (3 if gm.split else 1) * gm.K, what=f"lattice {gm.name()}")
    else:
        check_exact(gm, hi, lo, ref)


# the N of each (epilogue, kernel): an odd number of blocks where the engine has one (384 = 3 x 128, 768 = 3 x 256),
# 3H for QKV (H = 128 / 256), I for GELU (1280 = 5 x 256)
LATTICE_N = {(EPI_BIAS, 128): 384, (EPI_BIAS, 256): 768, (EPI_GELU, 128): 640, (EPI_GELU, 256): 1280,
             (EPI_QKV, 128): 384, (EPI_QKV, 256): 768, (EPI_RESID, 128): 384, (EPI_RESID, 256): 768,
             (EPI_PATCH, 128): 384, (EPI_PATCH, 256): 768}
M_SWEEP = [0, 1, 127, 128, 129, 255, 256, 257, 383, 2777]
RESID_KINDS = ["bf16", "lo", "y_src", "y"]


@pytest.mark.parametrize("split", [False, True], ids=["bf16", "split"])
@pytest.mark.parametrize("bn", [128, 256])
@pytest.mark.parametrize("epi", [EPI_BIAS, EPI_GELU, EPI_QKV, EPI_RESID, EPI_PATCH], ids=EPI_NAME.get)
def test_lattice_gemm_is_bit_exact(gemm, epi, bn, split):
    """Every kernel x mode x epilogue over the row counts, k-block counts and grids where tiling and the pipeline go
    wrong.  M: empty, one row, both sides of the 128- and 256-row tile edges, a few thousand ragged rows.  K: one k-block,
    exactly STAGES and STAGES + 1 k-blocks, and the engine's K values.  Grids: the engine's, one CTA (pair) running every
    tile so the stage ring and both accumulators wrap many times, a few CTAs, and more CTAs than tiles.  The A tensor map
    has exactly M rows (TMA zero-fills the tail) or more rows with NaN past M."""
    N = LATTICE_N[(epi, bn)]
    one = 2 if bn == 256 else 1
    cases = []                                                     # (M, K, grid, exact A rows)
    for i, M in enumerate(M_SWEEP):
        cases.append((M, 128, 0, M > 128 and i % 2 == 0))
    for K in sorted({64, 64 * STAGES[bn], 64 * (STAGES[bn] + 1), 256, 768, 1024, 3072}):
        cases.append((257, K, 0, K == 768))
    cases += [(2777, 192, one, False), (2777, 64, 3 * one, True), (1000, 448, 7 * one, False),
              (129, 128, 40 * one, False)]
    for c, (M, K, grid, exact) in enumerate(cases):
        kind = RESID_KINDS[c % len(RESID_KINDS)] if epi == EPI_RESID and not split else None
        gm = lattice_gemm(epi, bn, split, M, N, K, seed=1000 * c + 10 * epi + bn, a_rows=M if exact else None,
                          resid_kind=kind)
        run_lattice(gemm, gm, grid=grid)


@pytest.mark.parametrize("case", ["equal", "one_long", "300_slots", "lens"])
@pytest.mark.parametrize("split", [False, True], ids=["bf16", "split"])
def test_qkv_ragged_scatter_is_bit_exact(gemm, case, split):
    """V^T scatter over ragged documents: the proportional slot guess is exact for equal lengths, far off with one
    1024-row document among 198-row ones (long walks), and the slots run past 256 in a permuted length order.  Every
    V^T element of every (slot, head, d, token < len) is bit-exact; tokens in [len, kv_pitch) and slots >= n_slots stay
    untouched."""
    if case == "equal":
        lens, heads, kv = [709] * 8, 12, 768
    elif case == "one_long":
        lens, heads, kv = [198] * 20 + [1024] + [198] * 20, 16, 1024
    elif case == "300_slots":
        perm = np.random.default_rng(3).permutation(300)
        lens, heads, kv = [LENS[int(p) % 15] for p in perm], 2, 768
    else:
        lens, heads, kv = LENS, 6, 1024
    H = 64 * heads
    M = sum(lens)
    gm = lattice_gemm(EPI_QKV, bn_qkv(H), split, M, 3 * H, H, seed=heads, lens=lens, kv_pitch=kv)
    run_lattice(gemm, gm)


# ------------------------------------------------------------------------------------------------ random inputs
def rand_split(x, split):
    hi = x.to(torch.bfloat16)
    return (hi, (x - hi.float()).to(torch.bfloat16)) if split else (hi, None)


def random_gemm(epi, bn, split, M, N, K, seed, gelu_a=False):
    """Trained-like inputs: LayerNormed A ~ N(0, 1) (GELU outputs of N(0, 1) for the MLP-down), W and bias ~ N(0, 0.02);
    in the split mode every operand is the (hi, lo) pair of an fp32 value."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    a = torch.randn(M + 128, K, generator=g, device=DEV)
    if gelu_a:
        a = torch.nn.functional.gelu(a)
    a[M:] = float("nan")
    w = torch.randn(N, K, generator=g, device=DEV) * 0.02
    bias = torch.randn(N, generator=g, device=DEV) * 0.02
    a, a_lo = rand_split(a, split)
    w, w_lo = rand_split(w, split)
    return Gemm(epi, bn, split, M, N, K, a, w, bias, a_lo, w_lo), g


def random_resid(gm, g, kind):
    M, N = gm.M, gm.N
    x = torch.randn(M + 128, N, generator=g, device=DEV)
    if kind == "f32":
        gm.resid_f32 = x
    elif kind == "lo":
        gm.resid, gm.resid_lo = split_bf16(x)
    else:
        set_resid_y(gm, g, kind == "y_src", lattice=False)


def run_random(lib, gm, grid=0, what=None):
    gm.run(lib, grid=grid)
    hi, lo = gm.collect()
    return check_bound(gm, hi, lo, gm.reference(), (3 if gm.split else 1) * gm.K, what=what)


def run_kchunked(lib, gm, I):
    """The fp32-mode MLP-down as the engine runs it: n_kchunks launches over the K-chunk tensor maps (columns
    c * kchunk .. of rows of pitch I); launch c > 0 adds to the output in place (bias = 0, resid_f32 = out)."""
    kc = kchunk(I)
    a_resid, bias = gm.resid_f32, gm.bias
    gm.alloc_outputs()
    zero = torch.zeros_like(bias)
    for c in range(I // kc):
        av = (gm.a[:, c * kc:], gm.a_lo[:, c * kc:])
        wv = (gm.w[:, c * kc:], gm.w_lo[:, c * kc:])
        gm.bias, gm.resid_f32 = (bias, a_resid) if c == 0 else (zero, gm.out)
        gm.run(lib, a_view=av, w_view=wv, a_pitch=I, w_pitch=I, K=kc, a_rows=gm.a.shape[0], fresh=False)
    gm.bias, gm.resid_f32 = bias, a_resid
    hi, lo = gm.collect()
    ref = gm.reference()
    return check_bound(gm, hi, lo, ref, 3 * kc, n_rounds=I // kc,
                       what=f"{gm.name()} in {I // kc} K-chunks of {kc}")


HIDDEN = [128, 256, 384, 512, 640, 768, 896, 1024]
DOCS = LENS[:5]                                                    # 1165 ragged rows


@pytest.mark.parametrize("split", [False, True], ids=["bf16", "split"])
@pytest.mark.parametrize("H", HIDDEN)
def test_layer_gemms_within_derived_bound(gemm, H, split):
    """The four GEMMs of an encoder layer at every hidden size mmee_create accepts, I = 2H and 4H, on the kernel the
    engine picks for each: QKV, the out-projection with its residual (bf16 mode: recomputed from the LayerNorm sums
    through a row map; fp32 mode: the fp32 residual), MLP-up + GELU, MLP-down with its residual (fp32 mode: K-chunked
    as the engine runs it)."""
    M = sum(DOCS)
    gm, g = random_gemm(EPI_QKV, bn_qkv(H), split, M, 3 * H, H, seed=H)
    gm.lens, gm.kv_pitch = DOCS, 768
    run_random(gemm, gm)
    gm, g = random_gemm(EPI_RESID, pick_bn(H), split, M, H, H, seed=H + 1)
    random_resid(gm, g, "f32" if split else "y_src")
    run_random(gemm, gm, what=f"{gm.name()} out-projection")
    for I in (2 * H, 4 * H):
        gm, g = random_gemm(EPI_GELU, pick_bn(I), split, M, I, H, seed=H + I)
        run_random(gemm, gm)
        gm, g = random_gemm(EPI_RESID, pick_bn(H), split, M, H, I, seed=H + I + 1, gelu_a=True)
        random_resid(gm, g, "f32" if split else "y")
        if split and I // kchunk(I) > 1:
            run_kchunked(gemm, gm, I)
        else:
            run_random(gemm, gm, what=f"{gm.name()} MLP-down")


@pytest.mark.parametrize("split", [False, True], ids=["bf16", "split"])
@pytest.mark.parametrize("channels,H", [(1, 128), (3, 128), (1, 768), (3, 768), (3, 1024)])
def test_patch_gemm_within_derived_bound(gemm, channels, H, split):
    """The patch embedding as the engine runs it: K = channels * 16 * 16, 5 documents of 196 patches (m_static), +bias
    +pos_embed[1 + p] into rows doc * 197 + 1 + p; CLS rows untouched."""
    K = channels * 256
    gm, g = random_gemm(EPI_PATCH, pick_bn(H), split, 5 * N_PATCH, H, K, seed=K + H)
    gm.pos = torch.randn(N_PATCH + 1, H, generator=g, device=DEV) * 0.02
    gm.m_dev = False
    run_random(gemm, gm)


@pytest.mark.parametrize("split", [False, True], ids=["bf16", "split"])
@pytest.mark.parametrize("bn", [128, 256])
def test_gelu_over_its_whole_range(gemm, bn, split):
    """A = W = 0, so the GELU input is the fp32 bias itself: a dense sweep of [-12, 12] with the clamp point
    |x| = 4.3 sqrt2 and its fp32 neighbours, and values around 0.  Held to the bound of the random tests, which is the
    accuracy gemm.cuh claims for the fitted GELU (4.2e-7 on Phi below the clamp, the clamp's 6e-10 beyond it)."""
    N = 24576
    x = torch.linspace(-12.0, 12.0, N - 256, device=DEV)
    c = torch.tensor(GELU_CLAMP * math.sqrt(2.0), dtype=torch.float32)
    special = [0.0, -0.0, 1e-30, -1e-30, 1e-7, -1e-7, 1e-3, -1e-3, 0.5, -0.5, 1.0, -1.0]
    for s in (1.0, -1.0):
        v = c * s
        for _ in range(12):
            special += [float(v)]
            v = torch.nextafter(v, torch.tensor(100.0 * s))
        v = c * s
        for _ in range(12):
            v = torch.nextafter(v, torch.tensor(0.0))
            special += [float(v)]
    special += list(np.linspace(-6.2, -5.9, 256 - len(special)))
    bias = torch.cat([x, torch.tensor(special, dtype=torch.float32, device=DEV)])
    M, K = 128, 64
    z = torch.zeros(M + 128, K, dtype=torch.bfloat16, device=DEV)
    wz = torch.zeros(N, K, dtype=torch.bfloat16, device=DEV)
    gm = Gemm(EPI_GELU, bn, split, M, N, K, z, wz, bias, z.clone() if split else None, wz.clone() if split else None)
    run_random(gemm, gm, what=f"GELU sweep bn {bn} {'split' if split else 'bf16'}")


@pytest.mark.parametrize("kind,bn,H,prefetch", [
    ("y_src", 256, 768, 0), ("y_src", 256, 768, 1), ("y", 256, 1024, 1), ("y", 256, 256, 0),
    ("y_src", 128, 384, 0), ("y", 128, 640, 0), ("lo", 128, 384, 0), ("lo", 256, 768, 0)])
def test_residual_variants_within_derived_bound(gemm, kind, bn, H, prefetch):
    """The bf16-mode residuals the engine uses: LayerNorm(resid_y[src(r)]) recomputed from the sums, through a
    compaction map into a larger buffer (an exit in between) or row for row, with the pair kernel's L2 prefetch on and
    off; and resid + resid_lo.  Ragged M so the last tile has rows past M, which read row M - 1's source."""
    M = 2777
    gm, g = random_gemm(EPI_RESID, bn, False, M, H, H, seed=H + prefetch)
    random_resid(gm, g, kind)
    gm.resid_prefetch = prefetch
    run_random(gemm, gm, what=f"{gm.name()} resid {kind} prefetch {prefetch}")


@pytest.mark.parametrize("H,I", [(384, 1536), (768, 1536), (768, 3072), (1024, 4096)])
def test_kchunked_mlp_down_within_derived_bound(gemm, H, I):
    """The fp32-mode MLP-down in K chunks (I = 1536: two of 768, 3072: three of 1024, 4096: four of 1024) against fp64
    over the full K."""
    gm, g = random_gemm(EPI_RESID, pick_bn(H), True, 1165, H, I, seed=I + H, gelu_a=True)
    random_resid(gm, g, "f32")
    run_kchunked(gemm, gm, I)


# ------------------------------------------------------------------------------------------------ independence
def doc_rows(seed, L, K):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randn(L, K, generator=g, device=DEV)


@pytest.mark.parametrize("split", [False, True], ids=["bf16", "split"])
@pytest.mark.parametrize("H", [384, 768])
def test_qkv_independent_of_slot_and_neighbours(gemm, H, split):
    """The same documents in another slot order, with every other document's rows replaced: each kept document's Q, K
    and V^T are bit-identical."""
    lens = LENS[:9]
    n = len(lens)
    g = torch.Generator(device=DEV).manual_seed(H)
    w = torch.randn(3 * H, H, generator=g, device=DEV) * 0.02
    bias = torch.randn(3 * H, generator=g, device=DEV) * 0.02
    w, w_lo = rand_split(w, split)
    keep = set(range(0, n, 2))
    outs = []
    for order, seed in ((list(range(n)), 0), ([int(x) for x in np.random.default_rng(2).permutation(n)], 1)):
        rows = [doc_rows(d if d in keep else 100 + d + seed, lens[d], H) for d in order]
        a = torch.cat(rows + [torch.full((128, H), float("nan"), device=DEV)])
        a, a_lo = rand_split(a, split)
        M = sum(lens)
        gm = Gemm(EPI_QKV, bn_qkv(H), split, M, 3 * H, H, a, w, bias, a_lo, w_lo)
        gm.lens, gm.kv_pitch = [lens[d] for d in order], 1024
        gm.run(gemm)
        gm.collect()
        outs.append((gm, order))
    for d in keep:
        got = []
        for gm, order in outs:
            s = order.index(d)
            r0, L = int(gm.row0[s]), lens[d]
            parts = [gm.out[r0:r0 + L], gm.vt[s, :, :, :L]]
            if split:
                parts += [gm.out_lo[r0:r0 + L], gm.vt_lo[s, :, :, :L]]
            got.append([p.contiguous().view(torch.int16) for p in parts])
        for x, y in zip(*got):
            assert torch.equal(x, y), f"H {H}: document {d}: Q/K/V^T depends on its slot or its neighbours"


@pytest.mark.parametrize("split", [False, True], ids=["bf16", "split"])
@pytest.mark.parametrize("bn", [128, 256])
def test_output_independent_of_grid(gemm, bn, split):
    """A tile's k order does not depend on which CTA runs it: QKV and residual outputs are bit-identical for the
    engine's grid, one CTA (pair) and a few."""
    one = 2 if bn == 256 else 1
    H = 256 if bn == 256 else 384
    for epi in (EPI_QKV, EPI_RESID):
        N = 3 * H if epi == EPI_QKV else H
        gm, g = random_gemm(epi, bn, split, 1165, N, H, seed=bn + epi)
        if epi == EPI_QKV:
            gm.lens, gm.kv_pitch = DOCS, 768
        else:
            random_resid(gm, g, "f32" if split else "y_src")
        first = None
        for grid in (0, one, 5 * one):
            gm.run(gemm, grid=grid)
            hi, lo = gm.collect()
            bits = [hi.contiguous().view(torch.int16 if hi.dtype == torch.bfloat16 else torch.int32)]
            if lo is not None:
                bits.append(lo.contiguous().view(torch.int16))
            if first is None:
                first = bits
            else:
                for x, y in zip(first, bits):
                    assert torch.equal(x, y), f"{gm.name()}: output differs between the engine's grid and {grid} CTAs"
