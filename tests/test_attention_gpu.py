"""The fused attention kernel (csrc/attention.cuh) and the attention-bias kernels (csrc/norm_exit.cuh) element by element
against plain fp64 torch.

The logit tests only see attention through the CLS row, diluted over ~709 keys, and never read the bias at all.  Here
the attention kernel runs stand-alone through tests/kernels/attention_harness.cu (the engine's own tensor maps and
launch) on inputs built in the engine's layouts, and every ctx element is checked:

* one-hot attention (Q = K = 0, the bias alone picks one key per query row): the result must equal that key's V column
  bit for bit, so a failure names the document, head, query row and key tile;
* random trained-like inputs: every element within a bound derived from the kernel's arithmetic (not fitted);
* isolation: rows past the work list keep their contents, masked keys weigh exactly 0, a document's ctx does not
  depend on its slot or its neighbours, the row planner equals host prefix sums.

The bias test runs the engine itself (bias_build_kernel / bias_build_split_kernel) and compares its BIAS buffer with
`oracle.port.attention_bias` on a float64 state dict.

bf16 has 8 significand bits, so round-to-nearest errs by at most 2^-8 relative (fp16: 2^-11); the fp32 tensor-core
accumulations are charged one fp32 ulp (2^-23, truncation allowed) per added term.
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

HARNESS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "kernels", "attention_harness.cu")
LOG2E = 1.4426950408889634
MASKED = -60000.0                      # BIAS_MASKED (norm_exit.cuh)
U_BF16, U_FP16, U_ACC, U_FP32 = 2.0 ** -8, 2.0 ** -11, 2.0 ** -23, 2.0 ** -24
EX2_REL = 2.0 ** -22                   # ex2.approx.ftz.f32: 2 ulp (PTX ISA)
# lengths per document: the 198-row minimum (CLS + 197 visual), tile edges of 64 / 128, the tail-16 boundary (336: 16
# real keys in the last tile, 337: 17), 709 = a full document, 1024 = ATT_MAX_KV_TILES key tiles
LENS = [198, 199, 255, 256, 257, 320, 336, 337, 383, 384, 385, 641, 656, 657, 709, 1024]


@pytest.fixture(scope="module")
def att(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("attention_harness") / "libattention_harness.so")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    subprocess.check_call([nvcc] + ge.NVCC_FLAGS + ["-I", ge.CSRC, "--shared", HARNESS, "-o", out])
    lib = C.CDLL(out)
    p, i = C.c_void_p, C.c_int
    lib.att_plan.argtypes = [p] * 8
    lib.att_plan.restype = i
    lib.att_run.argtypes = [p] * 12 + [i] * 10
    lib.att_run.restype = i
    return lib


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def plan(att, slot_doc, doc_len):
    """plan_rows_kernel on the device -> dict of device tensors (row0, meta [n, 4], qt_slot, n_qt, m)."""
    dev = torch.device("cuda")
    n, B = len(slot_doc), len(doc_len)
    sd = torch.as_tensor(slot_doc, dtype=torch.int32, device=dev)
    dl = torch.as_tensor(doc_len, dtype=torch.int32, device=dev)
    max_qt = sum((int(x) + 127) // 128 for x in doc_len)
    r = dict(row0=torch.full((B + 1,), -7, dtype=torch.int32, device=dev),
             meta=torch.full((B, 4), -7, dtype=torch.int32, device=dev),
             qt_slot=torch.full((max_qt + 1,), -7, dtype=torch.int32, device=dev),
             n_qt=torch.zeros(1, dtype=torch.int32, device=dev), m=torch.zeros(1, dtype=torch.int32, device=dev))
    n_dev = torch.tensor([n], dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    assert att.att_plan(_p(sd), _p(dl), _p(n_dev), _p(r["row0"]), _p(r["meta"]), _p(r["qt_slot"]), _p(r["n_qt"]),
                        _p(r["m"])) == 0
    return r


def host_plan(slot_doc, doc_len):
    lens = np.array([doc_len[d] for d in slot_doc], dtype=np.int64)
    nq = (lens + 127) // 128
    row0 = np.concatenate([[0], np.cumsum(lens)])
    q0 = np.concatenate([[0], np.cumsum(nq)])
    qt_slot = np.repeat(np.arange(len(lens)), nq)
    meta = np.stack([row0[:-1], lens, np.asarray(slot_doc), q0[:-1]], axis=1)
    return row0, meta, qt_slot, int(q0[-1]), int(row0[-1])


def split_bf16(x):
    hi = x.to(torch.bfloat16)
    return hi, (x - hi.float()).to(torch.bfloat16)


class Problem:
    """Attention inputs of n_docs documents in the engine's layouts.  Document d has doc_len[d] rows; slot s holds
    document slot_doc[s].  Per-document contents come from `make(d)` -> (q [h,L,64], k [h,L,64], v [h,L,64],
    bias [h,L,L]) float32 on the device (bias already containing -60000 on masked keys), so they do not depend on
    the slot a document occupies."""

    def __init__(self, att, heads, seq, doc_len, slot_doc, make, split=False, fill_rows=None):
        dev = torch.device("cuda")
        slot_doc = [int(x) for x in slot_doc]
        self.att, self.heads, self.seq, self.doc_len, self.slot_doc, self.split = att, heads, seq, doc_len, slot_doc, split
        self.H = H = heads * 64
        self.kv_pitch = (seq + 127) // 128 * 128
        self.bias_pitch = (seq + 63) // 64 * 64
        B = len(doc_len)
        self.plan = plan(att, slot_doc, doc_len)
        self.M = int(self.plan["m"].item())
        self.m_rows = self.M + 128
        g = torch.Generator(device=dev).manual_seed(12345)
        # rows outside every document (past M) hold keys at the scale of real keys
        qk = torch.randn(self.m_rows, 2 * H, generator=g, device=dev) * (fill_rows if fill_rows is not None else 0.0)
        vt = torch.empty(B, heads, 64, self.kv_pitch, device=dev)
        # V^T columns between a document's row count and kv_pitch: large FINITE values (masked weight must be exactly 0)
        vt[...] = torch.where(torch.arange(self.kv_pitch, device=dev) % 2 == 0, 1e4, -1e4)
        bias = torch.full((B, heads, seq, self.bias_pitch), MASKED, device=dev)
        self.docs = {}
        row0 = self.plan["row0"].cpu().numpy()
        for s, d in enumerate(slot_doc):
            L = doc_len[d]
            q, k, v, b = make(d)
            self.docs[d] = (q, k, v, b)
            r0 = int(row0[s])
            qk[r0:r0 + L, :H] = q.transpose(0, 1).reshape(L, H)
            qk[r0:r0 + L, H:] = k.transpose(0, 1).reshape(L, H)
            vt[s, :, :, :L] = v.transpose(1, 2)
            bias[d, :, :L, :L] = b
        if split:
            self.qk, self.qk_lo = split_bf16(qk)
            self.vt, self.vt_lo = split_bf16(vt)
            self.bias = bias.half()
            self.bias_lo = torch.where(bias == MASKED, 0.0, bias - self.bias.float()).half()
        else:
            self.qk, self.vt, self.bias = qk.to(torch.bfloat16), vt.to(torch.bfloat16), bias.half()
            self.qk_lo = self.vt_lo = self.bias_lo = None

    def run(self, tail16=True, one_cta=False):
        """-> ctx [m_rows, H] as float64 (hi + lo in split mode); asserts rows >= M kept their NaN pre-fill and the
        error flag stayed 0."""
        dev = torch.device("cuda")
        ctx = torch.full((self.m_rows, self.H), float("nan"), dtype=torch.bfloat16, device=dev)
        ctx_lo = torch.full_like(ctx, float("nan")) if self.split else None
        err = torch.zeros(2, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        rc = self.att.att_run(_p(self.qk), _p(self.qk_lo), _p(self.vt), _p(self.vt_lo), _p(self.bias), _p(self.bias_lo),
                              _p(ctx), _p(ctx_lo), _p(self.plan["meta"]), _p(self.plan["qt_slot"]), _p(self.plan["n_qt"]),
                              _p(err), self.m_rows, self.H, self.heads, self.seq, len(self.doc_len), self.kv_pitch,
                              self.bias_pitch, int(tail16), int(self.split), int(one_cta))
        assert rc == 0
        assert int(err[0].item()) == 0, "attention error flag set"
        assert torch.isnan(ctx[self.M:].float()).all(), "the kernel wrote rows past the work list"
        if self.split:
            assert torch.isnan(ctx_lo[self.M:].float()).all()
            return ctx, ctx.double() + ctx_lo.double()
        return ctx, ctx.double()

    def operands(self, s):
        """fp64 operands of slot s exactly as the kernel reads them: q, k [h,L,64], v [h,L,64], bias [h,L,L], and the
        dropped split product |q_lo| |k_lo|^T (None in bf16 mode)."""
        d = self.slot_doc[s]
        L, H, h = self.doc_len[d], self.H, self.heads
        r0 = int(self.plan["row0"][s].item())

        def rows(t):
            return t[r0:r0 + L].double().view(L, 2, h, 64).permute(1, 2, 0, 3)     # [2, h, L, 64]

        qk = rows(self.qk)
        v = self.vt[s, :, :, :L].double().transpose(1, 2)
        b = self.bias[d, :, :L, :L].double()
        dropped = None
        if self.split:
            lo = rows(self.qk_lo)
            qk = qk + lo
            v = v + self.vt_lo[s, :, :, :L].double().transpose(1, 2)
            b = b + self.bias_lo[d, :, :L, :L].double()
            dropped = lo[0].abs() @ lo[1].abs().transpose(1, 2)
        return qk[0], qk[1], v, b, dropped


def reference(q, k, v, b):
    """fp64 attention in the log2 domain: s = q k^T + b, p = 2^(s - max s), ctx = sum p v / sum p."""
    s = q @ k.transpose(1, 2) + b
    m = s.amax(-1, keepdim=True)
    p = torch.exp2(s - m)
    l = p.sum(-1, keepdim=True)
    return s, m, p, l, (p @ v) / l


def error_bound(q, k, v, b, s, m, p, l, ctx, split, dropped):
    """Per-element bound on |kernel ctx - fp64 ctx| for one (slot): [h, L, 64].

    The kernel's P_j equals p_j (1 + e_j) up to the common factor 2^(ref - max s), with
      e_j <= u_P + EX2_REL + ln2 * (dS_j + 2^-24 (|s_j - max s| + 9))
    u_P: P rounded to bf16 (2^-8), or to the split pair hi + lo (2^-16); dS_j: fp32 tensor-core accumulation of the
    score (2^-23 per term: 64 products + the bias, three product sets + two bias parts when split) plus, when split,
    the dropped q_lo k_lo product; |s - ref| <= |s - max s| + 9 (the reference sits at most 2^8 below the running max,
    or <1 above it after a ceil).  P enters numerator and denominator (the ones row of V^T), so
      |ctx~ - ctx| <= sum_j p_j e_j |v_j - ctx| / sum_j p_j            ( = 2^-8 w + ... in the bf16 kernel)
    with second-order terms covered by a factor 1.01.  On top: the fp32 accumulation of P V and of the row sum over n
    keys, (n + 2) 2^-23 (sum p|v| / sum p + |ctx|), which also covers the 1/l and the product with it; in split mode
    the dropped P_lo V_lo term, 2^-16 sum p|v| / sum p; and the output rounding, 2^-8 |ctx| (bf16) or 2^-16 (hi + lo)."""
    n = k.shape[1]
    nterm = (3 * 64 + 2) if split else (64 + 1)
    qk_abs = q.abs() @ k.abs().transpose(1, 2)
    dS = (nterm + 1) * U_ACC * (qk_abs + b.abs())
    if dropped is not None:
        dS = dS + dropped
    u_p = 2.0 ** -16 if split else U_BF16
    e = u_p + EX2_REL + math.log(2.0) * (dS + U_FP32 * ((s - m).abs() + 9.0))
    pe = (p * e).float()
    v32, c32 = v.float(), ctx.float()
    first = torch.empty_like(c32)
    L = q.shape[1]
    step = max(1, (1 << 24) // (L * 64))
    for i in range(0, L, step):              # sum_j p_ij e_ij |v_j - ctx_i| (fp32 sum: < 1e-6 relative to itself)
        dv = (v32[:, None, :, :] - c32[:, i:i + step, None, :]).abs()
        first[:, i:i + step] = (pe[:, i:i + step, :, None] * dv).sum(2)
    first = first.double() / l * 1.01
    mabs = (p @ v.abs()) / l
    acc = (n + 2) * U_ACC * (mabs + ctx.abs())
    if split:
        acc = acc + 2.0 ** -16 * mabs
    out = (2.0 ** -16 if split else U_BF16) * (ctx.abs() + first + acc)
    return first + acc + out


def slot_ctx(prob, ctx, s):
    d = prob.slot_doc[s]
    L, h = prob.doc_len[d], prob.heads
    r0 = int(prob.plan["row0"][s].item())
    return ctx[r0:r0 + L].view(L, h, 64).transpose(0, 1)               # [h, L, 64]


# ------------------------------------------------------------------------------------------------ one-hot addressing
def preferred_key(L, i, h, d):
    """The key query row i of (document d, head h) attends to.  Over the rows of one (d, h): row 0 -> key 0, row 1 ->
    the last key, then one key in every key tile, then every key of the last tile (all positions of a 16-key tail
    tile), the rest spread.  Rows are rotated per head so every head sees every pattern on other rows."""
    r = (i + 3 * h) % L
    n_tiles = (L + 63) // 64
    last0 = (n_tiles - 1) * 64
    if r == 0:
        return 0
    if r == 1:
        return L - 1
    if r < 2 + n_tiles:
        t = r - 2
        return 64 * t + (r * 5 + d) % min(64, L - 64 * t)
    if r < 2 + n_tiles + (L - last0):
        return last0 + (r - 2 - n_tiles)
    return (r * 37 + h * 11 + d * 3) % L


OFFSETS = (-30.0, -45.0, MASKED)        # lazy rescale path, ATT_JUMP path, rescale factor underflowing to 0


def make_onehot(doc_len, heads):
    """Q = K = 0: the scores are the bias.  The preferred key of a row gets 0, every other key the row's offset (one
    of OFFSETS).  V^T holds integers in [1, 255] (exact in bf16) that encode (document, head, key).

    Why the result is exactly the preferred key's value v*: the kernel's P is a power of two for every key (2^0,
    2^-30, 2^-45 or 0 against the row reference, after the reference has been raised onto the preferred key by the lazy
    or the jump path; before that, other keys have P = 1 and the O they built is rescaled by 2^-30, 2^-45 or 0 when
    the preferred key arrives), so all products and the ones-row sum are exact up to fp32 accumulation.  The other
    keys' total weight relative to v* is at most 1024 * 2^-30 = 2^-20, so ctx = v* (1 + d) with
    |d| <= 255 * 2^-20 / 1 + 2^-20 < 2^-11, below half a bf16 ulp (2^-9 relative just under a power of two); the fp32
    accumulation adds < 2^-13.  Round-to-nearest then returns v* exactly."""
    dev = torch.device("cuda")
    pref = {}

    def make(d):
        L = doc_len[d]
        i = np.arange(L)
        P = np.stack([[preferred_key(L, int(r), hh, d) for r in i] for hh in range(heads)])     # [h, L]
        pref[d] = P
        off = torch.tensor([[OFFSETS[(r + hh + d) % 3] for r in range(L)] for hh in range(heads)], device=dev)
        b = off[:, :, None].expand(heads, L, L).clone()
        b.scatter_(2, torch.as_tensor(P, device=dev)[:, :, None], 0.0)
        j = torch.arange(L, device=dev)
        v = 1.0 + ((j[None, :, None] * 61 + torch.arange(64, device=dev)[None, None, :] * 17
                    + torch.arange(heads, device=dev)[:, None, None] * 29 + d * 11) % 255).float()
        z = torch.zeros(heads, L, 64, device=dev)
        return z, z, v, b

    return make, pref


def check_onehot(prob, ctx, pref, what):
    bad = []
    for s, d in enumerate(prob.slot_doc):
        got = slot_ctx(prob, ctx, s)                                     # bf16 [h, L, 64]
        v = prob.docs[d][2]                                              # [h, L, 64]
        P = torch.as_tensor(pref[d], device=got.device)
        want = torch.gather(v, 1, P[:, :, None].expand(-1, -1, 64)).to(torch.bfloat16)
        ne = (got.contiguous().view(torch.int16) != want.view(torch.int16)).any(-1)   # [h, L]
        if ne.any():
            hh, r = [int(x) for x in torch.nonzero(ne)[0]]
            bad.append(f"doc {d} (slot {s}, {prob.doc_len[d]} rows): {int(ne.sum())} rows wrong, first head {hh} row {r} "
                       f"(query tile {r // 128}), preferred key {pref[d][hh, r]} (key tile {pref[d][hh, r] // 64})")
    assert not bad, f"{what}: " + "; ".join(bad[:6])


@pytest.mark.parametrize("heads,tail16,one_cta,split", [
    (2, True, False, False), (6, True, False, False), (12, True, False, False), (16, True, False, False),
    (12, False, False, False), (12, True, True, False), (12, False, False, True)])
def test_onehot_attention_is_bit_exact(att, heads, tail16, one_cta, split):
    doc_len = LENS
    make, pref = make_onehot(doc_len, heads)
    prob = Problem(att, heads, 1024, doc_len, list(range(len(doc_len))), make, split=split)
    hi, ctx = prob.run(tail16=tail16, one_cta=one_cta)
    check_onehot(prob, hi, pref, f"heads {heads} tail16 {tail16} one_cta {one_cta} split {split}")
    if split:                                   # hi is v*, and hi + lo stays within 2^-11 of it (see make_onehot)
        for s, d in enumerate(prob.slot_doc):
            got = slot_ctx(prob, ctx, s)
            want = torch.gather(prob.docs[d][2].double(), 1,
                                torch.as_tensor(pref[d], device=got.device)[:, :, None].expand(-1, -1, 64))
            assert ((got - want).abs() <= 2.0 ** -11 * want).all()


def test_onehot_many_documents_walk_the_work_list(att):
    """300 documents x 12 heads: ~3000 (document, head, query tile) items, so every CTA of the persistent grid walks
    its work list several times; lengths cycle through LENS below 709, slots map to documents in a shuffled order."""
    heads = 12
    lens = [LENS[i % 15] for i in range(300)]
    order = [int(x) for x in np.random.default_rng(5).permutation(300)]
    make, pref = make_onehot(lens, heads)
    prob = Problem(att, heads, 712, lens, order, make)
    hi, _ = prob.run()
    check_onehot(prob, hi, pref, "300 documents")


# ------------------------------------------------------------------------------------------------ random, derived bound
def make_random(doc_len, heads, seed, ramps=True):
    """Trained-like scores: q.k with std ~6 log2 units plus a bias of std 2, so scores span tens of log2 units within
    a row.  On every third query row the bias carries a ramp of +12 per key tile (the row maximum moves up by more
    than 2^8 from tile to tile: lazy rescale on every tile); on every seventh row one key in the middle jumps 60 above
    its neighbours (ATT_JUMP path).  Some real keys are masked (-60000) as padded text keys / a masked CLS are."""
    dev = torch.device("cuda")

    def make(d):
        L = doc_len[d]
        g = torch.Generator(device=dev).manual_seed(seed * 100003 + d)
        q = torch.randn(heads, L, 64, generator=g, device=dev) * 0.87
        k = torch.randn(heads, L, 64, generator=g, device=dev) * 0.87
        v = torch.randn(heads, L, 64, generator=g, device=dev)
        b = torch.randn(heads, L, L, generator=g, device=dev) * 2.0
        if ramps:
            i = torch.arange(L, device=dev)
            ramp = 12.0 * (i // 64).float()
            b[:, i % 3 == 1, :] += ramp[None, None, :]
            b[:, i % 7 == 3, L // 2 + 5] += 60.0
        if d % 4 == 1:                                   # a masked CLS key and a masked run of keys
            b[:, :, 0] = MASKED
            b[:, :, 40:60] = MASKED
        return q, k, v, b

    return make


def check_bound(prob, ctx, what):
    worst = 0.0
    for s, d in enumerate(prob.slot_doc):
        q, k, v, b, dropped = prob.operands(s)
        sc, m, p, l, ref = reference(q, k, v, b)
        bound = error_bound(q, k, v, b, sc, m, p, l, ref, prob.split, dropped)
        got = slot_ctx(prob, ctx, s)
        assert torch.isfinite(got).all(), f"{what}: non-finite ctx in document {d}"
        ratio = (got - ref).abs() / bound
        r = float(ratio.max())
        if r > 1.0:
            hh, row, col = [int(x) for x in torch.nonzero(ratio == ratio.max())[0]]
            pytest.fail(f"{what}: document {d} ({prob.doc_len[d]} rows) head {hh} row {row} dim {col}: "
                        f"got {float(got[hh, row, col]):.6g} want {float(ref[hh, row, col]):.6g} "
                        f"bound {float(bound[hh, row, col]):.3g} (ratio {r:.3g})")
        worst = max(worst, r)
    print(f"{what}: worst |err| / bound = {worst:.3f}")
    return worst


@pytest.mark.parametrize("heads,tail16,one_cta,split", [
    (2, True, False, False), (6, True, False, False), (12, True, False, False), (16, True, False, False),
    (12, False, False, False), (12, True, True, False), (6, False, False, True), (12, False, False, True)])
def test_random_attention_within_derived_bound(att, heads, tail16, one_cta, split):
    make = make_random(LENS, heads, seed=heads)
    prob = Problem(att, heads, 1024, LENS, list(range(len(LENS))), make, split=split, fill_rows=0.87)
    _, ctx = prob.run(tail16=tail16, one_cta=one_cta)
    check_bound(prob, ctx, f"heads {heads} tail16 {tail16} one_cta {one_cta} split {split}")


# ------------------------------------------------------------------------------------------------ isolation
def test_ctx_independent_of_slot_and_neighbours(att):
    """The same documents in another slot order, with the contents of every other document replaced: each kept
    document's ctx is bit-identical.  Neighbouring K rows are real-scale keys, so only the finite -60000 mask (and the
    key-tile bounds) keep them out."""
    heads, lens = 6, LENS[:15]
    n = len(lens)
    a = Problem(att, heads, 712, lens, list(range(n)), make_random(lens, heads, seed=7), fill_rows=0.87)
    ctx_a, _ = a.run()
    keep = set(range(0, n, 2))
    other = make_random(lens, heads, seed=8)
    base = make_random(lens, heads, seed=7)
    order = [int(x) for x in np.random.default_rng(1).permutation(n)]
    b = Problem(att, heads, 712, lens, order, lambda d: base(d) if d in keep else other(d), fill_rows=0.87)
    ctx_b, _ = b.run()
    for d in keep:
        ga = slot_ctx(a, ctx_a, a.slot_doc.index(d)).contiguous().view(torch.int16)
        gb = slot_ctx(b, ctx_b, b.slot_doc.index(d)).contiguous().view(torch.int16)
        assert torch.equal(ga, gb), f"document {d}: ctx depends on its slot / neighbours"


@pytest.mark.parametrize("n_slots,n_docs", [(1, 1), (7, 9), (256, 256), (300, 400), (600, 600)])
def test_row_plan_equals_host_prefix_sums(att, n_slots, n_docs):
    """plan_rows_kernel: row0, meta, qt_slot, the query-tile count and M equal host prefix sums, also past 256 slots
    where the block walks the slots in chunks."""
    rng = np.random.default_rng(n_slots)
    doc_len = [int(x) for x in rng.integers(198, 1025, n_docs)]
    slot_doc = [int(x) for x in rng.permutation(n_docs)[:n_slots]]
    r = plan(att, slot_doc, doc_len)
    row0, meta, qt_slot, n_qt, M = host_plan(slot_doc, doc_len)
    assert int(r["m"].item()) == M and int(r["n_qt"].item()) == n_qt
    assert np.array_equal(r["row0"].cpu().numpy()[:n_slots + 1], row0)
    assert np.array_equal(r["meta"].cpu().numpy()[:n_slots], meta)
    assert np.array_equal(r["qt_slot"].cpu().numpy()[:n_qt], qt_slot)


# ------------------------------------------------------------------------------------------------ bias, through the engine
@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
@pytest.mark.parametrize("case", ["tiny", "base", "large", "h384"])
def test_bias_build_matches_port(case, dtype):
    """BIAS (and BIASlo in the fp32 mode) after a dense forward vs port.attention_bias on a float64 state dict, times
    log2(e)/8, at the kept-token ranks.  Relative-position tables at std 1 (trained-like), padded documents, one
    document with a masked CLS, boxes over the full [0, 1000] range.

    bias_build_kernel: T1 = fp32(W1 c), T2 = fp16(fp32(fp32(Wx + Wy) c)), out = fp16(fp32(T1 + T2)) with
    c = fp32(log2 e) / 8, so |out - want| <= 2^-11 (|want| + |(Wx + Wy) c|) + 5 * 2^-24 (|W1| + |Wx| + |Wy|) c + 2^-24
    (two fp16 subnormal half-ulps), times 1.01 for second-order terms.  bias_build_split_kernel: v = fp32(T1 + fp32(TX
    + TY)) from fp32 tables, hi = fp16(v), lo = fp16(v - hi): |hi + lo - want| <= 2^-22 |want| * 1.01
    + 5 * 2^-24 (|W1| + |Wx| + |Wy|) c + 2^-25."""
    from mmee import synth
    from mmee.config import ExitConfig, ModelDims
    from mmee.model import B200EEForSequenceClassification
    from oracle import port

    dims = {"tiny": ModelDims.tiny(layers=1), "base": ModelDims.base(layers=1), "large": ModelDims.large(layers=1),
            "h384": ModelDims(hidden=384, heads=6, inter=768, coord=64, shape=64, layers=1, vocab=1000)}[case]
    ee = ExitConfig.from_dict(dict(exits=["text_visual_concat", 1], encoder_layer_strategy="ramp",
                                   inference_strategy="max_confidence"))
    sd = synth.make_state_dict(dims, ee, seed=17)
    g = torch.Generator().manual_seed(23)
    for k in ("rel_pos_bias", "rel_pos_x_bias", "rel_pos_y_bias"):
        key = f"layoutlmv3.encoder.{k}.weight"
        sd[key] = torch.randn(sd[key].shape, generator=g)
    n = 4
    docs = synth.make_docs(dims, n, seed=29, pad=True)
    T = dims.n_text
    x0 = torch.randint(0, 1001, (n, T), generator=g)               # the bias reads x0 and y1
    y1 = torch.randint(0, 1001, (n, T), generator=g)
    docs["bbox"] = torch.stack([x0, y1 // 2, (x0 + 1000) // 2, y1], -1)
    docs["attention_mask"][2, 0] = 0                                   # masked CLS (kept as a row, masked as a key)
    model = B200EEForSequenceClassification(dims, ee, sd, device=0, max_batch=n, dtype=dtype)
    model.forward(**{k: v.cuda() for k, v in docs.items()})
    torch.cuda.synchronize()
    S, h = dims.seq, dims.heads
    pitch = (S + 63) // 64 * 64
    count = n * h * S * pitch
    got = model.debug_read("BIAS", np.float16, count).reshape(n, h, S, pitch).astype(np.float64)
    if dtype == "fp32":
        lo = model.debug_read("BIASlo", np.float16, count).reshape(n, h, S, pitch).astype(np.float64)
    model.close()

    sd64 = {k: v.double() for k, v in sd.items()}
    c = LOG2E / 8.0
    want = port.attention_bias(sd64, dims, docs["bbox"]).numpy() * c
    sd_xy = dict(sd64)
    sd_xy["layoutlmv3.encoder.rel_pos_bias.weight"] = torch.zeros_like(sd64["layoutlmv3.encoder.rel_pos_bias.weight"])
    txy = np.abs(port.attention_bias(sd_xy, dims, docs["bbox"]).numpy()) * c
    sd_abs = {k: v.abs() for k, v in sd64.items()}
    tabs = port.attention_bias(sd_abs, dims, docs["bbox"]).numpy() * c
    worst = 0.0
    for d in range(n):
        mask = docs["attention_mask"][d].numpy()
        kept = [t for t in range(T) if mask[t] != 0 or t == 0] + list(range(T, S))
        L = len(kept)
        key_masked = np.array([t < T and mask[t] == 0 for t in kept])
        ix = np.ix_(range(h), kept, kept)
        w, wxy, wabs = want[d][ix], txy[d][ix], tabs[d][ix]
        gd = got[d, :, :L, :]
        assert (gd[:, :, L:] == MASKED).all(), f"document {d}: pitch columns >= the row count are not masked"
        assert (gd[:, :, :L][:, :, key_masked] == MASKED).all(), f"document {d}: a masked key is not masked"
        live = ~key_masked
        gv = gd[:, :, :L][:, :, live]
        if dtype == "fp32":
            gv = gv + lo[d, :, :L, :L][:, :, live]
            bound = 2.0 ** -22 * np.abs(w[:, :, live]) * 1.01 + 5 * U_FP32 * wabs[:, :, live] + 2.0 ** -25
        else:
            bound = (U_FP16 * (np.abs(w[:, :, live]) + wxy[:, :, live]) + 5 * U_FP32 * wabs[:, :, live] + U_FP32) * 1.01
        ratio = np.abs(gv - w[:, :, live]) / bound
        if ratio.max() > 1.0:
            hh, i, j = np.unravel_index(np.argmax(ratio), ratio.shape)
            pytest.fail(f"{case} [{dtype}] document {d} head {hh} query row {i} key {np.flatnonzero(live)[j]}: "
                        f"got {gv[hh, i, j]:.6g} want {w[:, :, live][hh, i, j]:.6g} (ratio {ratio.max():.3g})")
        worst = max(worst, float(ratio.max()))
    print(f"bias {case} [{dtype}]: worst |err| / bound = {worst:.3f}")
