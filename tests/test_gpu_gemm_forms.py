"""The tcgen05 GEMM family (csrc/gemm_sm100.cuh, host side csrc/gemm.cu) checked kernel by kernel against fp64.

Every case calls one entry point (``vqa_b200_gemm``, ``vqa_b200_gemm_batched``, ``vqa_b200_mfb_fused``) directly, with
tails in M, N and K, and compares each output element with an fp64 reference computed on the GPU from exactly the bf16
(or fp32) values the kernel reads.  The only legitimate differences are then fp32 rounding in the accumulation and in
the epilogue, and each element is held to a bound derived from them (u = 2^-24, the fp32 unit roundoff):

    |C - C64| <= 4·K·u·(|A|·|B|^T)[m, n] + eps_epi

The first term bounds any fp32 summation order of K products, with 2x to spare for truncating adders.  ``eps_epi``
follows the epilogue step by step (``_rnd``, ``_store_bound``): every fp32 operation adds at most u·|its result|, tanhf at most 2 ulp
(4u·|tanh|), a bf16 store 2^-8·|value|, and every fp32 atomic add of a split-K slice u·(|prefill| + |A|·|B|^T).
A dropped or doubled 64-wide k-block, or a row, column or group written to the wrong place, is an error of the size
of the products themselves and exceeds the bound many times over at these shapes.

Outputs live inside larger buffers filled with a NaN sentinel (extra rows, ld > N, gaps between batch entries); every
element outside the logical window must keep its sentinel bits.  Operand padding is NaN too, so a read past K or past
the rows poisons the result.  Accumulating outputs (accumulate mode, ``dot_out``, ``ssq``) start from random values
and must equal prefill + product.

``_select_gemm`` / ``_select_mfb`` mirror the instantiation choice of gemm.cu (tile width, CTA pairs, split-K scheme).
Shapes whose form depends on the SM count are derived from it, and ``test_every_instance_launches`` checks under
torch.profiler that each case launched the instance the mirror names and that the cases together launch all nine.
The worst error-to-bound ratio of each case family goes to ``_parity_util.record``.
"""
import os
import re
import zlib

import pytest
import torch

from _parity_util import record

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U = 2.0 ** -24             # fp32 unit roundoff (round to nearest)
U16 = 2.0 ** -8            # bf16 unit roundoff
K_MAJOR, MN_MAJOR = 0, 1
F32, BF16 = 0, 1
EALIGN = -2
BLOCK_K = 64


def _cdiv(a, b):
    return -(-a // b)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ----------------------------------------------------------------------------------------------------------------------
# mirror of the launch-form selection in csrc/gemm.cu
# ----------------------------------------------------------------------------------------------------------------------
def _use_cta2(M, N, K, batch):
    try:
        forced = int(os.environ.get("VQA_B200_CTA2", "-1"))
    except ValueError:
        forced = 0
    if forced == 0:
        return False
    if forced == 1:
        return batch == 1 and M >= 256
    return batch == 1 and M >= 2048 and N >= 240 and M * N * K >= 1e10


def _select_gemm(M, N, K, batch, accumulate, k_split, sms):
    """(kernel instance, k_split, full_units, k_blocks) that gemm_impl launches for this problem."""
    bn = 256 if N >= 256 and batch * _cdiv(M, 128) * _cdiv(N, 256) >= sms else 128
    cta2 = bn == 256 and _use_cta2(M, N, K, batch)
    tiles = batch * _cdiv(M, 256 if cta2 else 128) * _cdiv(N, bn)
    k_blocks = _cdiv(K, BLOCK_K)
    workers = sms // 2 if cta2 else sms
    ks, full = 1, 0
    if accumulate:
        ks = k_split
        if ks <= 0:
            max_ks = max(k_blocks // 4, 1)
            if tiles < workers:
                best, ks = -1.0, 1
                for c in range(1, min(max_ks, 32) + 1):
                    units = tiles * c
                    score = units / (_cdiv(units, workers) * workers) - 0.004 * (c - 1)
                    if score > best + 1e-9:
                        best, ks = score, c
            else:
                tail = tiles % workers
                if tail:
                    full = tiles - tail
                    ks = max(min(workers // tail, max_ks), 1)
        ks = min(ks, k_blocks)
    kern = "gemm_tcgen05_kernel<%d, %d, %s, false>" % (bn, int(bool(accumulate)), str(cta2).lower())
    return kern, ks, full, k_blocks


def _select_mfb(M, N, K, seg_cols, extra, prod):
    extras = seg_cols not in (0, N) or extra or prod
    cta2 = not extras and _use_cta2(M, N, K, 1)
    return "gemm_tcgen05_kernel<240, 2, %s, %s>" % (str(cta2).lower(), str(bool(extras)).lower())


ALL_INSTANCES = {"gemm_tcgen05_kernel<%s>" % s for s in (
    "128, 0, false, false", "256, 0, false, false", "256, 0, true, false",
    "128, 1, false, false", "256, 1, false, false", "256, 1, true, false",
    "240, 2, false, false", "240, 2, true, false", "240, 2, false, true")}


# ----------------------------------------------------------------------------------------------------------------------
# operands, guarded outputs, comparison
# ----------------------------------------------------------------------------------------------------------------------
def _gen(name):
    return torch.Generator(device=DEV).manual_seed(zlib.crc32(name.encode()))


def _uniform(gen, shape, scale=1.0, dtype=torch.float32):
    return ((torch.rand(shape, generator=gen, device=DEV) * 2 - 1) * scale).to(dtype)


def _ld(n, dtype):
    """A row pitch > n that keeps rows 16-byte aligned."""
    step = 8 if dtype == torch.bfloat16 else 4
    return _cdiv(n, step) * step + step


def _operand(gen, batch, rows, K, layout, scale=1.0):
    """bf16 operand of logical shape [batch, rows, K] in `layout`, NaN in the row padding and between batch entries.
    Returns (buffer, ld, bstride, fp64 values [batch, rows, K])."""
    outer, inner = (rows, K) if layout == K_MAJOR else (K, rows)
    ld = _ld(inner, torch.bfloat16)
    buf = torch.full((batch, outer + 1, ld), float("nan"), device=DEV, dtype=torch.bfloat16)
    buf[:, :outer, :inner] = _uniform(gen, (batch, outer, inner), scale, torch.bfloat16)
    val = buf[:, :outer, :inner].double()
    if layout == MN_MAJOR:
        val = val.transpose(1, 2)
    return buf, ld, (outer + 1) * ld, val


class _Guarded:
    """A [batch, rows, cols] window (pitch ld, batch stride bstride) inside a larger sentinel-filled buffer."""

    def __init__(self, batch, rows, cols, ld, dtype, offset=0, bstride=None, extra_rows=3):
        self.shape = (batch, rows, cols)
        self.bstride = bstride if bstride is not None else (rows + extra_rows) * ld
        self.dtype, self.ld, self.offset = dtype, ld, offset
        n = offset + batch * max(self.bstride, rows * ld) + ld
        self.flat = torch.full((n,), float("nan"), device=DEV, dtype=dtype)
        self.win = torch.zeros(n, device=DEV, dtype=torch.bool)
        self._view(self.win).fill_(True)
        self.sentinel = self.flat[:1].clone()
        self.t = self._view(self.flat)

    def _view(self, flat):
        return flat[self.offset:].as_strided(self.shape, (self.bstride, self.ld, 1))

    def check_guard(self, what):
        ib = torch.int16 if self.dtype == torch.bfloat16 else torch.int32
        outside = self.flat.view(ib)[~self.win]
        bad = outside != self.sentinel.view(ib)
        assert not bad.any(), "%s: %d element(s) outside the logical window were written, first at flat index %d" % (
            what, int(bad.sum()), int((~self.win).nonzero()[bad.nonzero()[0, 0]]))


_WORST = {}


def _compare(got, ref, bound, what, family):
    """Elementwise |got - ref| <= bound; records the worst ratio of the family (bf16 outputs apart: their store rounding
    alone can use up nearly all of the bound)."""
    if got.dtype == torch.bfloat16:
        family += "_bf16_out"
    err = (got.double() - ref).abs()
    ratio = torch.where(err == 0, torch.zeros_like(err), err / bound)
    worst = float(ratio.max())
    if not worst <= 1.0:                    # NaN fails too
        bad = ~(err <= bound)
        idx = bad.nonzero()
        raise AssertionError("%s: %d element(s) out of bound (worst ratio %s); first at %s: got %r ref %r bound %r" % (
            what, int(bad.sum()), worst, tuple(idx[0].tolist()), float(got.double()[tuple(idx[0])]),
            float(ref[tuple(idx[0])]), float(bound[tuple(idx[0])])))
    _WORST[family] = max(_WORST.get(family, 0.0), worst)
    record("test_gpu_gemm_forms", family, _WORST[family])
    return worst


def _rnd(r, e):
    """One fp32 operation whose exact result (on the computed operands) is within e of r: adds u·|result|."""
    return e + U * (r.abs() + e)


def _store_bound(r, e, dtype):
    return e + U16 * (r.abs() + e) if dtype == torch.bfloat16 else e


def _group_sum(x, rpg, groups):
    """[M, N] -> [groups]: sum over the rows of each group and over the columns."""
    idx = torch.arange(x.shape[0], device=DEV) // rpg
    return torch.zeros(groups, device=DEV, dtype=torch.float64).index_add_(0, idx, x.sum(1))


def _launch(name, args):
    from vqa_attention_networks_b200 import ops
    ops.launch_direct(name, args)
    torch.cuda.synchronize()


# ----------------------------------------------------------------------------------------------------------------------
# vqa_b200_gemm
# ----------------------------------------------------------------------------------------------------------------------
def _run_gemm(name, sms, M, N, K, a_layout=K_MAJOR, b_layout=K_MAJOR, c_dtype=torch.float32, ldc=None, offset=0,
              bias=False, row_scale=False, rpg=1, relu=False, accumulate=False, k_split=0, dot=False, split=None,
              expect=None, same_as_aligned=False):
    kern, ks, full, k_blocks = _select_gemm(M, N, K, 1, accumulate, k_split, sms)
    if expect is not None:
        assert kern == expect, "shape (%d, %d, %d) no longer selects %s but %s" % (M, N, K, expect, kern)
    if split == "uniform":
        assert full == 0 and ks > 1 and k_blocks % ks != 0, (ks, full, k_blocks)
    elif split == "tail":
        assert full > 0 and ks > 1, (ks, full)
    family = "gemm_accumulate" if accumulate else ("gemm_dot" if dot else "gemm_store")
    g = _gen(name)
    A, lda, _, a64 = _operand(g, 1, M, K, a_layout)
    B, ldb, _, b64 = _operand(g, 1, N, K, b_layout, scale=K ** -0.5)
    a64, b64 = a64[0], b64[0]
    acc64, absprod = a64 @ b64.t(), a64.abs() @ b64.abs().t()
    e = 4 * K * U * absprod
    groups = _cdiv(M, rpg)
    bias_t = _uniform(g, (N,)) if bias else None
    rs_t = _uniform(g, (groups,), 2.0) if row_scale else None
    ldc = ldc or _ld(N, c_dtype)
    C = _Guarded(1, M, N, ldc, c_dtype, offset)
    if accumulate:
        C.t.copy_(_uniform(g, (1, M, N)))
    pre = C.t[0].double()
    dw = dout = None
    if dot:
        ld_dot = _ld(N, torch.bfloat16)
        dw = torch.full((M + 1, ld_dot), float("nan"), device=DEV, dtype=torch.bfloat16)
        dw[:M, :N] = _uniform(g, (M, N), 1.0, torch.bfloat16)
        dout = _Guarded(1, 1, groups, groups, torch.float32)
        dout.t.copy_(_uniform(g, (1, 1, groups)))
        dpre = dout.t[0, 0].double()

    args = [A, a_layout, lda, B, b_layout, ldb, C.t, BF16 if c_dtype == torch.bfloat16 else F32, ldc, M, N, K,
            bias_t, rs_t, rpg, int(relu), int(accumulate), k_split, dw, dw.stride(0) if dot else 0,
            dout.t if dot else None]
    _launch("vqa_b200_gemm", args)
    C.check_guard(name + " C")

    if accumulate:
        ref = pre + acc64
        bound = e + ks * U * (pre.abs() + absprod + e)       # one fp32 atomic add per k-slice
    else:
        r, bnd = acc64, e
        rs_rows = rs_t.double()[torch.arange(M, device=DEV) // rpg][:, None] if row_scale else None
        if rs_rows is not None:
            r, bnd = r * rs_rows, bnd * rs_rows.abs()
            bnd = _rnd(r, bnd)
        if bias:
            r = r + bias_t.double()
            bnd = _rnd(r, bnd)
        if relu:
            r = r.clamp_min(0)
        if dot:
            dwd = dw[:M, :N].double()
            terms = (r * dwd).abs() + bnd * dwd.abs()
            depth = N + 6 + 2 * rpg * _cdiv(N, 128)         # per-thread chain + warp tree + atomics per group
            dref = dpre + _group_sum(r * dwd, rpg, groups)
            dbound = _group_sum(bnd * dwd.abs(), rpg, groups) + depth * U * (_group_sum(terms, rpg, groups) + dpre.abs())
            dout.check_guard(name + " dot_out")
            _compare(dout.t[0, 0], dref, dbound, name + " dot_out", family)
        ref, bound = r, _store_bound(r, bnd, c_dtype)
    _compare(C.t[0], ref, bound, name + " C", family)
    if same_as_aligned:
        # the scalar store path must write what the vector path writes
        C2 = _Guarded(1, M, N, _ld(N, c_dtype), c_dtype)
        args[6], args[8] = C2.t, C2.ld
        _launch("vqa_b200_gemm", args)
        assert torch.equal(C.t, C2.t), name + ": scalar store path differs from the aligned vector path"
    return kern


def _n_wide(m_blocks, sms, rest):
    """N with enough 256-wide column blocks that m_blocks x them reach the SM count; `rest` columns in the last."""
    return 256 * (_cdiv(sms, m_blocks) - 1) + rest


GEMM_CASES = {
    # 1. BN = 128, the four layout pairs, and a bf16 C whose odd pitch forces the scalar bf16 stores
    "store128_kk": dict(M=300, N=200, K=200),
    "store128_kmn": dict(M=300, N=200, K=200, b_layout=MN_MAJOR),
    "store128_mnk": dict(M=300, N=200, K=200, a_layout=MN_MAJOR),
    "store128_mnmn": dict(M=300, N=200, K=200, a_layout=MN_MAJOR, b_layout=MN_MAJOR),
    "store128_bf16_ldc_odd": dict(M=300, N=200, K=200, c_dtype=torch.bfloat16, ldc=203),
    # 2. the fast epilogue: bias, row scale, both with ReLU; groups straddling 32-row warps; N % 32 = 8 partial chunk
    "fast_bias": dict(M=300, N=200, K=200, bias=True),
    "fast_rowscale_rpg26": dict(M=300, N=200, K=200, row_scale=True, rpg=26),
    "fast_rowscale_rpg196": dict(M=300, N=200, K=200, row_scale=True, rpg=196),
    "fast_bias_rowscale_relu_rpg1": dict(M=300, N=200, K=200, bias=True, row_scale=True, rpg=1, relu=True),
    "fast_bias_rowscale_relu_rpg26_bf16": dict(M=300, N=200, K=200, bias=True, row_scale=True, rpg=26, relu=True,
                                               c_dtype=torch.bfloat16),
    "fast_bias_rowscale_relu_rpg196": dict(M=300, N=200, K=200, bias=True, row_scale=True, rpg=196, relu=True),
    # 3. dot_with / dot_out: mixed groups per warp (per-row atomics) and one group per warp
    "dot_rpg26": dict(M=300, N=200, K=200, bias=True, rpg=26, dot=True),
    "dot_rpg32": dict(M=300, N=200, K=200, bias=True, rpg=32, dot=True),
    # 4. vec_ok == 0: misaligned C base, odd fp32 pitch
    "scalar_c_offset1": dict(M=300, N=200, K=200, bias=True, offset=1, same_as_aligned=True),
    "scalar_ldc_odd": dict(M=300, N=200, K=200, bias=True, relu=True, ldc=203, same_as_aligned=True),
    # 5. 256-wide tiles without pairs (M < 2048)
    "store256": lambda s: dict(M=1900, N=256 * _cdiv(s, 15) + 40, K=200,
                               expect="gemm_tcgen05_kernel<256, 0, false, false>"),
    # 6. CTA pairs; M % 256 < 128 leaves the second CTA of the last pair without rows; the wgrad layout at pair size
    "store256_cta2": lambda s: dict(M=4200, N=_n_wide(33, s, 176), K=2100,
                                    expect="gemm_tcgen05_kernel<256, 0, true, false>"),
    "store256_cta2_mnmn": lambda s: dict(M=2300, N=_n_wide(18, s, 52), K=2200, a_layout=MN_MAJOR, b_layout=MN_MAJOR,
                                         expect="gemm_tcgen05_kernel<256, 0, true, false>"),
    # 7. - 11. accumulate mode
    "acc_uniform_split": dict(M=200, N=300, K=5000, accumulate=True, split="uniform",
                              expect="gemm_tcgen05_kernel<128, 1, false, false>"),
    "acc_tail_split": lambda s: dict(M=2500, N=128 * (s // 20) + 104, K=1000, accumulate=True, split="tail",
                                     expect="gemm_tcgen05_kernel<128, 1, false, false>"),
    "acc_ksplit3": dict(M=300, N=200, K=1000, accumulate=True, k_split=3),
    "acc_ksplit_clamped": dict(M=300, N=200, K=1000, accumulate=True, k_split=1000),
    "acc256_tail_split": lambda s: dict(M=1900, N=256 * _cdiv(s, 15) + 40, K=1100, accumulate=True, split="tail",
                                        expect="gemm_tcgen05_kernel<256, 1, false, false>"),
    "acc256_cta2_tail_split": lambda s: dict(M=4200, N=_n_wide(33, s, 176), K=2100, accumulate=True, split="tail",
                                             expect="gemm_tcgen05_kernel<256, 1, true, false>"),
    "acc_ldc_odd": dict(M=300, N=200, K=1000, accumulate=True, ldc=203),
}


@pytest.mark.parametrize("case", list(GEMM_CASES))
def test_gemm(case):
    _gemm_case(case)


def _gemm_case(case):
    spec = GEMM_CASES[case]
    spec = spec(_sms()) if callable(spec) else spec
    return _run_gemm(case, _sms(), **spec)


# ----------------------------------------------------------------------------------------------------------------------
# vqa_b200_gemm_batched
# ----------------------------------------------------------------------------------------------------------------------
def _run_batched(name, sms, batch=5, M=196, N=26, K=512, ldc=32, a_layout=K_MAJOR, b_layout=K_MAJOR,
                 c_dtype=torch.float32, act=0, add=None, bias=False, drop_p=0.0, seed_dev=False, accumulate=False,
                 bstride0=False):
    from vqa_attention_networks_b200 import ops
    kern, ks, _, _ = _select_gemm(M, N, K, batch, accumulate, 0, sms)
    g = _gen(name)
    A, lda, abs_, a64 = _operand(g, batch, M, K, a_layout)
    B, ldb, bbs, b64 = _operand(g, batch, N, K, b_layout, scale=K ** -0.5)
    acc64, absprod = torch.bmm(a64, b64.transpose(1, 2)), torch.bmm(a64.abs(), b64.abs().transpose(1, 2))
    e = 4 * K * U * absprod
    cbs = 0 if bstride0 else (M + 3) * ldc
    C = _Guarded(batch, M, N, ldc, c_dtype, bstride=cbs if bstride0 else None)
    if accumulate:
        C.t.copy_(_uniform(g, (batch, M, N)))
    pre = C.t.double()
    bias_t = _uniform(g, (N,)) if bias else None
    add_g = None
    if add is not None:
        add_g = _Guarded(batch, M, N, ldc, add, bstride=C.bstride)
        add_g.t.copy_(_uniform(g, (batch, M, N), 1.0, add))
    seed, sd = 12345, (torch.tensor([7], device=DEV, dtype=torch.int32) if seed_dev else None)
    _launch("vqa_b200_gemm_batched", [
        A, a_layout, lda, 0 if bstride0 else abs_, B, b_layout, ldb, 0 if bstride0 else bbs, C.t,
        BF16 if c_dtype == torch.bfloat16 else F32, ldc, cbs, batch, M, N, K, bias_t, act,
        add_g.t if add is not None else None, BF16 if add == torch.bfloat16 else F32, drop_p, seed, sd, int(accumulate)])
    C.check_guard(name + " C")
    if accumulate:
        ref, bound = pre + acc64, e + ks * U * (pre.abs() + absprod + e)
    else:
        r, bnd = acc64, e
        if bias:
            r = r + bias_t.double()
            bnd = _rnd(r, bnd)
        if add is not None:
            r = r + add_g.t.double()
            bnd = _rnd(r, bnd)
        if act == 1:
            r = r.clamp_min(0)
        elif act == 2:
            r = torch.tanh(r)
            bnd = bnd + 4 * U * r.abs()                     # tanh is 1-Lipschitz; tanhf is within 2 ulp
        if drop_p > 0:
            # the epilogue hashes row bz * M + m
            mask = ops.dropout_mask(batch * M, N, drop_p, seed, DEV, sd).double().view(batch, M, N)
            r = r * mask
            bnd = _rnd(r, bnd * mask)
        ref, bound = r, _store_bound(r, bnd, c_dtype)
    _compare(C.t, ref, bound, name + " C", "gemm_batched")
    return kern


BATCHED_CASES = {
    "kk_act0_add_f32": dict(add=torch.float32),
    "mnmn_act1_add_bf16_bias": dict(a_layout=MN_MAJOR, b_layout=MN_MAJOR, act=1, add=torch.bfloat16, bias=True),
    "kmn_act2_bias": dict(b_layout=MN_MAJOR, act=2, bias=True),
    "mnk_act2_add_f32_bias_drop": dict(a_layout=MN_MAJOR, act=2, add=torch.float32, bias=True, drop_p=0.3),
    "kk_act0_drop": dict(drop_p=0.3),
    "kk_act1_bias_drop_seeddev": dict(act=1, bias=True, drop_p=0.3, seed_dev=True),
    "mnmn_act2_add_bf16_drop_seeddev_bf16c": dict(a_layout=MN_MAJOR, b_layout=MN_MAJOR, act=2, add=torch.bfloat16,
                                                  drop_p=0.3, seed_dev=True, c_dtype=torch.bfloat16),
    # 13. one batch entry with zero batch strides, and batched accumulate mode
    "batch1_bstride0": dict(batch=1, bias=True, act=1, bstride0=True),
    "accumulate": dict(batch=3, accumulate=True),
}


@pytest.mark.parametrize("case", list(BATCHED_CASES))
def test_gemm_batched(case):
    _run_batched(case, _sms(), **BATCHED_CASES[case])


# ----------------------------------------------------------------------------------------------------------------------
# vqa_b200_mfb_fused
# ----------------------------------------------------------------------------------------------------------------------
def _run_mfb(name, sms, M, N, K, rpg, y_dtype=torch.bfloat16, ldy=None, keep=None, drop_p=0.0, seg_cols=0,
             extra=False, prod=False, expect=None):
    """acc = X·W^T + b, keep = acc·mask, z = sum_5 keep·Q[m / rpg] (·extra), y = sign(z)·sqrt|z|, ssq[g, seg] += sum |z|.
    y is compared in the z domain (sign(y)·y^2 against z64): sqrt would turn rounding near 0 into a large relative
    error."""
    from vqa_attention_networks_b200 import ops
    kern = _select_mfb(M, N, K, seg_cols, extra, prod)
    if expect is not None:
        assert kern == expect, (kern, expect)
    g = _gen(name)
    X, ldx, _, x64 = _operand(g, 1, M, K, K_MAJOR)
    W, ldw, _, w64 = _operand(g, 1, N, K, K_MAJOR, scale=K ** -0.5)
    x64, w64 = x64[0], w64[0]
    groups, No = _cdiv(M, rpg), N // 5
    nseg = N // seg_cols if seg_cols else 1
    bias = _uniform(g, (N,), 0.5)
    ldq = N + 4
    Q = torch.full((groups + 1, ldq), float("nan"), device=DEV)
    Q[:groups, :N] = _uniform(g, (groups, N))
    E = None
    if extra:
        E = torch.full((groups + 1, ldq), float("nan"), device=DEV)
        E[:groups, :N] = _uniform(g, (groups, N))
    ldy = ldy or _ld(No, y_dtype)
    Y = _Guarded(1, M, No, ldy, y_dtype)
    ssq = _Guarded(1, 1, groups * nseg, groups * nseg, torch.float32)
    ssq.t.copy_(torch.rand((1, 1, groups * nseg), generator=g, device=DEV))
    ssq_pre = ssq.t[0, 0].double().view(groups, nseg)
    kp = _Guarded(1, M, N, N, keep, extra_rows=1) if keep is not None else None
    pr = _Guarded(1, M, N, N, torch.float32, extra_rows=1) if prod else None
    seed = 4242
    _launch("vqa_b200_mfb_fused", [
        X, ldx, W, ldw, bias, Q, ldq, rpg, Y.t, BF16 if y_dtype == torch.bfloat16 else F32, ldy, ssq.t,
        kp.t if kp else None, F32 if keep == torch.float32 else BF16, M, N, K, seg_cols, E, pr.t if pr else None,
        drop_p, seed, None])
    for buf, what in ((Y, "y"), (ssq, "ssq"), (kp, "keep"), (pr, "prod")):
        if buf is not None:
            buf.check_guard(name + " " + what)

    rows = torch.arange(M, device=DEV) // rpg
    r = x64 @ w64.t() + bias.double()
    e = _rnd(r, 4 * K * U * (x64.abs() @ w64.abs().t()))
    if drop_p > 0:
        mask = ops.dropout_mask(M, N, drop_p, seed, DEV).double()
        r = r * mask
        e = _rnd(r, e * mask)
    if kp is not None:
        _compare(kp.t[0], r, _store_bound(r, e, keep), name + " keep", "mfb_keep")
    q = Q[:groups, :N].double()[rows]
    eq = torch.zeros_like(q)
    if extra:
        q = q * E[:groups, :N].double()[rows]
        eq = U * q.abs()                                    # the rounded product Q·extra
    p64 = r * q
    ep = _rnd(p64, e * (q.abs() + eq) + r.abs() * eq)
    if pr is not None:
        _compare(pr.t[0], p64, ep, name + " prod", "mfb_prod")
    z = p64.view(M, No, 5).sum(2)
    ez = ep.view(M, No, 5).sum(2) + 4 * U * (p64.abs() + ep).view(M, No, 5).sum(2)    # four fp32 additions
    y = Y.t[0].double()
    rel = (1 + U) ** 2 * ((1 + U16) ** 2 if y_dtype == torch.bfloat16 else 1) - 1      # sqrtf (+ bf16 store), squared
    _compare(torch.sign(y) * y * y, z, ez + rel * (z.abs() + ez), name + " y",
             "mfb_y_bf16_out" if y_dtype == torch.bfloat16 else "mfb_y")
    seg_of = torch.arange(No, device=DEV) * 5 // (seg_cols or N)
    depth = No + 6 + 2 * rpg * _cdiv(N, 240)            # per-thread chain + warp tree + atomics per group and segment
    sref, sb, sabs = [], [], []
    for s in range(nseg):
        cols = seg_of == s
        sref.append(_group_sum(z.abs()[:, cols], rpg, groups))
        sb.append(_group_sum(ez[:, cols], rpg, groups))
        sabs.append(_group_sum((z.abs() + ez)[:, cols], rpg, groups))
    sref, sb, sabs = (torch.stack(t, 1) for t in (sref, sb, sabs))
    _compare(ssq.t[0, 0].view(groups, nseg), ssq_pre + sref, sb + depth * U * (sabs + ssq_pre), name + " ssq",
             "mfb_ssq")
    return kern


MFB_CASES = {
    # 14. grid form: groups of 196 rows straddle tiles, N % 40 = 20 leaves the last chunk half full
    "grid_ybf16_nokeep_p0": dict(M=588, N=1020, K=520, rpg=196),
    "grid_ybf16_keepbf16_p01": dict(M=588, N=1020, K=520, rpg=196, keep=torch.bfloat16, drop_p=0.1),
    "grid_yf32pad_keepf32_p01": dict(M=588, N=1020, K=520, rpg=196, y_dtype=torch.float32, ldy=212,
                                     keep=torch.float32, drop_p=0.1),
    "grid_yf32pad_keepbf16_p0": dict(M=588, N=1020, K=520, rpg=196, y_dtype=torch.float32, ldy=212,
                                     keep=torch.bfloat16),
    # 15. CTA pairs with a partial last group
    "cta2_keepbf16_p01": dict(M=4200, N=1000, K=2500, rpg=196, keep=torch.bfloat16, drop_p=0.1,
                              expect="gemm_tcgen05_kernel<240, 2, true, false>"),
    # 16. the vector-block form: two L2-norm segments per row, the cascade multiplier and the product output
    "mfbx_seg_extra_prod": dict(M=300, N=2000, K=520, rpg=1, seg_cols=1000, extra=True, prod=True,
                                keep=torch.bfloat16, drop_p=0.1, expect="gemm_tcgen05_kernel<240, 2, false, true>"),
}


@pytest.mark.parametrize("case", list(MFB_CASES))
def test_mfb_fused(case):
    _run_mfb(case, _sms(), **MFB_CASES[case])


# ----------------------------------------------------------------------------------------------------------------------
# the fp32-mode wrapper and argument checks
# ----------------------------------------------------------------------------------------------------------------------
def _run_fp32_mode(name, sms, layout, M=296, N=200, K=504):
    """ops.gemm(mode="fp32") runs one bf16 GEMM over 3K: hi·hi + hi·lo + lo·hi of the bf16 splits x = hi + lo + r.
    |x - hi| <= 2^-8|x| and |r| <= 2^-16|x|, so the dropped lo·lo, r·b and a·r terms are each <= 2^-16|a||b|: bound
    3·2^-16·(|A|·|B|^T) + 4·3K·u·(|A|·|B|^T) against fp64 of the unrounded fp32 inputs.  M, N and K are multiples of 8
    (not of the tile sizes): the split operands are packed without padding and their row pitch must stay 16-byte
    aligned."""
    from vqa_attention_networks_b200 import ops
    g = _gen(name)
    A = _uniform(g, (M, K) if layout == K_MAJOR else (K, M))
    B = _uniform(g, (N, K) if layout == K_MAJOR else (K, N), K ** -0.5)
    a64 = A.double() if layout == K_MAJOR else A.double().t()
    b64 = B.double() if layout == K_MAJOR else B.double().t()
    C = ops.gemm(A, layout, B, layout, "fp32")
    torch.cuda.synchronize()
    absprod = a64.abs() @ b64.abs().t()
    ref = a64 @ b64.t()
    _compare(C, ref, (3 * 2.0 ** -16 + 4 * 3 * K * U) * absprod, name, "fp32_mode")
    err = (C.double() - ref).abs()
    record("test_gpu_gemm_forms", "fp32_mode_max_err_over_absprod_" + name, float((err / absprod).max()))
    record("test_gpu_gemm_forms", "fp32_mode_rel_l2_" + name, float((C.double() - ref).norm() / ref.norm()))
    return _select_gemm(M, N, 3 * K, 1, False, 0, sms)[0]


def _run_misaligned(name, sms, how):
    """A misaligned A base or an lda that is not a multiple of 8 is refused before anything is launched."""
    M, N, K = 300, 200, 200
    g = _gen(name)
    B, ldb, _, _ = _operand(g, 1, N, K, K_MAJOR)
    flat = _uniform(g, ((M + 1) * (K + 8),), 1.0, torch.bfloat16)
    if how == "base":
        A, lda = flat[1:1 + M * (K + 8)], K + 8
    else:
        A, lda = flat, K + 3
    C = _Guarded(1, M, N, _ld(N, torch.float32), torch.float32)
    with pytest.raises(RuntimeError, match=r"status %d\).*16-byte aligned" % EALIGN):
        _launch("vqa_b200_gemm", [A, K_MAJOR, lda, B, K_MAJOR, ldb, C.t, F32, C.ld, M, N, K, None, None, 1, 0, 0, 0,
                                  None, 0, None])
    torch.cuda.synchronize()
    assert C.win.sum() > 0
    C.win.zero_()
    C.check_guard(name + " C")                        # nothing written anywhere
    return None


OTHER_CASES = {
    "fp32_mode_k_major": lambda s: _run_fp32_mode("fp32_mode_k_major", s, K_MAJOR),
    "fp32_mode_mn_major": lambda s: _run_fp32_mode("fp32_mode_mn_major", s, MN_MAJOR),
    "misaligned_a_base": lambda s: _run_misaligned("misaligned_a_base", s, "base"),
    "misaligned_lda": lambda s: _run_misaligned("misaligned_lda", s, "lda"),
}


@pytest.mark.parametrize("case", list(OTHER_CASES))
def test_wrappers_and_arguments(case):
    OTHER_CASES[case](_sms())


# ----------------------------------------------------------------------------------------------------------------------
# which instance ran
# ----------------------------------------------------------------------------------------------------------------------
def _all_cases():
    for c in GEMM_CASES:
        yield "gemm/" + c, lambda s, c=c: _gemm_case(c)
    for c, kw in BATCHED_CASES.items():
        yield "batched/" + c, lambda s, c=c, kw=kw: _run_batched(c, s, **kw)
    for c, kw in MFB_CASES.items():
        yield "mfb/" + c, lambda s, c=c, kw=kw: _run_mfb(c, s, **kw)
    for c, fn in OTHER_CASES.items():
        yield c, fn


def _launched_gemm_kernels(prof):
    names = set()
    for ev in prof.events():
        m = re.search(r"gemm_tcgen05_kernel<[^>]*>", ev.name)
        if m and ev.device_type == torch.autograd.DeviceType.CUDA:
            names.add(m.group(0))
    return names


def test_every_instance_launches():
    from torch.profiler import ProfilerActivity, profile
    sms = _sms()
    seen = set()
    for case, run in _all_cases():
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            expected = run(sms)
            torch.cuda.synchronize()
        launched = _launched_gemm_kernels(prof)
        assert launched == ({expected} if expected else set()), (case, launched, expected)
        seen |= launched
    assert seen == ALL_INSTANCES, "never launched: %s" % sorted(ALL_INSTANCES - seen)
