"""Grouped expert GEMMs on the hand-written tcgen05 kernel (csrc/gemm_sm100.cu) with autograd.

The reference runs its experts through ``torch.matmul`` -> cuBLAS (tutel/experts/ffn.py:114-118) followed by separate
bias / activation kernels.  Here forward, data-gradient and weight-gradient are all launches of one persistent
tcgen05/TMEM/TMA kernel; bias, ReLU and the ReLU gradient mask are fused into its epilogue, operands are consumed in
whatever major-ness they already have (no transposes are materialised).

Shapes (G = groups / local experts):
    ``x [G, T, K]``;  weights either ``[G, N, K]`` ("nk", like ``batched_fc1_w``) or ``[G, K, N]`` ("kn", like
    ``batched_fc2_w``);  result ``[G, T, N]``.
"""
from __future__ import annotations

from typing import Any, Optional

import torch

from . import backend

EPI_NONE, EPI_BIAS, EPI_BIAS_RELU, EPI_BIAS_GELU, EPI_BIAS_SILU, EPI_RELU_BWD = 0, 1, 2, 3, 4, 5
EPI_GLU, EPI_GLU_BWD, EPI_ADD, EPI_ACT_BWD = 6, 7, 8, 9
FWD_EPILOGUE = {'relu': EPI_BIAS_RELU, 'gelu': EPI_BIAS_GELU, 'silu': EPI_BIAS_SILU}
ACT_CODES = {'relu': 1, 'gelu': 2, 'silu': 3}


def _ok_stride(t: torch.Tensor) -> bool:
    es = t.element_size()
    return (t.stride(-1) == 1 and (t.stride(-2) * es) % 16 == 0 and (t.dim() < 3 or (t.stride(0) * es) % 16 == 0 or t.size(0) == 1)
            and t.data_ptr() % 16 == 0)


def _prep(t: torch.Tensor) -> torch.Tensor:
    if t.dim() == 2:
        t = t.unsqueeze(0)
    return t if _ok_stride(t) else t.contiguous()


def raw_gemm(a: torch.Tensor, b: torch.Tensor, *, a_mn: bool = False, b_mn: bool = False, epilogue: int = EPI_NONE,
             bias: Optional[torch.Tensor] = None, aux: Optional[torch.Tensor] = None,
             row_counts: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
             out_dtype: Optional[torch.dtype] = None, alpha: float = 1.0, b_group_div: int = 1, cta_group: int = 0,
             block_n: int = 0, d_ptr_table: int = 0, signal_ptr_table: int = 0, wait_flags: int = 0,
             wait_rows_per_flag: int = 0, wait_flags_per_group: int = 0, wait_target: int = 0,
             max_ctas: int = 0, group_rot: int = 0, group_mod: int = 1, scale_a: Optional[torch.Tensor] = None,
             scale_b: Optional[torch.Tensor] = None, colsum: Optional[torch.Tensor] = None,
             d2: Optional[torch.Tensor] = None, act: int = 0) -> torch.Tensor:
    """D[g] = epilogue(A[g] @ B[g // b_group_div]).

    ``a``: ``[G, M, K]`` (or ``[G, K, M]`` when ``a_mn``);  ``b``: ``[Gb, N, K]`` (or ``[Gb, K, N]`` when ``b_mn``).
    """
    C = backend.require_ext()
    a, b = _prep(a), _prep(b)
    G = a.size(0)
    M = a.size(2) if a_mn else a.size(1)
    N = b.size(2) if b_mn else b.size(1)
    if out is None:
        if out_dtype is None:
            out_dtype = a.dtype if a.element_size() > 1 else torch.bfloat16
        out = torch.empty([G, M, N], dtype=out_dtype, device=a.device)
    d = out if out.dim() == 3 else out.unsqueeze(0)
    if bias is not None:
        bias = bias.reshape(b.size(0), N)
        want = a.dtype if a.element_size() > 1 else out.dtype
        if bias.stride(-1) != 1 or bias.dtype != want:
            bias = bias.to(want).contiguous()
    if aux is not None:
        aux = _prep(aux)
    backend.count_launch()
    C.gemm_ex(a, b, d, a_mn, b_mn, epilogue, bias, aux, row_counts, float(alpha), int(b_group_div), int(cta_group),
              int(block_n), int(d_ptr_table), int(signal_ptr_table), int(wait_flags), int(wait_rows_per_flag),
              int(wait_flags_per_group), int(wait_target), int(max_ctas), int(group_rot), int(group_mod), scale_a, scale_b, colsum,
              d2, int(act))
    return out


def column_sums(t: torch.Tensor) -> torch.Tensor:
    """``[G, T, N] -> [G, N]`` sums over the rows of every group (bias gradients) in t's dtype with fp32 accumulation:
    a bandwidth-bound kernel (csrc/gate_route.cu) instead of torch's strided reduction + cast."""
    if t.is_cuda and t.dim() == 3 and t.dtype in (torch.float32, torch.float16, torch.bfloat16) and backend.has_cuda_ext():
        es = t.element_size()
        if (t.stride(2) == 1 and t.data_ptr() % 16 == 0 and (t.stride(1) * es) % 16 == 0 and (t.stride(0) * es) % 16 == 0 and
                (t.size(2) * es) % 16 == 0):
            backend.count_launch()
            return backend.require_ext().grouped_colsum(t)
    return t.sum(dim=1, dtype=torch.float32).to(t.dtype)


def _aligned(*dims: int) -> bool:
    return all(d % 8 == 0 for d in dims)


def can_use_tcgen05(x: torch.Tensor, w: torch.Tensor) -> bool:
    return (backend.use_tcgen05(x) and w.dtype == x.dtype and w.is_cuda and x.dim() == 3 and w.dim() == 3 and
            _aligned(x.size(-1), w.size(-1), w.size(-2)))


class GroupedLinear(torch.autograd.Function):
    """y[g] = x[g] @ W[g]^T (+ b)  for ``w_layout == 'nk'``  or  x[g] @ W[g] (+ b)  for ``'kn'`` - all on tcgen05."""

    @staticmethod
    def forward(ctx: Any, x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], w_layout: str,
                row_counts: Optional[torch.Tensor], fp8: bool = False):
        ctx.w_layout = w_layout
        ctx.has_bias = bias is not None
        ctx.save_for_backward(x, w)
        ctx.row_counts = row_counts
        if fp8:     # e4m3 forward, bf16/fp16 backward on the master weights
            return fp8_linear(x, w, bias, w_layout, None, row_counts)
        return raw_gemm(x, w, b_mn=(w_layout == 'kn'), epilogue=EPI_BIAS if bias is not None else EPI_NONE, bias=bias,
                        row_counts=row_counts)

    @staticmethod
    def backward(ctx: Any, dy: torch.Tensor):
        x, w = ctx.saved_tensors
        dy = dy if _ok_stride(dy) else dy.contiguous()
        kn = ctx.w_layout == 'kn'
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            # dx[T,K] = dy[T,N] @ W (nk: W is [N,K] i.e. "kn" for this product; kn: W is [K,N] i.e. "nk")
            dx = raw_gemm(dy, w, b_mn=not kn, row_counts=ctx.row_counts)
            if ctx.row_counts is not None:
                dx = _zero_tail(dx, ctx.row_counts)
        if ctx.needs_input_grad[1]:
            if kn:   # dW[K,N] = x^T[K,T] @ dy[T,N]
                dw = raw_gemm(x, dy, a_mn=True, b_mn=True)
            else:    # dW[N,K] = dy^T[N,T] @ x[T,K]
                dw = raw_gemm(dy, x, a_mn=True, b_mn=True)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = column_sums(dy)
        return dx, dw, db, None, None, None


def _zero_tail(t: torch.Tensor, counts: torch.Tensor) -> torch.Tensor:
    rows = torch.arange(t.size(1), device=t.device).view(1, -1, 1)
    return torch.where(rows < counts.view(-1, 1, 1), t, torch.zeros((), dtype=t.dtype, device=t.device))


def grouped_linear(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, w_layout: str = 'nk',
                   row_counts: Optional[torch.Tensor] = None, fp8: bool = False) -> torch.Tensor:
    """Batched per-expert linear layer; falls back to ``torch.matmul`` for dtypes/devices the kernel does not cover."""
    if can_use_tcgen05(x, w) and (bias is None or bias.numel() == w.size(0) * (w.size(1) if w_layout == 'nk' else w.size(2))):
        b = None if bias is None else bias.reshape(w.size(0), -1)
        fp8 = fp8 and x.size(-1) % 16 == 0
        return GroupedLinear.apply(x, w, b, w_layout, row_counts, fp8)
    y = torch.matmul(x, w.transpose(1, 2) if w_layout == 'nk' else w)
    if bias is not None:
        y = y + bias.reshape(w.size(0), 1, -1)
    return y


class FusedReluFFN(torch.autograd.Function):
    """y = act(x @ W1^T + b1) @ W2 + b2 with 2 forward and 4 backward launches, nothing else (act: relu / gelu / silu).

    ``w1 [G, H, M]`` (nk), ``w2 [G, H, Mout]`` (kn) - the reference's ``batched_fc1_w`` / ``batched_fc2_w`` layout.
    ReLU keeps only the post-activation tensor (its sign doubles as the gradient mask fused into the dgrad epilogue);
    GELU / SiLU also store the pre-activation from the same epilogue and apply act'(pre) in the dgrad epilogue.
    """

    @staticmethod
    def forward(ctx: Any, x, w1, b1, w2, b2, row_counts, act_kind='relu'):
        need_grad = any(ctx.needs_input_grad[:5])
        pre = None
        if act_kind == 'relu':
            act = raw_gemm(x, w1, epilogue=EPI_BIAS_RELU, bias=b1, row_counts=row_counts)
        else:
            pre = torch.empty([x.size(0), x.size(1), w1.size(1)], dtype=x.dtype, device=x.device) if need_grad else None
            act = raw_gemm(x, w1, epilogue=FWD_EPILOGUE[act_kind], bias=b1, row_counts=row_counts, d2=pre)
        y = raw_gemm(act, w2, b_mn=True, epilogue=EPI_BIAS if b2 is not None else EPI_NONE, bias=b2,
                     row_counts=row_counts)
        ctx.save_for_backward(x, w1, w2, act, pre)
        ctx.has_b1, ctx.has_b2, ctx.act_kind = b1 is not None, b2 is not None, act_kind
        ctx.row_counts = row_counts
        return y

    @staticmethod
    def backward(ctx: Any, dy: torch.Tensor):
        x, w1, w2, act, pre = ctx.saved_tensors
        rc = ctx.row_counts
        dy = dy if _ok_stride(dy) else dy.contiguous()
        if rc is not None:
            dy = _zero_tail(dy, rc)
        # dh[T,H] = (dy[T,Mout] @ W2^T) * act'(.)           W2 [H,Mout] is "nk" for this product
        want_db1 = ctx.has_b1 and ctx.needs_input_grad[2]
        db1_acc = torch.zeros([w1.size(0), w1.size(1)], dtype=torch.float32, device=dy.device) if want_db1 else None
        if ctx.act_kind == 'relu':
            dh = raw_gemm(dy, w2, epilogue=EPI_RELU_BWD, aux=act, row_counts=rc, colsum=db1_acc)   # db1 fused in the epilogue
        else:
            dh = raw_gemm(dy, w2, epilogue=EPI_ACT_BWD, aux=pre, act=ACT_CODES[ctx.act_kind], row_counts=rc, colsum=db1_acc)
        if rc is not None:
            dh = _zero_tail(dh, rc)
            act = _zero_tail(act, rc)
        dw2 = raw_gemm(act, dy, a_mn=True, b_mn=True) if ctx.needs_input_grad[3] else None      # [H,Mout] = act^T @ dy
        db2 = column_sums(dy) if ctx.has_b2 and ctx.needs_input_grad[4] else None
        dx = raw_gemm(dh, w1, b_mn=True, row_counts=rc) if ctx.needs_input_grad[0] else None    # [T,M] = dh @ W1
        if dx is not None and rc is not None:
            dx = _zero_tail(dx, rc)
        dw1 = raw_gemm(dh, x, a_mn=True, b_mn=True) if ctx.needs_input_grad[1] else None        # [H,M] = dh^T @ x
        db1 = db1_acc.to(dh.dtype) if want_db1 else None
        return dx, dw1, db1, dw2, db2, None, None


def fused_relu_ffn(x, w1, b1, w2, b2, row_counts=None, act_kind='relu'):
    b1 = None if b1 is None else b1.reshape(w1.size(0), -1)
    b2 = None if b2 is None else b2.reshape(w2.size(0), -1)
    return FusedReluFFN.apply(x, w1, b1, w2, b2, row_counts, act_kind)


fused_act_ffn = fused_relu_ffn


_PROBE = None


def classify_activation(fn) -> Optional[str]:
    """Recognise ReLU / SiLU / GELU (also when wrapped in a lambda, as the reference examples do) by probing once."""
    global _PROBE
    if fn is None or fn is torch.relu or fn is torch.nn.functional.relu or isinstance(fn, torch.nn.ReLU):
        return 'relu'
    if fn is torch.nn.functional.silu or isinstance(fn, torch.nn.SiLU):
        return 'silu'
    if isinstance(fn, str):
        return fn
    cached = getattr(fn, '_tutel_b200_kind', None)
    if cached is not None:
        return cached or None
    if _PROBE is None:
        # dense around zero plus magnitudes up to 3e4 (fp16 range): clamped look-alikes (relu6, hardtanh, clamp(0, c)) differ
        # from ReLU only on large inputs and must not be classified as ReLU
        big = torch.logspace(0.7, 4.5, 64)
        _PROBE = torch.cat([torch.linspace(-4.0, 4.0, 257), big, -big])
    kind = ''
    try:
        with torch.no_grad():
            a, b = fn(_PROBE.clone()), fn(_PROBE.clone())
        if isinstance(a, torch.Tensor) and a.shape == _PROBE.shape and torch.equal(a, b):
            if torch.equal(a, torch.relu(_PROBE)):
                kind = 'relu'
            elif torch.allclose(a, torch.nn.functional.silu(_PROBE), atol=1e-6, rtol=1e-6):
                kind = 'silu'
            elif torch.allclose(a, torch.nn.functional.gelu(_PROBE), atol=1e-6, rtol=1e-6):
                kind = 'gelu'
    except Exception:  # noqa
        kind = ''
    try:
        fn._tutel_b200_kind = kind
    except Exception:  # noqa
        pass
    return kind or None


def can_use_skinny(x: torch.Tensor, w: torch.Tensor) -> bool:
    """Few rows per expert (decoder inference / dropless routing) on CUDA, no autograd: use the weight-streaming kernel."""
    return (x.is_cuda and x.dim() == 3 and x.size(1) <= 64 and x.dtype == w.dtype and not torch.is_grad_enabled() and
            x.dtype in (torch.float32, torch.float16, torch.bfloat16) and backend.has_cuda_ext())


_SKINNY_ACTS = {'relu': 1, 'gelu': 2, 'silu': 3}


def can_use_skinny_ffn(x: torch.Tensor, w1: torch.Tensor, w2: torch.Tensor, act_kind) -> bool:
    """Both expert layers in one weight-streaming launch (csrc/skinny_gemm.cu: skinny_ffn_kernel)."""
    v = 16 // x.element_size()
    return (can_use_skinny(x, w1) and act_kind in _SKINNY_ACTS and w1.dtype == w2.dtype and w1.size(2) == x.size(2) and
            w2.size(1) == w1.size(1) and x.size(2) % v == 0 and w2.size(2) % v == 0 and 16 * x.size(2) + 1024 <= 100 * 1024)


def skinny_ffn(x, w1, b1, w2, b2, row_counts, act_kind):
    """y[g, r] = act(x[g, r] @ W1[g]^T + b1[g]) @ W2[g] + b2[g] for r < row_counts[g]; other rows are zero."""
    backend.count_launch(2)          # zero-fill of the fp32 accumulator + the kernel
    b1 = None if b1 is None else b1.reshape(w1.size(0), -1).contiguous()
    b2 = None if b2 is None else b2.reshape(w2.size(0), -1).contiguous()
    y = backend.require_ext().skinny_ffn(x.contiguous(), w1.contiguous(), b1, w2.contiguous(), b2, row_counts,
                                         _SKINNY_ACTS[act_kind])
    return y if y.dtype == x.dtype else y.to(x.dtype)


def skinny_linear(x, w, bias, w_layout, row_counts, relu=False):
    """y[g, r] = act(x[g, r] @ W[g] + b[g]) for r < row_counts[g] (csrc/skinny_gemm.cu); other rows are zero."""
    backend.count_launch()
    b = None if bias is None else bias.reshape(w.size(0), -1).contiguous()
    return backend.require_ext().skinny_gemm(x.contiguous(), w.contiguous(), b, row_counts, w_layout == 'kn', relu)


# ----------------------------------------------------------------------------------------------------------------
# fp8 (e4m3) expert GEMMs: per-row (per-token) activation scales x per-output-channel weight scales, applied in the
# epilogue.  Forward AND data-gradient GEMMs run at the fp8 tensor-core rate; weight gradients stay in 16 bit (their
# reduction dimension is the token axis, along which the row scales vary).
# ----------------------------------------------------------------------------------------------------------------
_FP8_WEIGHT_CACHE = {}
_FP8_STEP = [0]          # bumped by every optimizer.step() in the process: quantised weights are valid for one step
_FP8_HOOKED = [False]


def invalidate_fp8_cache():
    """Force re-quantisation of all cached fp8 weights (call after changing weights outside an optimizer step)."""
    _FP8_STEP[0] += 1


def _ensure_step_hook():
    if _FP8_HOOKED[0]:
        return
    _FP8_HOOKED[0] = True
    try:
        from torch.optim.optimizer import register_optimizer_step_post_hook
        register_optimizer_step_post_hook(lambda *_: invalidate_fp8_cache())
    except Exception:  # noqa - very old torch: fall back to the version counter alone
        pass


def quantize_rows(x: torch.Tensor):
    """(q e4m3 [.., K], scale fp32 [..]) with one scale per row (native kernel)."""
    backend.count_launch()
    return backend.require_ext().quantize_rows(x.contiguous())


def fp8_operand(w: torch.Tensor, transpose: bool):
    """e4m3 copy of ``w [G, R, K]`` (or of ``w^T`` when ``transpose``) quantised along its last dim with one scale per
    row - the K-major B operand of ``A @ B`` - plus the scales ``[G, R]``.  Cached until the next optimizer step (an
    optimizer-step hook invalidates the cache: in-place ``.data`` updates do not bump a tensor's version counter) or
    until the tensor's version changes."""
    import weakref
    _ensure_step_hook()
    anchor = w._base if w._base is not None else w      # views of a parameter are re-created every forward
    key = (id(anchor), w.data_ptr(), bool(transpose), tuple(w.shape), tuple(w.stride()))
    stamp = (w._version, _FP8_STEP[0])
    hit = _FP8_WEIGHT_CACHE.get(key)
    if hit is not None and hit[0] == stamp and hit[3]() is anchor:
        return hit[1], hit[2]
    src = w.detach()
    if transpose and src.dim() == 3 and src.is_contiguous() and src.element_size() == 2 and src.size(1) % 128 == 0 and src.size(2) % 64 == 0:
        backend.count_launch(2)        # column |max| + transposing quantisation: no 16-bit transpose copy
        q, s = backend.require_ext().quantize_transpose(src)
    else:
        q, s = quantize_rows((src.transpose(1, 2) if transpose else src).contiguous())
    if len(_FP8_WEIGHT_CACHE) > 256:
        for k in [k for k, v in _FP8_WEIGHT_CACHE.items() if v[3]() is None]:
            del _FP8_WEIGHT_CACHE[k]
    _FP8_WEIGHT_CACHE[key] = (stamp, q, s, weakref.ref(anchor))
    return q, s


def fp8_weight(w: torch.Tensor, layout: str):
    """K-major e4m3 copy [G, N, K] + per-output-channel scales [G, N] of a weight stored 'nk' ([G, N, K]) or 'kn'."""
    return fp8_operand(w, transpose=(layout == 'kn'))


def fp8_linear(x: torch.Tensor, w: torch.Tensor, bias, w_layout: str, epilogue: int = None, row_counts=None):
    """y = act(x @ W + b) with both operands quantised to e4m3 on the fly; result in x.dtype."""
    xq, sx = quantize_rows(x)
    wq, sw = fp8_weight(w, w_layout)
    if epilogue is None:
        epilogue = EPI_BIAS if bias is not None else EPI_NONE
    return raw_gemm(xq, wq, epilogue=epilogue, bias=bias, row_counts=row_counts, out_dtype=x.dtype, scale_a=sx, scale_b=sw)


class FusedReluFFNFp8(torch.autograd.Function):
    """ReLU FFN with e4m3 forward and data-gradient GEMMs (2x tensor-core rate), 16-bit weight-gradient GEMMs on the
    master weights.  Quantised weight copies (both orientations) are made once per optimizer step."""

    @staticmethod
    def forward(ctx: Any, x, w1, b1, w2, b2, row_counts):
        act = fp8_linear(x, w1, b1, 'nk', EPI_BIAS_RELU, row_counts)
        y = fp8_linear(act, w2, b2, 'kn', None, row_counts)
        ctx.save_for_backward(x, w1, w2, act)
        ctx.has_b1, ctx.has_b2 = b1 is not None, b2 is not None
        ctx.row_counts = row_counts
        return y

    @staticmethod
    def backward(ctx: Any, dy: torch.Tensor):
        x, w1, w2, act = ctx.saved_tensors
        rc = ctx.row_counts
        dy = dy if _ok_stride(dy) else dy.contiguous()
        if rc is not None:
            dy = _zero_tail(dy, rc)
        want_db1 = ctx.has_b1 and ctx.needs_input_grad[2]
        db1_acc = torch.zeros([w1.size(0), w1.size(1)], dtype=torch.float32, device=dy.device) if want_db1 else None
        dyq, sdy = quantize_rows(dy)
        w2q, s2 = fp8_operand(w2, transpose=False)             # dh = dy @ W2^T: W2 [H, Mout] is already K-major for it
        dh = raw_gemm(dyq, w2q, epilogue=EPI_RELU_BWD, aux=act, row_counts=rc, colsum=db1_acc, out_dtype=dy.dtype,
                      scale_a=sdy, scale_b=s2)
        if rc is not None:
            dh = _zero_tail(dh, rc)
            act = _zero_tail(act, rc)
        dw2 = raw_gemm(act, dy, a_mn=True, b_mn=True) if ctx.needs_input_grad[3] else None
        db2 = column_sums(dy) if ctx.has_b2 and ctx.needs_input_grad[4] else None
        dx = None
        if ctx.needs_input_grad[0]:
            dhq, sdh = quantize_rows(dh)
            w1q, s1 = fp8_operand(w1, transpose=True)           # dx = dh @ W1: needs W1^T [M, H] K-major
            dx = raw_gemm(dhq, w1q, row_counts=rc, out_dtype=dy.dtype, scale_a=sdh, scale_b=s1)
            if rc is not None:
                dx = _zero_tail(dx, rc)
        dw1 = raw_gemm(dh, x, a_mn=True, b_mn=True) if ctx.needs_input_grad[1] else None
        db1 = db1_acc.to(dh.dtype) if want_db1 else None
        return dx, dw1, db1, dw2, db2, None


def fused_relu_ffn_fp8(x, w1, b1, w2, b2, row_counts=None):
    b1 = None if b1 is None else b1.reshape(w1.size(0), -1)
    b2 = None if b2 is None else b2.reshape(w2.size(0), -1)
    return FusedReluFFNFp8.apply(x, w1, b1, w2, b2, row_counts)


def _glu_extra(kw):
    return (int(kw.get('b_group_div', 1)), int(kw.get('cta_group', 0)), int(kw.get('wait_flags', 0)),
            int(kw.get('wait_rows_per_flag', 0)), int(kw.get('wait_flags_per_group', 0)), int(kw.get('wait_target', 0)),
            int(kw.get('group_rot', 0)), int(kw.get('group_mod', 1)), int(kw.get('max_ctas', 0)))


def glu_gemm(a, b, b2, *, b_mn, act, save_pre=False, scale_a=None, scale_b=None, scale_b2=None, row_counts=None,
             out_dtype=None, **kw):
    """h = act(a @ B) * (a @ B2) in ONE tcgen05 launch (each CTA of a pair stages one of the two weight tiles; the
    gate/up halves meet in the TMEM accumulator).  ``save_pre`` also returns the pre-activations (g, u)."""
    C = backend.require_ext()
    a, b, b2 = _prep(a), _prep(b), _prep(b2)
    if b2.stride() != b.stride():
        b, b2 = b.contiguous(), b2.contiguous()
    N = b.size(2) if b_mn else b.size(1)
    dt = out_dtype or (a.dtype if a.element_size() > 1 else torch.bfloat16)
    h = torch.empty([a.size(0), a.size(1), N], dtype=dt, device=a.device)
    g, u = (torch.empty_like(h), torch.empty_like(h)) if save_pre else (None, None)
    backend.count_launch()
    C.gemm_glu(a, b, b2, h, g, u, None, None, b_mn, ACT_CODES[act], scale_a, scale_b, scale_b2, row_counts, *_glu_extra(kw))
    return h, g, u


def glu_gemm_bwd(dy, w, g, u, *, b_mn, act, row_counts=None, scale_a=None, scale_b=None, **kw):
    """(dg, du) for h = act(g) * u with dh = dy @ W formed in TMEM only (never written to memory); dy / W may be e4m3
    with per-row scales."""
    C = backend.require_ext()
    dy, w = _prep(dy), _prep(w)
    dg, du = torch.empty_like(g), torch.empty_like(g)
    backend.count_launch()
    C.gemm_glu(dy, w, None, dg, du, None, g, u, b_mn, ACT_CODES[act], scale_a, scale_b, None, row_counts, *_glu_extra(kw))
    return dg, du


class FusedGLUFFN(torch.autograd.Function):
    """y = (act(x @ W1) * (x @ W2)) @ W3 - the SwiGLU / "LLaMA" expert (reference: tutel/experts/llama_ffn.py:38-41,
    three cuBLAS GEMMs + activation + multiply, and their five autograd kernels in backward).

    Here: 2 launches forward (dual-B GLU GEMM, down projection), 4-6 backward (dh GEMM whose epilogue emits dg and du,
    three wgrads, optionally two dgrads with the add fused), no elementwise kernels at all.
    ``w1, w2: [G, M, H]``, ``w3: [G, H, Mout]`` (all "kn", the reference's parameter layout).
    """

    @staticmethod
    def forward(ctx: Any, x, w1, w2, w3, act: str, fp8: bool):
        need_grad = any(ctx.needs_input_grad[:4])
        if fp8:
            xq, sx = quantize_rows(x)
            (q1, s1), (q2, s2), (q3, s3) = fp8_weight(w1, 'kn'), fp8_weight(w2, 'kn'), fp8_weight(w3, 'kn')
            h, g, u = glu_gemm(xq, q1, q2, b_mn=False, act=act, save_pre=need_grad, scale_a=sx, scale_b=s1, scale_b2=s2,
                               out_dtype=x.dtype)
            hq, sh = quantize_rows(h)
            y = raw_gemm(hq, q3, out_dtype=x.dtype, scale_a=sh, scale_b=s3)
            ctx.fp8 = True
        else:
            h, g, u = glu_gemm(x, w1, w2, b_mn=True, act=act, save_pre=need_grad)
            y = raw_gemm(h, w3, b_mn=True)
        ctx.act = act
        if need_grad:
            ctx.save_for_backward(x, w1, w2, w3, g, u, h)
        return y

    @staticmethod
    def backward(ctx: Any, dy: torch.Tensor):
        x, w1, w2, w3, g, u, h = ctx.saved_tensors
        dy = dy if _ok_stride(dy) else dy.contiguous()
        if getattr(ctx, 'fp8', False):
            # e4m3 data-gradient GEMMs: dh = dy @ W3^T uses W3 as stored ([H, Mout] is K-major for it), dx uses W1 / W2 as stored
            dyq, sdy = quantize_rows(dy)
            q3, s3 = fp8_operand(w3, transpose=False)
            dg, du = glu_gemm_bwd(dyq, q3, g, u, b_mn=False, act=ctx.act, scale_a=sdy, scale_b=s3)
        else:
            dg, du = glu_gemm_bwd(dy, w3, g, u, b_mn=False, act=ctx.act)    # dh = dy @ W3^T (W3 [H,Mout] is "nk" here)
        dw3 = raw_gemm(h, dy, a_mn=True, b_mn=True) if ctx.needs_input_grad[3] else None   # [H,Mout] = h^T @ dy
        dw1 = raw_gemm(x, dg, a_mn=True, b_mn=True) if ctx.needs_input_grad[1] else None   # [M,H] = x^T @ dg
        dw2 = raw_gemm(x, du, a_mn=True, b_mn=True) if ctx.needs_input_grad[2] else None
        dx = None
        if ctx.needs_input_grad[0] and getattr(ctx, 'fp8', False):
            (dgq, sg), (duq, su) = quantize_rows(dg), quantize_rows(du)
            (q1, s1), (q2, s2) = fp8_operand(w1, transpose=False), fp8_operand(w2, transpose=False)   # [M, H]: K-major here
            dx = raw_gemm(dgq, q1, out_dtype=dy.dtype, scale_a=sg, scale_b=s1)
            dx = raw_gemm(duq, q2, epilogue=EPI_ADD, aux=dx, out_dtype=dy.dtype, scale_a=su, scale_b=s2)
        elif ctx.needs_input_grad[0]:
            dx = raw_gemm(dg, w1)                                            # [T,M] = dg @ W1^T
            dx = raw_gemm(du, w2, epilogue=EPI_ADD, aux=dx)                  # += du @ W2^T (add fused in the epilogue)
        return dx, dw1, dw2, dw3, None, None


def fused_glu_ffn(x, w1, w2, w3, act='silu', fp8=False):
    return FusedGLUFFN.apply(x, w1, w2, w3, act, fp8)
