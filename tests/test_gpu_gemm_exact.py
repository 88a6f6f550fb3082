"""Exact conformance of the tcgen05 grouped GEMM (csrc/gemm_sm100.cu) across its configurations.

A and B hold small integers (fp8 scales are powers of two) and every partial sum stays below 2^16, so the fp32
accumulation is exact in any order: the kernel must equal a float64 reference, rounded once to the output dtype, bit
for bit (`torch.equal`).  The GELU / SiLU epilogues evaluate erff / __expf / __fdividef in fp32, which are not correctly
rounded; their results are checked against an error bound instead (see `assert_matches`), and their saved
pre-activations exactly.

Outputs start as NaN, so an element the kernel never wrote cannot pass.  Operands, side inputs and outputs are also
passed as slices of wider and taller buffers (leading dimension > logical width, group stride > dense) whose margins
hold SENTINEL: a read of the margin changes the result, a write into it is caught directly.

Output paths: 16-bit local outputs leave through TMA tensor stores; with `row_counts` or a pointer table, 16-bit outputs
of the non-GLU epilogues leave through per-row bulk stores; fp32 outputs, and GLU outputs with `row_counts`, are stored
directly from registers.
"""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

EPI_NONE, EPI_BIAS, EPI_BIAS_RELU, EPI_BIAS_GELU, EPI_BIAS_SILU, EPI_RELU_BWD = 0, 1, 2, 3, 4, 5
EPI_GLU, EPI_GLU_BWD, EPI_ADD, EPI_ACT_BWD = 6, 7, 8, 9
RELU, GELU, SILU = 1, 2, 3
BF16, FP16, FP32 = torch.bfloat16, torch.float16, torch.float32
E4M3, E5M2 = torch.float8_e4m3fn, torch.float8_e5m2
SENTINEL = -96.0          # exactly representable in every operand and output dtype, e4m3 / e5m2 included
NAN = float('nan')
LAYOUTS = [(False, False), (False, True), (True, False), (True, True)]


@pytest.fixture(scope='module')
def C():
    from tutel_b200.ops import backend
    return backend.require_ext()


# ------------------------------------------------------------------------------------------------------------------
# raw bindings with keyword defaults
# ------------------------------------------------------------------------------------------------------------------
def gemm_ex(C, a, b, d, *, a_mn=False, b_mn=False, epi=EPI_NONE, bias=None, aux=None, counts=None, alpha=1.0, div=1, cg=0,
            bn=0, d_table=0, s_table=0, wait=None, max_ctas=0, rot=0, mod=1, sa=None, sb=None, colsum=None, d2=None, act=0):
    wf, wr, wpg, wt = wait if wait is not None else (0, 0, 0, 0)
    C.gemm_ex(a, b, d, a_mn, b_mn, epi, bias, aux, counts, float(alpha), div, cg, bn, d_table, s_table, wf, wr, wpg, wt,
              max_ctas, rot, mod, sa, sb, colsum, d2, act)


def gemm_glu(C, a, b, b2, d, *, d2=None, d3=None, aux=None, aux2=None, b_mn=False, act=RELU, sa=None, sb=None, sb2=None,
             counts=None, div=1, cg=0, wait=None, rot=0, mod=1, max_ctas=0):
    wf, wr, wpg, wt = wait if wait is not None else (0, 0, 0, 0)
    C.gemm_glu(a, b, b2, d, d2, d3, aux, aux2, b_mn, act, sa, sb, sb2, counts, div, cg, wf, wr, wpg, wt, rot, mod, max_ctas)


# ------------------------------------------------------------------------------------------------------------------
# data, layouts, references
# ------------------------------------------------------------------------------------------------------------------
def _gen(seed):
    return torch.Generator(device='cuda').manual_seed(seed)


def ints(gen, shape, lo, hi):
    """Uniform integers in [lo, hi] as float64 on the GPU."""
    return torch.randint(lo, hi + 1, shape, generator=gen, device='cuda', dtype=torch.float64)


def sparse01(gen, shape):
    """{0, 1} with P(1) = 1/4."""
    return (ints(gen, shape, 0, 3) == 0).double()


def quarters(gen, shape, act, lo=-3, hi=6):
    """Pre-activations for the activation-gradient epilogues: multiples of 1/4 in [lo, hi], exact in bf16 / fp16.  GELU'
    has a zero near -0.7518, and GELU'(-0.75) = 7.7e-4 is the difference of two terms near 0.226: its fp32 evaluation
    error (a few 1e-7) can exceed an fp16 ulp there, so -0.75 is replaced by -1.  On the remaining points |act'| >= 0.006
    and the fp32 evaluation (CUDA: erff <= 2 ulp, __expf <= 2 + floor(1.173 |x|) ulp, __fdividef <= 2 ulp) stays within
    1e-5 relative of the float64 value."""
    x = ints(gen, shape, 4 * lo, 4 * hi) / 4
    return torch.where(x == -0.75, torch.full_like(x, -1.0), x) if act == GELU else x


def with_signed_zeros(gen, x):
    """Replace about an eighth of the entries by -0.0 (the integers already contain +0.0)."""
    return torch.where(ints(gen, x.shape, 0, 7) == 0, torch.full_like(x, -0.0), x)


def _esize(dtype):
    return torch.empty((), dtype=dtype).element_size()


def canvas(G, rows, cols, dtype, pad, fill):
    """(view [G, rows, cols], backing buffer or None).  With `pad` the view is a slice of a taller and wider buffer whose
    margins hold SENTINEL; a leading dimension that is not 16-byte aligned also gets such a buffer."""
    align = 16 // _esize(dtype)
    ld = -(-cols // align) * align + (align if pad else 0)
    if ld == cols:
        return torch.full((G, rows, cols), fill, dtype=FP32, device='cuda').to(dtype), None
    top, extra = (2, 5) if pad else (0, 0)
    buf = torch.full((G, rows + extra, ld), SENTINEL, dtype=FP32, device='cuda')
    buf[:, top:top + rows, :cols] = fill
    buf = buf.to(dtype)
    return buf[:, top:top + rows, :cols], buf


def margin_ok(view, buf):
    if buf is None:
        return True
    inside = torch.zeros(buf.shape, dtype=torch.bool, device='cuda')
    top = (view.data_ptr() - buf.data_ptr()) // view.element_size() // buf.stride(1)
    inside[:, top:top + view.size(1), :view.size(2)] = True
    return bool((buf.float()[~inside] == SENTINEL).all())


def place(x, mn_major, dtype, pad):
    """Kernel layout of a logical [G, R, K] operand (K-major [G, R, K] or MN-major [G, K, R]) -> (tensor, buffer)."""
    t = x.transpose(1, 2) if mn_major else x
    view, buf = canvas(t.size(0), t.size(1), t.size(2), dtype, pad, 0.0)
    if buf is None:
        return t.to(FP32).to(dtype).contiguous(), None
    buf_f = buf.float()
    top = (view.data_ptr() - buf.data_ptr()) // view.element_size() // buf.stride(1)
    buf_f[:, top:top + t.size(1), :t.size(2)] = t.float()
    buf = buf_f.to(dtype)
    return buf[:, top:top + t.size(1), :t.size(2)], buf


def act_f64(act, x):
    if act == RELU:
        return torch.relu(x)
    if act == GELU:
        return 0.5 * x * (1 + torch.special.erf(x / math.sqrt(2)))
    return x * torch.sigmoid(x)


def dact_f64(act, x):
    if act == RELU:
        return (x > 0).double()
    if act == GELU:
        return 0.5 * (1 + torch.special.erf(x / math.sqrt(2))) + x * torch.exp(-0.5 * x * x) / math.sqrt(2 * math.pi)
    s = torch.sigmoid(x)
    return s * (1 + x * (1 - s))


def ulp(ref, dtype):
    """Spacing of `dtype` at |ref| (subnormal spacing below the normal range)."""
    mant, emin = {BF16: (7, -126), FP16: (10, -14)}[dtype]
    _, e = torch.frexp(ref.abs().clamp_min(2.0 ** emin))
    return torch.exp2((e - 1 - mant).double())


def assert_matches(name, got, ref, valid, exact):
    """Rows [0, valid[g]) of group g match `ref`; the rows after them still hold the NaN fill.

    `exact`: bit for bit after rounding `ref` to the output dtype.  Otherwise (GELU / SiLU): a 16-bit output within one
    ulp of `ref` - half an ulp for the final rounding plus the fp32 evaluation error, which on the inputs used here
    (pre-activations >= -3, see `quarters`) is below 1e-4 relative, i.e. below 0.2 fp16 ulp; an fp32 output within
    1e-6 + 1e-5 |ref| (about 80 fp32 ulp: the fp32 result is final, and GELU at x = -3 loses 4e-5 relative to the
    cancellation in 1 + erff, which the 1e-6 absolute term covers)."""
    for g, v in enumerate(valid):
        have, want = got[g, :v], ref[g, :v]
        if exact:
            ok = torch.equal(have, want.to(got.dtype))
        elif got.dtype == FP32:
            ok = bool(((have.double() - want).abs() <= 1e-6 + 1e-5 * want.abs()).all())
        else:
            ok = bool(torch.isfinite(have).all()) and bool(((have.double() - want).abs() <= ulp(want, got.dtype)).all())
        if not ok:
            bad = (have.double() != want.to(got.dtype).double()).nonzero()[:5].tolist()
            raise AssertionError('%s: group %d differs from the float64 reference at %s' % (name, g, bad))
        assert bool(got[g, v:].isnan().all()), '%s: group %d has writes past row %d' % (name, g, v)


def run(C, epi, *, G=2, M=129, N=264, K=72, dtype=BF16, out=None, a_mn=False, b_mn=False, cg=1, bn=0, act=0, div=1,
        alpha=1.0, bias=False, counts=None, colsum=False, scales=False, pad=False, max_ctas=0, rot=0, mod=1, wait=None,
        rnd=False, seed=0, check=True, lim=3, save_pre=True):
    """One launch of `epi` on generated data, checked against float64 (unless `check` is False).  Returns the outputs."""
    gen = _gen(seed)
    glu, fwd_glu = epi in (EPI_GLU, EPI_GLU_BWD), epi == EPI_GLU
    out = out or (dtype if _esize(dtype) == 2 else BF16)
    Gb = -(-G // div)
    # pre-activations of GELU / SiLU forward epilogues must stay >= -3: column 0 of A is 1, column 0 of B is in [-3, 0]
    smooth_fwd = epi in (EPI_BIAS_GELU, EPI_BIAS_SILU) or (fwd_glu and act != RELU)
    if rnd:
        A = torch.randn(G, M, K, generator=gen, device='cuda', dtype=torch.float64) * 0.5
        B = torch.randn(Gb, N, K, generator=gen, device='cuda', dtype=torch.float64) * 0.5
    elif smooth_fwd:
        A, B = sparse01(gen, (G, M, K)), sparse01(gen, (Gb, N, K))
        A[:, :, 0] = 1
        B[:, :, 0] = ints(gen, (Gb, N), -3, 0)
    else:
        A, B = ints(gen, (G, M, K), -lim, lim), ints(gen, (Gb, N, K), -lim, lim)
    B2 = ints(gen, (Gb, N, K), -lim, lim) if fwd_glu else None
    a, a_buf = place(A, a_mn, dtype, pad)
    b, b_buf = place(B, b_mn, dtype, pad)
    b2 = place(B2, b_mn, dtype, pad)[0] if fwd_glu else None
    A, B = a.double().transpose(1, 2) if a_mn else a.double(), b.double().transpose(1, 2) if b_mn else b.double()
    Bx = B.repeat_interleave(div, 0)[:G]
    acc = torch.matmul(A, Bx.transpose(1, 2))
    sa = sb = None
    if scales:
        sa = torch.exp2(ints(gen, (G, M), -2, 2)).float()
        sb = torch.exp2(ints(gen, (Gb, N), -2, 2)).float()
        acc = acc * sa.double()[:, :, None] * sb.double().repeat_interleave(div, 0)[:G, None, :]

    bias_t = None
    if bias:
        bias_t = (ints(gen, (Gb, N), 0, 1) if smooth_fwd else ints(gen, (Gb, N), -lim, lim)).to(dtype if _esize(dtype) == 2 else out)
    d, d_buf = canvas(G, M, N, out, pad, NAN)
    new = lambda: canvas(G, M, N, out, pad, NAN)[0]  # noqa: E731  (same layout as d)

    def side(x):
        t = new()
        t.copy_(x)
        return t

    aux = aux2 = d2 = d3 = None
    if epi in (EPI_RELU_BWD, EPI_ADD) or (epi == EPI_ACT_BWD and act == RELU):
        x = ints(gen, (G, M, N), -lim, lim)
        aux = side(with_signed_zeros(gen, x) if epi != EPI_ADD else x)
    elif epi == EPI_ACT_BWD:
        aux = side(quarters(gen, (G, M, N), act))
    elif epi == EPI_GLU_BWD:
        aux = side(with_signed_zeros(gen, ints(gen, (G, M, N), -lim, lim)) if act == RELU else quarters(gen, (G, M, N), act))
        aux2 = side(ints(gen, (G, M, N), -lim, lim))
    if epi in (EPI_BIAS_GELU, EPI_BIAS_SILU, EPI_GLU_BWD) or (fwd_glu and save_pre):
        d2 = new()
    if fwd_glu and save_pre:
        d3 = new()
    counts_t = torch.tensor(counts, dtype=torch.int32, device='cuda') if counts is not None else None
    colsum_t = torch.zeros(Gb, N, dtype=FP32, device='cuda') if colsum else None
    if rnd:
        for t in (aux, aux2):
            if t is not None:
                t.copy_(torch.randn(t.shape, generator=gen, device='cuda'))

    if glu:
        gemm_glu(C, a, b, b2, d, d2=d2, d3=d3, aux=aux, aux2=aux2, b_mn=b_mn, act=act, counts=counts_t, div=div, cg=cg,
                 wait=wait, rot=rot, mod=mod, max_ctas=max_ctas)
    else:
        gemm_ex(C, a, b, d, a_mn=a_mn, b_mn=b_mn, epi=epi, bias=bias_t, aux=aux, counts=counts_t, alpha=alpha, div=div, cg=cg,
                bn=bn, wait=wait, max_ctas=max_ctas, rot=rot, mod=mod, sa=sa, sb=sb, colsum=colsum_t, d2=d2, act=act)
    torch.cuda.synchronize()
    outs = {'d': d, 'd2': d2, 'd3': d3, 'colsum': colsum_t}
    if not check:
        return outs

    # ---- float64 reference ----
    smooth = act in (GELU, SILU) or epi in (EPI_BIAS_GELU, EPI_BIAS_SILU)
    refs = {}
    if bias_t is not None:
        acc = acc + bias_t.double().repeat_interleave(div, 0)[:G, None, :]
    if epi == EPI_NONE:
        refs['d'] = acc * alpha
    elif epi == EPI_BIAS:
        refs['d'] = acc
    elif epi == EPI_BIAS_RELU:
        refs['d'] = torch.relu(acc)
    elif epi in (EPI_BIAS_GELU, EPI_BIAS_SILU):
        refs['d'] = act_f64(GELU if epi == EPI_BIAS_GELU else SILU, acc)
        refs['d2'] = acc
    elif epi == EPI_RELU_BWD:
        refs['d'] = torch.where(aux.double() > 0, acc, torch.zeros_like(acc))
    elif epi == EPI_ADD:
        refs['d'] = acc + aux.double()
    elif epi == EPI_ACT_BWD:
        refs['d'] = acc * dact_f64(act, aux.double())
    elif epi == EPI_GLU:
        B2x = b2.double().repeat_interleave(div, 0)[:G]              # [G, K, N] (b_mn) or [G, N, K]
        u = torch.matmul(A, B2x if b_mn else B2x.transpose(1, 2))
        refs['d'] = act_f64(act, acc) * u
        if save_pre:
            refs['d2'], refs['d3'] = acc, u
    else:
        g, u = aux.double(), aux2.double()
        refs['d'], refs['d2'] = acc * u * dact_f64(act, g), acc * act_f64(act, g)
    valid = [min(M, c) for c in counts] if counts is not None else [M] * G
    for name, ref in refs.items():
        exact = not smooth or (name in ('d2', 'd3') and epi != EPI_GLU_BWD)
        assert_matches('epilogue %d %s' % (epi, name), outs[name], ref, valid, exact)
    if colsum:
        want = torch.zeros(Gb, N, dtype=torch.float64, device='cuda')
        for g, v in enumerate(valid):
            want[g // div] += refs['d'][g, :v].sum(0)
        assert torch.equal(colsum_t.double(), want), 'fused column sums differ'
    for name, view, buf in (('a', a, a_buf), ('b', b, b_buf), ('d', d, d_buf)):
        assert margin_ok(view, buf), 'margin of %s was written' % name
    for t in (aux, aux2, d2, d3):
        if t is not None and t._base is not None:
            assert margin_ok(t, t._base), 'margin of a side tensor was written'
    return outs


def same(x, y):
    return all((x[k] is None and y[k] is None) or torch.equal(x[k], y[k]) for k in x)


# ------------------------------------------------------------------------------------------------------------------
# core: CTA group x BN x operand majorness x 16-bit input dtype, over M / N / K tails
# ------------------------------------------------------------------------------------------------------------------
CORE_SHAPES = [(2, 1, 136, 200), (2, 8, 8, 72), (2, 129, 264, 8), (2, 257, 136, 72), (3, 328, 264, 200)]


@pytest.mark.parametrize('dtype', [BF16, FP16])
@pytest.mark.parametrize('a_mn,b_mn', LAYOUTS)
@pytest.mark.parametrize('bn', [128, 256])
@pytest.mark.parametrize('cg', [1, 2])
def test_core_layouts_and_tails(C, cg, bn, a_mn, b_mn, dtype):
    other = FP16 if dtype == BF16 else BF16
    for i, (G, M, N, K) in enumerate(CORE_SHAPES):
        out = (dtype, FP32, other, FP32, dtype)[i]
        run(C, EPI_NONE, G=G, M=M, N=N, K=K, dtype=dtype, out=out, a_mn=a_mn, b_mn=b_mn, cg=cg, bn=bn, pad=(i == 2), seed=i)


@pytest.mark.parametrize('cg', [1, 2])
def test_second_band_of_row_blocks(C, cg):
    """M = 2312: 19 row blocks of 128 (cg 1) or 10 of 256 (cg 2), i.e. more than one band of 16 / 8 and a partial one."""
    for out in (BF16, FP32):
        run(C, EPI_BIAS, G=2, M=2312, N=264, K=72, bias=True, cg=cg, out=out, seed=cg)


# ------------------------------------------------------------------------------------------------------------------
# fp8 operands
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('bn', [128, 256])
@pytest.mark.parametrize('cg', [1, 2])
@pytest.mark.parametrize('dtype', [E4M3, E5M2])
def test_fp8_operands_scales_and_shared_b(C, dtype, cg, bn):
    # K = 144 / 1040: multiples of 16, not of 128 (a partial last 128-byte K block)
    for i, (K, scales, div) in enumerate([(144, False, 1), (1040, True, 1), (144, True, 2), (1040, False, 2)]):
        run(C, EPI_NONE, G=4, M=129, N=136, K=K, dtype=dtype, cg=cg, bn=bn, scales=scales, div=div, pad=(i == 1), seed=i)
    run(C, EPI_BIAS_RELU, G=4, M=129, N=264, K=144, dtype=dtype, out=FP16, cg=cg, bn=bn, scales=True, div=2, bias=True)


# ------------------------------------------------------------------------------------------------------------------
# epilogues with exact results
# ------------------------------------------------------------------------------------------------------------------
EXACT_EPILOGUES = [('none_alpha_0.5', EPI_NONE, 0, 0.5), ('none_alpha_4', EPI_NONE, 0, 4.0), ('bias', EPI_BIAS, 0, 1.0),
                   ('bias_relu', EPI_BIAS_RELU, 0, 1.0), ('relu_bwd', EPI_RELU_BWD, 0, 1.0), ('add', EPI_ADD, 0, 1.0),
                   ('act_bwd_relu', EPI_ACT_BWD, RELU, 1.0)]


@pytest.mark.parametrize('a_mn,b_mn', LAYOUTS)
@pytest.mark.parametrize('bn', [128, 256])
@pytest.mark.parametrize('cg', [1, 2])
@pytest.mark.parametrize('name,epi,act,alpha', EXACT_EPILOGUES, ids=[e[0] for e in EXACT_EPILOGUES])
def test_exact_epilogues(C, name, epi, act, alpha, cg, bn, a_mn, b_mn):
    dtype = BF16 if bn == 256 else FP16
    outs = [dtype] if epi in (EPI_RELU_BWD, EPI_ADD, EPI_ACT_BWD) else [dtype, FP32]
    for i, out in enumerate(outs):
        run(C, epi, act=act, alpha=alpha, bias=epi in (EPI_BIAS, EPI_BIAS_RELU), dtype=dtype, out=out, a_mn=a_mn, b_mn=b_mn,
            cg=cg, bn=bn, pad=(a_mn == b_mn), seed=i)


@pytest.mark.parametrize('epi,dtype,out,shape', [(EPI_BIAS_RELU, FP16, FP16, (2, 512, 520, 1096)),
                                                 (EPI_BIAS_RELU, BF16, FP32, (2, 512, 520, 1096)),
                                                 (EPI_RELU_BWD, FP16, FP16, (2, 512, 520, 1096)),
                                                 (EPI_ADD, BF16, BF16, (2, 300, 264, 128))])
def test_epilogues_with_default_tiling(C, epi, dtype, out, shape):
    """cta_group and BN picked by the launcher (0 = auto), as the layers call it."""
    G, M, N, K = shape
    run(C, epi, G=G, M=M, N=N, K=K, dtype=dtype, out=out, cg=0, bn=0, bias=epi == EPI_BIAS_RELU)


# ------------------------------------------------------------------------------------------------------------------
# GELU / SiLU epilogues (one ulp of a 16-bit output; the saved pre-activation exactly)
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('out', [BF16, FP16, FP32])
@pytest.mark.parametrize('cg', [1, 2])
@pytest.mark.parametrize('epi', [EPI_BIAS_GELU, EPI_BIAS_SILU])
def test_gelu_silu_forward_saves_exact_pre_activation(C, epi, cg, out):
    """d2 receives acc + bias.  With an fp32 output it has fp32 rows (it once was addressed with 2-byte rows)."""
    dtype = out if out != FP32 else BF16
    run(C, epi, dtype=dtype, out=out, cg=cg, bias=True)
    if out == FP32:     # also in a padded buffer: ldd = N + 4, group stride > dense
        run(C, epi, dtype=dtype, out=out, cg=cg, bias=True, pad=True, seed=1)


@pytest.mark.parametrize('dtype', [BF16, FP16])
@pytest.mark.parametrize('cg', [1, 2])
@pytest.mark.parametrize('act', [GELU, SILU])
def test_activation_gradient_epilogue(C, act, cg, dtype):
    for bn in (128, 256):
        run(C, EPI_ACT_BWD, act=act, dtype=dtype, cg=cg, bn=bn, b_mn=(bn == 128))


# ------------------------------------------------------------------------------------------------------------------
# gated linear unit (dual-B forward, fused backward)
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('dtype', [BF16, FP16])
@pytest.mark.parametrize('b_mn', [False, True])
@pytest.mark.parametrize('cg', [1, 2])
@pytest.mark.parametrize('act', [RELU, GELU, SILU])
def test_glu_forward_and_backward(C, act, cg, b_mn, dtype):
    """h = act(A.B) * (A.B2) with g = A.B, u = A.B2 saved; backward dg = dh * u * act'(g), du = dh * act(g).  ReLU exact;
    K = 72 keeps the products of two accumulators below 2^24."""
    run(C, EPI_GLU, act=act, dtype=dtype, b_mn=b_mn, cg=cg, N=328, pad=b_mn)
    run(C, EPI_GLU, act=act, dtype=dtype, b_mn=b_mn, cg=cg, N=328, pad=not b_mn, save_pre=False, seed=2)   # h only
    run(C, EPI_GLU_BWD, act=act, dtype=dtype, b_mn=b_mn, cg=cg, N=328, pad=not b_mn, seed=1)


# ------------------------------------------------------------------------------------------------------------------
# fused bias-gradient column sums
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('div', [1, 2])
@pytest.mark.parametrize('cg', [1, 2])
@pytest.mark.parametrize('epi', [EPI_BIAS_RELU, EPI_RELU_BWD, EPI_ACT_BWD])
def test_fused_column_sums(C, epi, cg, div):
    """colsum[g // div] += column sums of the fp32 epilogue result over the M valid rows.  M = 129 leaves 127 (cg 1) or
    127 + 128 (cg 2) masked rows in the last tile; with a bias those rows would add relu(bias) if they were counted."""
    run(C, epi, act=RELU if epi == EPI_ACT_BWD else 0, G=4, M=129, bias=epi == EPI_BIAS_RELU, colsum=True, cg=cg, div=div,
        seed=div)


# ------------------------------------------------------------------------------------------------------------------
# row_counts (dropless / Megablocks): direct side loads, bulk or direct stores, skipped tiles
# ------------------------------------------------------------------------------------------------------------------
ROW_COUNT_CASES = [('none', EPI_NONE, 0, {}), ('none_fp32', EPI_NONE, 0, {'out': FP32}), ('bias', EPI_BIAS, 0, {'bias': True}),
                   ('bias_relu', EPI_BIAS_RELU, 0, {'bias': True, 'colsum': True}),
                   ('relu_bwd', EPI_RELU_BWD, 0, {'colsum': True}), ('add', EPI_ADD, 0, {}),
                   ('act_bwd_relu', EPI_ACT_BWD, RELU, {'colsum': True}), ('act_bwd_gelu', EPI_ACT_BWD, GELU, {}),
                   ('bias_gelu', EPI_BIAS_GELU, 0, {'bias': True}), ('bias_silu_fp32', EPI_BIAS_SILU, 0, {'bias': True, 'out': FP32}),
                   ('glu_relu', EPI_GLU, RELU, {}), ('glu_silu', EPI_GLU, SILU, {}),
                   ('glu_bwd_relu', EPI_GLU_BWD, RELU, {}), ('glu_bwd_gelu', EPI_GLU_BWD, GELU, {})]


@pytest.mark.parametrize('cg', [1, 2])
@pytest.mark.parametrize('name,epi,act,kw', ROW_COUNT_CASES, ids=[c[0] for c in ROW_COUNT_CASES])
def test_row_counts(C, name, epi, act, kw, cg):
    """Rows below the count are exact, rows past it inside a computed tile keep the NaN fill, skipped tiles too."""
    run(C, epi, act=act, G=6, M=300, counts=[0, 1, 127, 128, 129, 1000], cg=cg, pad=(cg == 2), **kw)


def test_row_counts_with_default_tiling(C):
    run(C, EPI_NONE, G=4, M=512, N=256, K=256, counts=[512, 0, 130, 257], cg=0, bn=0)


# ------------------------------------------------------------------------------------------------------------------
# persistent schedule: several tiles per CTA
# ------------------------------------------------------------------------------------------------------------------
PERSISTENT_CASES = [('none', EPI_NONE, {'bn': 128}), ('relu_bwd', EPI_RELU_BWD, {'bn': 128}), ('add', EPI_ADD, {'bn': 128}),
                    ('glu_save_pre', EPI_GLU, {'act': RELU}), ('glu_bwd', EPI_GLU_BWD, {'act': RELU})]


@pytest.mark.parametrize('rnd', [False, True], ids=['integers', 'random'])
@pytest.mark.parametrize('cg', [1, 2])
@pytest.mark.parametrize('name,epi,kw', PERSISTENT_CASES, ids=[c[0] for c in PERSISTENT_CASES])
def test_persistent_schedule_is_grid_independent(C, name, epi, kw, cg, rnd):
    """G = 4, M = 1024 * cg, N = 1024: 256 tiles (128 for the GLU backward, BN 256).  max_ctas = cg runs all of them on
    one CTA / pair (both TMEM accumulators and the operand ring wrap many times, the side inputs of the next tile are
    prefetched while the current one drains); 3 and 7 CTAs / pairs run 19-86 tiles each; the default grid (148 CTAs or 74
    pairs) 1-4.  The per-tile accumulation order does not depend on the grid, so the results are bitwise equal."""
    shape = dict(G=4, M=1024 * cg, N=1024, K=128, cg=cg, rnd=rnd, check=not rnd, seed=7)
    base = run(C, epi, **shape, **kw)
    for n in (cg, 3 * cg, 7 * cg):
        assert same(run(C, epi, max_ctas=n, **shape, **kw), base), 'max_ctas=%d changed the result' % n


def test_one_cta_budget_still_runs_a_pair(C):
    """max_ctas = 1 with CTA pairs runs on one pair (it used to launch an empty grid)."""
    base = run(C, EPI_BIAS, bias=True, G=2, M=600, cg=2)
    assert same(run(C, EPI_BIAS, bias=True, G=2, M=600, cg=2, max_ctas=1), base)


# ------------------------------------------------------------------------------------------------------------------
# tile order: group rotation as the fused engine uses it
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('cg', [1, 2])
@pytest.mark.parametrize('mod', [2, -2, 3, -3])
def test_group_rotation_is_only_an_order(C, mod, cg):
    W = abs(mod)
    for epi, kw in ((EPI_NONE, {}), (EPI_RELU_BWD, {}), (EPI_GLU, {'act': RELU})):
        shape = dict(G=6, M=300, div=W, cg=cg, seed=W)
        base = run(C, epi, **shape, **kw)
        for rot in range(W):
            assert same(run(C, epi, rot=rot, mod=mod, **shape, **kw), base), 'rot=%d mod=%d changed the result' % (rot, mod)


# ------------------------------------------------------------------------------------------------------------------
# pointer-table output and completion counters (the combine fusion), on one GPU
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('cap', [100, 300])
@pytest.mark.parametrize('out', [BF16, FP32])
def test_pointer_table_output_and_completion_counters(C, out, cap):
    """Group g's [cap, N] rows go to slot perm[g] of one buffer, with sentinel rows between the slots; each group bumps
    its counter once per tile and CTA, which must be the count FusedEngine.tile_counts() tells the combine to wait for."""
    from tutel_b200.parallel.fused import FusedEngine
    W, El, N, K, gap = 4, 2, 264, 72, 3
    G = El * W
    cg, bn, per_group = FusedEngine.tile_counts(cap, N)
    gen = _gen(cap)
    perm = torch.randperm(G, generator=torch.Generator().manual_seed(cap)).tolist()
    starts = [gap + perm[g] * (cap + gap) for g in range(G)]
    A, B = ints(gen, (G, cap, K), -3, 3), ints(gen, (El, N, K), -3, 3)
    a, b = A.to(BF16), B.to(BF16)
    ref = torch.matmul(A, B.repeat_interleave(W, 0).transpose(1, 2))
    epis = [EPI_NONE] + ([EPI_ADD] if out == BF16 else [])
    for epi in epis:
        aux = ints(gen, (G, cap, N), -3, 3).to(out) if epi == EPI_ADD else None
        want = ref + aux.double() if aux is not None else ref
        for rank in range(W):
            buf = torch.full((gap + G * (cap + gap), N), SENTINEL, dtype=out, device='cuda')
            for s in starts:
                buf[s:s + cap] = NAN
            table = torch.tensor([buf[s].data_ptr() for s in starts], dtype=torch.int64, device='cuda')
            counters = torch.zeros(G, dtype=torch.int32, device='cuda')
            signals = torch.tensor([counters[g].data_ptr() for g in range(G)], dtype=torch.int64, device='cuda')
            d = buf[gap:].view(G, cap + gap, N)[:, :cap]
            gemm_ex(C, a, b, d, epi=epi, aux=aux, div=W, cg=cg, bn=bn, d_table=table.data_ptr(), s_table=signals.data_ptr(),
                    rot=rank, mod=-W)
            torch.cuda.synchronize()
            for g, s in enumerate(starts):
                assert torch.equal(buf[s:s + cap], want[g].to(out)), 'group %d (rank %d)' % (g, rank)
            mask = torch.ones(buf.size(0), dtype=torch.bool, device='cuda')
            for s in starts:
                mask[s:s + cap] = False
            assert bool((buf[mask].float() == SENTINEL).all()), 'a sentinel row was written'
            assert counters.tolist() == [per_group] * G


# ------------------------------------------------------------------------------------------------------------------
# dispatch wait flags that are already satisfied
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('cg', [1, 2])
def test_satisfied_wait_flags_change_nothing(C, cg):
    """Every flag holds the target before the launch, so the producer never waits; the flag array is padded well past
    G * flags_per_group.  (Flag indexing under real arrival order is exercised by the multi-GPU tests.)"""
    G, M, per_group, target = 4, 300, 8, 5
    flags = torch.full((G * per_group + 256,), target, dtype=torch.int32, device='cuda')
    for epi, kw in ((EPI_NONE, {}), (EPI_RELU_BWD, {}), (EPI_GLU, {'act': RELU}), (EPI_GLU_BWD, {'act': SILU})):
        base = run(C, epi, G=G, M=M, cg=cg, **kw)
        for rows in (64, 0):       # 0: one flag per tile height
            got = run(C, epi, G=G, M=M, cg=cg, wait=(flags.data_ptr(), rows, per_group, target), **kw)
            assert same(got, base)


# ------------------------------------------------------------------------------------------------------------------
# the six GEMMs of one bench.py training step, at full size
# ------------------------------------------------------------------------------------------------------------------
BENCH = [  # name, epilogue, M, N, K, a_mn, b_mn, operand bound, bias, colsum
    ('fc1_fwd', EPI_BIAS_RELU, 2048, 14336, 4096, False, False, 3, True, False),
    ('fc2_fwd', EPI_BIAS, 2048, 4096, 14336, False, True, 2, True, False),
    ('fc1_dgrad_relu_bwd_colsum', EPI_RELU_BWD, 2048, 14336, 4096, False, False, 1, False, True),
    ('fc2_dgrad', EPI_NONE, 2048, 4096, 14336, False, True, 2, False, False),
    ('fc2_wgrad', EPI_NONE, 14336, 4096, 2048, True, True, 3, False, False),
    ('fc1_wgrad', EPI_NONE, 14336, 4096, 2048, True, True, 3, False, False),
]


@pytest.mark.parametrize('name,epi,M,N,K,a_mn,b_mn,lim,bias,colsum', BENCH, ids=[b[0] for b in BENCH])
def test_bench_step_gemms_at_full_size(C, name, epi, M, N, K, a_mn, b_mn, lim, bias, colsum):
    """8 local experts, 2048 rows, model 4096, hidden 14336, default tiling.  Operand bounds keep every partial sum below
    2^16 and the column sums (2048 rows x 4096) below 2^24."""
    run(C, epi, G=8, M=M, N=N, K=K, a_mn=a_mn, b_mn=b_mn, lim=lim, bias=bias, colsum=colsum, cg=0, bn=0, seed=M + K)


# ------------------------------------------------------------------------------------------------------------------
# host-side refusals (nothing is launched)
# ------------------------------------------------------------------------------------------------------------------
def _small(dtype=BF16, G=4, M=300, N=136, K=64, out=BF16):
    a = torch.ones(G, M, K, device='cuda').to(dtype)
    b = torch.ones(G, N, K, device='cuda').to(dtype)
    return a, b, torch.empty(G, M, N, device='cuda', dtype=out)


@pytest.mark.parametrize('dtype', [torch.float32, torch.int32, torch.int8])
def test_refuses_non_gemm_operand_dtypes(C, dtype):
    a, b, d = _small(dtype)
    with pytest.raises(RuntimeError):
        gemm_ex(C, a, b, d)
    with pytest.raises(RuntimeError):
        gemm_glu(C, a, b, b.clone(), d)
    u = torch.zeros_like(d)
    with pytest.raises(RuntimeError):
        gemm_glu(C, a, b, None, d, d2=torch.empty_like(d), aux=u, aux2=u.clone())


def test_refuses_side_tensors_of_the_wrong_shape(C):
    G, M, N = 4, 300, 136
    a, b, d = _small(G=G, M=M, N=N)
    f32 = dict(device='cuda', dtype=FP32)
    cases = {
        'bias columns': dict(epi=EPI_BIAS, bias=torch.zeros(G, N + 8, device='cuda', dtype=BF16)),
        'bias rows': dict(epi=EPI_BIAS, bias=torch.zeros(1, N, device='cuda', dtype=BF16), div=2),
        'aux rows': dict(epi=EPI_ADD, aux=torch.zeros(G, M - 1, N, device='cuda', dtype=BF16)),
        'aux columns': dict(epi=EPI_ADD, aux=torch.zeros(G, M, N + 8, device='cuda', dtype=BF16)),
        'aux groups': dict(epi=EPI_RELU_BWD, aux=torch.zeros(G - 1, M, N, device='cuda', dtype=BF16)),
        'colsum rows': dict(epi=EPI_BIAS_RELU, colsum=torch.zeros(1, N, **f32), div=2),
    }
    for name, kw in cases.items():
        with pytest.raises(RuntimeError):
            gemm_ex(C, a, b, d, **kw)
            pytest.fail(name)
    aq, bq = a.to(E4M3), b.to(E4M3)
    with pytest.raises(RuntimeError):
        gemm_ex(C, aq, bq, d, sb=torch.ones(1, N, **f32), div=2)
    with pytest.raises(RuntimeError):
        gemm_glu(C, aq, bq, bq.clone(), d, sb=torch.ones(1, N, **f32), div=2)
    with pytest.raises(RuntimeError):
        gemm_glu(C, aq, bq, bq.clone(), d, sa=torch.ones(G - 1, M, **f32))


def test_refuses_group_rotation_out_of_range(C):
    a, b, d = _small(G=5)
    for rot, mod in ((1, 2), (0, -3), (-1, 1), (-1, 5), (5, 5), (2, -2)):
        with pytest.raises(RuntimeError):
            gemm_ex(C, a, b, d, rot=rot, mod=mod)
        with pytest.raises(RuntimeError):
            gemm_glu(C, a, b, b.clone(), d, rot=rot, mod=mod)


def test_refuses_more_than_64_wait_flags_per_group(C):
    a, b, d = _small(M=300)
    flags = torch.full((4 * 128,), 1, dtype=torch.int32, device='cuda')     # satisfied: never a wait, even if not refused
    for rows, per_group in ((4, 128), (64, 4)):      # 75 flags per group; 5 flags in a 4-flag stride
        with pytest.raises(RuntimeError):
            gemm_ex(C, a, b, d, wait=(flags.data_ptr(), rows, per_group, 1))
        with pytest.raises(RuntimeError):
            gemm_glu(C, a, b, b.clone(), d, wait=(flags.data_ptr(), rows, per_group, 1))


def test_refuses_unsupported_fp8_combinations(C):
    a, b, d = _small(E4M3, M=256, N=128)
    pre = torch.empty_like(d)
    for epi, act in ((EPI_BIAS_GELU, 0), (EPI_BIAS_SILU, 0), (EPI_ACT_BWD, GELU)):
        with pytest.raises(RuntimeError):
            gemm_ex(C, a, b, d, epi=epi, act=act, aux=pre if epi == EPI_ACT_BWD else None)
    at, bt = a.transpose(1, 2).contiguous(), b.transpose(1, 2).contiguous()
    for a_mn, b_mn in ((True, False), (False, True), (True, True)):
        with pytest.raises(RuntimeError):
            gemm_ex(C, at if a_mn else a, bt if b_mn else b, d, a_mn=a_mn, b_mn=b_mn)
