"""Numerics of every native CUDA kernel against plain PyTorch fp32 references (run with `pytest -m gpu` on a B200)."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def C():
    from tutel_b200.ops import backend
    return backend.require_ext()


@pytest.mark.parametrize('S,E,k', [(8192, 8, 2), (5000, 130, 3), (33, 128, 1)])
def test_routing_kernels_match_cpu(C, S, E, k):
    torch.manual_seed(S)
    idx = torch.topk(torch.rand(S, E), k, dim=1).indices.t().contiguous().to(torch.int32)
    loc_ref, cnt_ref = C.cpu_route_locations(idx, E)
    cap = max(1, S * k // E // 2)
    loc, cnt, slot = C.route_locations(idx.cuda(), E, cap)
    assert torch.equal(loc.cpu(), loc_ref) and torch.equal(cnt.cpu(), cnt_ref)
    ok = loc_ref < cap
    want = torch.full((E * cap,), -1, dtype=torch.int32)
    tok = torch.arange(S, dtype=torch.int32).unsqueeze(0) * k + torch.arange(k, dtype=torch.int32).unsqueeze(1)
    want[(idx.long() * cap + loc_ref.long())[ok]] = tok[ok]
    assert torch.equal(slot.cpu(), want)


@pytest.mark.parametrize('dtype,M', [(torch.bfloat16, 4096), (torch.float16, 264), (torch.float32, 257)])
def test_encode_decode_gate_grad_match_cpu(C, dtype, M):
    torch.manual_seed(3)
    S, E, k, cap = 1000, 6, 2, 200
    idx = torch.topk(torch.rand(S, E), k, dim=1).indices.t().contiguous().to(torch.int32)
    loc, _ = C.cpu_route_locations(idx, E)
    gates = torch.rand(k, S)
    x = torch.randn(S, M).to(dtype)
    y = torch.randn(E * cap, M).to(dtype)
    tol = 1e-5 if dtype == torch.float32 else 3e-2
    idx_d, loc_d = idx.cuda(), loc.cuda()
    slot = C.build_slot_map(idx_d, loc_d, E, cap)
    out = torch.empty(E * cap, M, dtype=dtype, device='cuda')
    C.encode_rows(x.cuda(), gates.cuda(), slot, out, k, E, cap, 0, 0, 0, 0, 0, 0, None)
    assert torch.allclose(out.float().cpu(), C.cpu_encode(x.float(), gates, idx, loc, E, cap), atol=tol, rtol=tol)
    dec = C.decode_rows(y.cuda(), gates.cuda(), idx_d, loc_d, E, cap, 0, 0)
    ref = C.cpu_decode(y.float(), gates, idx, loc, E, cap)
    assert torch.allclose(dec.float().cpu(), ref, atol=tol * 4, rtol=tol)
    gg = C.gate_grad(x.cuda(), y.cuda(), idx_d, loc_d, E, cap)
    ref = C.cpu_gate_grad(x.float(), y.float(), idx, loc, E, cap)
    assert torch.allclose(gg.cpu(), ref, atol=tol * M ** 0.5, rtol=tol)


def test_nvrtc_jit_kernel():
    from tutel_b200 import jit
    fn = jit.create_cuda_kernel(r'''
      extern "C" __global__ void axpb(float* x, float* y, int n, int a) {
        // [thread_extent] blockIdx.x = @grid@
        // [thread_extent] threadIdx.x = 256
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) y[i] = x[i] * a + 1.0f;
      }''', {'grid': 64})
    x = torch.randn(100000, device='cuda')
    y = torch.empty_like(x)
    fn(x, y, extra=[x.numel(), 3])
    assert torch.allclose(y, x * 3 + 1, atol=1e-5)


def _layer(dtype, **kw):
    from tutel_b200 import moe
    torch.manual_seed(0)
    return moe.moe_layer(gate_type={'type': 'top', 'k': 2, 'capacity_factor': kw.pop('cf', 1.25)}, model_dim=256,
                         experts={'type': 'ffn', 'num_experts_per_device': 4, 'hidden_size_per_expert': 512,
                                  'activation_fn': lambda t: F.relu(t)}, seeds=(1, 1, 1), **kw).to(dtype)


def test_moe_layer_fp32_gpu_matches_cpu():
    cpu = _layer(torch.float32)
    gpu = _layer(torch.float32).cuda()
    x = torch.randn(3, 100, 256)
    xc, xg = x.clone().requires_grad_(True), x.cuda().requires_grad_(True)
    yc, yg = cpu(xc), gpu(xg)
    assert torch.allclose(yg.cpu(), yc, atol=1e-4, rtol=1e-4)
    (yc.pow(2).sum() + yc.l_aux).backward()
    (yg.pow(2).sum() + yg.l_aux).backward()
    assert torch.allclose(xg.grad.cpu(), xc.grad, atol=1e-3, rtol=1e-3)
    for pc, pg in zip(cpu.parameters(), gpu.parameters()):
        assert torch.allclose(pg.grad.cpu(), pc.grad, atol=2e-3, rtol=2e-3)


@pytest.mark.parametrize('is_postscore', [True, False])
def test_moe_layer_bf16_tcgen05_path_vs_fp32_reference(is_postscore):
    from tutel_b200.ops import backend
    ref = _layer(torch.float32, is_postscore=is_postscore).cuda()
    low = _layer(torch.float32, is_postscore=is_postscore).cuda().to(torch.bfloat16)
    x = torch.randn(4, 128, 256, device='cuda')
    xr, xl = x.clone().requires_grad_(True), x.bfloat16().requires_grad_(True)
    n0 = backend.launch_count()
    yr, yl = ref(xr), low(xl)
    yr.float().pow(2).mean().backward()
    yl.float().pow(2).mean().backward()
    assert backend.launch_count() > n0, 'native kernels were not used'
    # same routing is not guaranteed under bf16 rounding of the logits; compare aggregate error instead of exact values
    rel = (yl.float() - yr).norm() / yr.norm()
    assert rel < 0.08, rel
    g = (xl.grad.float() - xr.grad).norm() / xr.grad.norm()
    assert g < 0.15, g
    w = (low.experts.batched_fc1_w.grad.float() - ref.experts.batched_fc1_w.grad).norm() / ref.experts.batched_fc1_w.grad.norm()
    assert w < 0.15, w


def test_dropless_megablocks_inference_matches_padded():
    torch.manual_seed(0)
    from tutel_b200 import moe
    layer = moe.moe_layer(gate_type={'type': 'top', 'k': 1, 'capacity_factor': 0}, model_dim=256,
                          experts={'type': 'ffn', 'num_experts_per_device': 16, 'hidden_size_per_expert': 256,
                                   'activation_fn': lambda t: F.relu(t)}).cuda().to(torch.bfloat16).eval()
    x = torch.randn(1, 32, 256, device='cuda', dtype=torch.bfloat16)
    with torch.no_grad():
        a = layer(x)
        b = layer(x, megablocks_size=1)
    assert layer.megablocks_size == 1
    assert torch.allclose(a.float(), b.float(), atol=2e-2, rtol=2e-2)


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16])
@pytest.mark.parametrize('kn', [False, True])
def test_skinny_grouped_gemm(C, dtype, kn):
    torch.manual_seed(5)
    G, R, K, N = 9, 11, 1300, 520
    x = torch.randn(G, R, K, device='cuda').to(dtype)
    w = (torch.randn(G, K, N, device='cuda') * 0.05).to(dtype)
    b = torch.randn(G, N, device='cuda').to(dtype)
    counts = torch.tensor([11, 0, 3, 8, 1, 0, 9, 11, 2], device='cuda', dtype=torch.int32)
    w_op = w if kn else w.transpose(1, 2).contiguous()
    y = C.skinny_gemm(x, w_op, b, counts, kn, True)
    ref = torch.relu(torch.matmul(x.float(), w.float()) + b.float().unsqueeze(1))
    tol = 1e-3 if dtype == torch.float32 else 6e-2
    for g, c in enumerate(counts.tolist()):
        assert torch.allclose(y[g, :c].float(), ref[g, :c], atol=tol, rtol=tol)
        assert torch.count_nonzero(y[g, c:]) == 0


def test_dropless_fp32_many_experts_uses_skinny_path():
    torch.manual_seed(0)
    from tutel_b200 import moe
    from tutel_b200.ops import backend
    layer = moe.moe_layer(gate_type={'type': 'top', 'k': 1, 'capacity_factor': 0}, model_dim=256,
                          experts={'type': 'ffn', 'num_experts_per_device': 64, 'hidden_size_per_expert': 256,
                                   'activation_fn': lambda t: F.relu(t)}).cuda().eval()
    x = torch.randn(1, 32, 256, device='cuda')
    with torch.no_grad():
        a = layer(x)
        n0 = backend.launch_count()
        b = layer(x, megablocks_size=1)
    assert backend.launch_count() - n0 >= 2
    assert torch.allclose(a, b, atol=1e-4, rtol=1e-4)


@pytest.mark.parametrize('cg', [1, 2])
def test_fp8_gemm_with_row_col_scales(C, cg):
    from tutel_b200.ops import gemm as G
    torch.manual_seed(6)
    Gn, M, N, K = 2, 384, 272, 512
    a = torch.randn(Gn, M, K, device='cuda').bfloat16() * torch.rand(Gn, M, 1, device='cuda').bfloat16() * 4
    b = (torch.randn(Gn, N, K, device='cuda') * 0.1).bfloat16()
    bias = torch.randn(Gn, N, device='cuda').bfloat16()
    aq, sa = G.quantize_rows(a)
    bq, sb = G.quantize_rows(b)
    assert aq.dtype == torch.float8_e4m3fn and sa.shape == (Gn, M)
    deq = aq.float() * sa.unsqueeze(-1)
    assert (deq - a.float()).abs().max() <= a.float().abs().amax() * 0.07
    d = G.raw_gemm(aq, bq, epilogue=G.EPI_BIAS_RELU, bias=bias, out_dtype=torch.bfloat16, scale_a=sa, scale_b=sb, cta_group=cg)
    ref_q = torch.relu(torch.matmul(deq, (bq.float() * sb.unsqueeze(-1)).transpose(1, 2)) + bias.float().unsqueeze(1))
    assert torch.allclose(d.float(), ref_q, atol=0.06, rtol=2e-2)          # exact up to bf16 output rounding
    ref = torch.relu(torch.matmul(a.float(), b.float().transpose(1, 2)) + bias.float().unsqueeze(1))
    assert (d.float() - ref).norm() / ref.norm() < 0.06                    # quantisation error budget


def test_fp8_forward_layer_close_to_bf16():
    from tutel_b200 import moe
    def build(fp8):
        torch.manual_seed(0)
        return moe.moe_layer(gate_type={'type': 'top', 'k': 2}, model_dim=256, seeds=(1, 1, 1),
                             experts={'type': 'ffn', 'num_experts_per_device': 4, 'hidden_size_per_expert': 512,
                                      'activation_fn': lambda t: F.relu(t), 'fp8': fp8}).cuda().bfloat16()
    a, b = build(False), build(True)
    x = torch.randn(4, 128, 256, device='cuda', dtype=torch.bfloat16)
    xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    ya, yb = a(xa), b(xb)
    assert (yb.float() - ya.float()).norm() / ya.float().norm() < 0.08
    ya.float().pow(2).mean().backward()
    yb.float().pow(2).mean().backward()
    assert (xb.grad.float() - xa.grad.float()).norm() / xa.grad.float().norm() < 0.15


def _act(name, t):
    return {'relu': torch.relu, 'silu': F.silu, 'gelu': F.gelu}[name](t)


@pytest.mark.parametrize('act', ['silu', 'relu', 'gelu'])
@pytest.mark.parametrize('M,b_mn', [(96, True), (328, True), (328, False), (1000, True)])
def test_glu_dual_b_gemm_forward_and_backward_epilogues(C, act, M, b_mn):
    """h = act(x@W1) * (x@W2) from ONE launch (gate/up halves share a TMEM tile), and the dh GEMM that emits dg/du."""
    from tutel_b200.ops import gemm as G
    torch.manual_seed(3)
    Gn, K, N = 2, 264, 328          # N not a multiple of the 128-column half tile
    x = (torch.randn(Gn, M, K, device='cuda') * 0.5).bfloat16()
    w1 = (torch.randn(Gn, K, N, device='cuda') * 0.1).bfloat16()
    w2 = (torch.randn(Gn, K, N, device='cuda') * 0.1).bfloat16()
    b1 = w1 if b_mn else w1.transpose(1, 2).contiguous()
    b2 = w2 if b_mn else w2.transpose(1, 2).contiguous()
    h, g, u = G.glu_gemm(x, b1, b2, b_mn=b_mn, act=act, save_pre=True)
    g_ref, u_ref = x.float() @ w1.float(), x.float() @ w2.float()
    assert torch.allclose(g.float(), g_ref, atol=0.05, rtol=2e-2)
    assert torch.allclose(u.float(), u_ref, atol=0.05, rtol=2e-2)
    assert torch.allclose(h.float(), _act(act, g_ref) * u_ref, atol=0.05, rtol=3e-2)
    h_only, _, _ = G.glu_gemm(x, b1, b2, b_mn=b_mn, act=act)
    assert torch.equal(h_only, h)

    # backward epilogue: dh = dy @ W3^T stays in TMEM, the epilogue writes dg and du
    Mo = 136
    dy = (torch.randn(Gn, M, Mo, device='cuda') * 0.5).bfloat16()
    w3 = (torch.randn(Gn, N, Mo, device='cuda') * 0.1).bfloat16()
    dg, du = G.glu_gemm_bwd(dy, w3, g, u, b_mn=False, act=act)
    gf = g.float().requires_grad_(True)
    uf = u.float().requires_grad_(True)
    dh = dy.float() @ w3.float().transpose(1, 2)
    (_act(act, gf) * uf).backward(dh)
    assert torch.allclose(dg.float(), gf.grad, atol=0.05, rtol=3e-2)
    assert torch.allclose(du.float(), uf.grad, atol=0.05, rtol=3e-2)


@pytest.mark.parametrize('act', ['silu', 'relu'])
@pytest.mark.parametrize('fp8', [False, True])
def test_llama_ffn_expert_fused_glu_matches_autograd(act, fp8):
    """The llama_ffn expert (reference tutel/experts/llama_ffn.py) through the fused GLU path vs plain fp32 autograd."""
    from tutel_b200.ops import gemm as G
    torch.manual_seed(5)
    Gn, T, M, H = 2, 512, 256, 384
    x = (torch.randn(Gn, T, M, device='cuda') * 0.5).bfloat16().requires_grad_(True)
    ws = [(torch.randn(Gn, *s, device='cuda') * 0.05).bfloat16().requires_grad_(True) for s in ((M, H), (M, H), (H, M))]
    y = G.fused_glu_ffn(x, *ws, act, fp8)
    dy = (torch.randn_like(y) * 0.1)
    y.backward(dy)
    xr = x.detach().float().requires_grad_(True)
    wr = [w.detach().float().requires_grad_(True) for w in ws]
    yr = (_act(act, xr @ wr[0]) * (xr @ wr[1])) @ wr[2]
    yr.backward(dy.float())
    def rel(a, b):
        return ((a.float() - b).norm() / b.norm()).item()
    errs = [rel(y, yr), rel(x.grad, xr.grad)] + [rel(w.grad, r.grad) for w, r in zip(ws, wr)]
    if fp8:     # e4m3 forward: ~4 % per GEMM; its pre-activations also decide the ReLU mask used in backward
        assert errs[0] < 0.1 and max(errs) < 0.3, errs
    else:       # bf16: rounding of the saved activations
        assert max(errs) < 0.02, errs


