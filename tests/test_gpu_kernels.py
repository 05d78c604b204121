"""Kernel-level parity (GPU): every exported kernel entry point of libhh_b200.so against a plain PyTorch fp32
statement of the same op (the floating-point counterpart of the oracle), through the C ABI.

Tolerances: kernels that take bf16 operands are compared on the SAME bf16-rounded inputs, so what is left is the fp32
accumulation order and the bf16 rounding of the output (rel 2^-8); fp32 kernels use 1e-5 relative; the box kernels are
bit-exact."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from oracle import hh_oracle as O  # noqa: E402


def _ops():
    from helping_hand_for_egocentric_videos_b200 import ops
    return ops


def _rand(*shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).cuda()


def _close(got, want, rtol, atol, name=""):
    got, want = got.float(), want.float()
    err = (got - want).abs()
    lim = atol + rtol * want.abs()
    bad = err > lim
    assert not bad.any(), "%s: %d/%d out of tolerance, max err %.3e (ref scale %.3e)" % (
        name, int(bad.sum()), bad.numel(), err.max().item(), want.abs().max().item())


GEMM_SHAPES = [
    (128, 256, 64), (300, 3072, 1024), (4097, 1024, 1024), (1000, 4096, 1024), (515, 1024, 4096),
    (777, 768, 768), (260, 2304, 768), (1568, 1024, 640), (100, 22048, 512), (4100, 6144, 512), (65, 128, 128),
    (129, 96, 72), (1, 8, 8),
    # M >= 74 row tiles: CTA-pair path (W tile multicast across a 2-CTA cluster); odd and even tile counts, ragged tails
    (9600, 512, 256), (9601, 1024, 1024), (12288, 3072, 128), (20000, 256, 4096), (9473, 384, 64),
]


@pytest.mark.parametrize("M,N,K", GEMM_SHAPES)
@pytest.mark.parametrize("epi", [0, 1, 2, 3])
def test_gemm_tcgen05(M, N, K, epi):
    ops = _ops()
    if epi in (0, 1) and N % 2:
        pytest.skip("bf16 output needs even N")
    a = _rand(M, K, seed=1).bfloat16()
    w = _rand(N, K, seed=2, scale=1 / math.sqrt(K)).bfloat16()
    bias = _rand(N, seed=3, scale=0.5)
    res = _rand(M, N, seed=4) if epi == 2 else None
    ref = a.float() @ w.float().t() + bias
    if epi == 1:
        ref = O.quick_gelu(ref)
    if epi == 2:
        ref = ref + res
    got = ops.gemm_bf16(a, w, bias, epilogue=epi, residual=res)
    if epi in (0, 1):
        _close(got, ref, 2 ** -7, 2e-3, "gemm epi%d" % epi)
    else:
        _close(got, ref, 1e-4, 2e-4, "gemm epi%d" % epi)


def test_gemm_no_bias_and_inplace_residual():
    ops = _ops()
    a = _rand(333, 256, seed=5).bfloat16()
    w = _rand(512, 256, seed=6, scale=1 / 16).bfloat16()
    x = _rand(333, 512, seed=7)
    want = x + a.float() @ w.float().t()
    got = ops.gemm_bf16(a, w, None, epilogue=2, residual=x, out=x)      # x <- x + a w^T, in place
    assert got.data_ptr() == x.data_ptr()
    _close(got, want, 1e-4, 2e-4, "in-place residual")


def test_gemm_is_deterministic():
    ops = _ops()
    a = _rand(2000, 1024, seed=8).bfloat16()
    w = _rand(1024, 1024, seed=9, scale=1 / 32).bfloat16()
    r1 = ops.gemm_bf16(a, w, None, epilogue=3)
    r2 = ops.gemm_bf16(a, w, None, epilogue=3)
    assert torch.equal(r1, r2)


def test_gemm_rejects_bad_arguments():
    ops = _ops()
    a = _rand(16, 12, seed=1).bfloat16()      # K = 12: not a multiple of 8
    w = _rand(8, 12, seed=2).bfloat16()
    with pytest.raises(RuntimeError, match="multiples of 8"):
        ops.gemm_bf16(a, w)


@pytest.mark.parametrize("M,D", [(1, 128), (37, 512), (4097, 1024), (785, 768)])
def test_layernorm(M, D):
    ops = _ops()
    x = _rand(M, D, seed=10, scale=3.0) + 0.7
    w = 1 + 0.1 * _rand(D, seed=11)
    b = 0.1 * _rand(D, seed=12)
    for eps in (1e-5, 1e-6):
        o32, o16 = ops.layernorm(x, w, b, eps, want_f32=True, want_bf16=True)
        ref = F.layer_norm(x, (D,), w, b, eps)
        _close(o32, ref, 1e-5, 1e-5, "ln f32")
        _close(o16, ref, 2 ** -8, 1e-3, "ln bf16")


def _ref_attention(qkv, B, T, n, H, mode):
    """Masked dense attention on the packed (already bf16-rounded, q pre-scaled) qkv."""
    N = 1 + T * n
    D = H * 64
    q, k, v = qkv.float().view(B, N, 3, H, 64).permute(2, 0, 3, 1, 4)
    s = q @ k.transpose(-1, -2)
    s = s.masked_fill(~O._group_mask(T, n, mode).to(s.device), float("-inf"))
    return (torch.softmax(s, -1) @ v).permute(0, 2, 1, 3).reshape(B * N, D)


@pytest.mark.parametrize("B,T,n,H", [(2, 3, 16, 2), (1, 4, 196, 12), (2, 16, 256, 2), (1, 4, 256, 16), (3, 1, 4, 1),
                                     (1, 2, 50, 3), (1, 32, 16, 4), (1, 8, 64, 5), (1, 2, 300, 2)])
def test_divided_attention(B, T, n, H):
    """n > 256 runs the spatial mma.sync kernel instead of the tcgen05 one; T other than 4 / 8 / 16 runs the runtime-T
    temporal kernel, T > 16 the SIMT one."""
    ops = _ops()
    N = 1 + T * n
    qkv = _rand(B * N, 3 * H * 64, seed=20, scale=1.0)
    qkv[:, :H * 64] *= 0.35            # plausible pre-scaled q magnitude
    qkv = qkv.bfloat16()
    outs = ops.attention(qkv, B, T, n, H)
    alone = ops.attention(qkv, B, T, n, H, standalone_cls=True)
    for mode in ("space", "time"):
        ref = _ref_attention(qkv, B, T, n, H, mode)
        # P is rounded to bf16 before P.V in the tensor-core kernel: allow 2^-7 relative on O(1) outputs
        _close(outs[mode], ref, 2 ** -6, 6e-3, "attention %s" % mode)
        _close(alone[mode], ref, 2 ** -6, 6e-3, "attention %s (stand-alone CLS row)" % mode)
        cls_rows = torch.arange(B, device=qkv.device) * N
        # the CLS query sees all N keys: its output is a near-uniform average, so check it on its own scale
        _close(outs[mode][cls_rows], ref[cls_rows], 2 ** -6, 1e-3, "CLS row %s" % mode)


@pytest.mark.parametrize("B,T,n,H", [(3, 16, 256, 16), (5, 4, 196, 12)])
def test_attention_kernels_are_deterministic_under_stress(B, T, n, H):
    """500 launches of both attention kernels on the same input, more tasks than SMs (several tasks per persistent CTA,
    both pipeline stages and both TMEM halves recycled many times): every launch must reproduce the first one bit for
    bit.  The spatial kernel orders its shared-memory / TMEM hand-overs with mbarriers that racecheck cannot model
    (profiles/r1_compute_sanitizer_racecheck.md); a missed hand-over shows up here as a differing launch."""
    lib, L = _ops().L.load(), _ops().L
    N = 1 + T * n
    qkv = _rand(B * N, 3 * H * 64, seed=77, scale=1.0)
    qkv[:, :H * 64] *= 0.35
    qkv = qkv.bfloat16()
    for kind in (0, 1):
        first = None
        o = torch.empty(B * N, H * 64, dtype=torch.bfloat16, device="cuda")
        bad = 0
        for i in range(500):
            o.fill_(float("nan"))
            L.check(lib.hh_attention(L.ptr(qkv), L.ptr(o), B, T, n, H, kind, L.stream_ptr()), "hh_attention")
            if first is None:
                first = o.clone()
                assert torch.isfinite(first.float()).all()
                _close(first, _ref_attention(qkv, B, T, n, H, "space" if kind == 0 else "time"), 2 ** -6, 6e-3, "stress ref")
            elif i % 10 == 0 or i > 480:          # compare on the device, without a host sync per launch
                bad += int((o.view(torch.int16) != first.view(torch.int16)).any())
        assert bad == 0, "attention kind %d: %d launches differ from the first" % (kind, bad)


@pytest.mark.parametrize("G,Lc,H", [(3, 77, 8), (2, 77, 12), (5, 16, 2), (2, 33, 4), (1, 130, 2), (4, 1, 2)])
def test_causal_attention(G, Lc, H):
    """Text-tower attention core against dense masked softmax (nn.MultiheadAttention + triu(-inf) mask,
    reference model/openai_model.py:199-201) on the same bf16-rounded, pre-scaled qkv."""
    g = torch.Generator().manual_seed(G * 1000 + Lc)
    qkv = (torch.randn(G * Lc, 3 * H * 64, generator=g) * 0.7)
    qkv[:, :H * 64] *= 0.125
    qkv = qkv.to(torch.bfloat16).cuda()
    got = _ops().attention_causal(qkv, G, Lc, H)
    x = qkv.float().view(G, Lc, 3, H, 64).permute(2, 0, 3, 1, 4)
    s = x[0] @ x[1].transpose(-1, -2) + torch.full((Lc, Lc), float("-inf"), device="cuda").triu_(1)
    ref = (torch.softmax(s, -1) @ x[2]).permute(0, 2, 1, 3).reshape(G * Lc, H * 64)
    _close(got, ref, 2 ** -6, 6e-3, "causal attention")


@pytest.mark.parametrize("B,Q,heads,S", [(2, 5, 2, 48), (1, 13, 8, 4096), (3, 13, 8, 784), (2, 16, 1, 100), (1, 1, 2, 31)])
def test_cross_attention(B, Q, heads, S):
    ops = _ops()
    C_ = heads * 64
    q = _rand(B * Q, C_, seed=30, scale=0.3)
    K = _rand(B * S, C_, seed=31).bfloat16()
    V = _rand(B * S, C_, seed=32).bfloat16()
    got = ops.cross_attention(q, K, V, B, Q, heads, S)
    qh = q.view(B, Q, heads, 64).transpose(1, 2)
    kh = K.float().view(B, S, heads, 64).transpose(1, 2)
    vh = V.float().view(B, S, heads, 64).transpose(1, 2)
    ref = (torch.softmax(qh @ kh.transpose(-1, -2), -1) @ vh).transpose(1, 2).reshape(B * Q, C_)
    # P is rounded to bf16 for the P.V tensor-core product (q enters as a bf16 hi+lo pair, so logits are fp32-accurate)
    # With few keys the softmax is peaked (p up to ~0.5), so the bf16 rounding of P costs up to 2^-9 * p * |v| ~ 3e-3.
    _close(got, ref, 2 ** -7, 4e-3, "cross attention")
    simt = ops.cross_attention(q, K, V, B, Q, heads, S, simt=True)     # fp32 SIMT statement of the same kernel
    _close(simt, ref, 1e-4, 2e-5, "cross attention (SIMT)")


@pytest.mark.parametrize("R,N,K", [(13, 512, 512), (832, 2048, 512), (65, 4, 512), (7, 256, 768), (100, 100, 32)])
def test_linear_f32(R, N, K):
    ops = _ops()
    x = _rand(R, K, seed=40)
    w = _rand(N, K, seed=41, scale=1 / math.sqrt(K))
    b = _rand(N, seed=42)
    _close(ops.linear_f32(x, w, b), F.linear(x, w, b), 1e-5, 1e-5, "linear")
    _close(ops.linear_f32(x, w, b, act=1), F.relu(F.linear(x, w, b)), 1e-5, 1e-5, "linear+relu")
    _close(ops.linear_f32(x, w, b, act=2), torch.sigmoid(F.linear(x, w, b)), 1e-5, 1e-5, "linear+sigmoid")
    _close(ops.linear_f32(x, w, None, in_relu=True), F.linear(F.relu(x), w), 1e-5, 1e-5, "relu+linear")


def test_linear_f32_odd_width_and_unaligned_operands():
    """Shapes lin3.cu refuses (odd N) go to the first-generation kernel; operands that are not 16-byte aligned are an
    argument error (both kernels read 16-byte pieces), not a misaligned-address fault."""
    ops = _ops()
    R, N, K = 70, 33, 64
    x, w, b = _rand(R, K, seed=43), _rand(N, K, seed=44, scale=1 / math.sqrt(K)), _rand(N, seed=45)
    _close(ops.linear_f32(x, w, b, act=1), F.relu(F.linear(x, w, b)), 1e-5, 1e-5, "linear (odd N)")
    flat = _rand(R * K + 1, seed=46)
    xu = flat[1:].view(R, K)                       # contiguous, 4 bytes off a 16-byte boundary
    assert xu.data_ptr() % 16 != 0
    with pytest.raises(RuntimeError, match="16-byte aligned"):
        ops.linear_f32(xu, w, b)
    torch.cuda.synchronize()                      # the context is intact
    _close(ops.linear_f32(xu.clone(), w, b), F.linear(xu, w, b), 1e-5, 1e-5, "linear (re-aligned copy)")


def test_sim_matrix_and_reductions():
    ops = _ops()
    a = _rand(70, 256, seed=50)
    b = _rand(133, 256, seed=51)
    a[3] = 0                                # eps clamp (model/metric.py:368-370)
    sim = ops.sim_matrix(a, b)
    _close(sim, O.sim_matrix(a, b), 1e-5, 1e-6, "sim_matrix")
    assert torch.equal(ops.row_argmax(sim), sim.argmax(-1))
    _close(ops.row_softmax(sim, 1 / 0.07), torch.softmax(sim / 0.07, -1), 1e-4, 1e-7, "softmax")
    _close(ops.row_softmax(sim, 1 / 0.07, log=True), torch.log_softmax(sim / 0.07, -1), 1e-5, 1e-5, "log_softmax")
    ties = torch.tensor([[1.0, 3.0, 3.0, 2.0, 3.0], [5.0, 5.0, 5.0, 5.0, 5.0]]).cuda()
    assert ops.row_argmax(ties).tolist() == [1, 0]      # first maximum, like torch.argmax
    _close(ops.l2_normalize(a), F.normalize(a, dim=-1), 1e-6, 1e-7, "l2_normalize")


def test_sim_matrix_large_is_symmetric_and_unit_diagonal():
    """Size-independent properties at the EPIC-MIR scale (BASELINE config 4): sim(a,a) is symmetric with a unit
    diagonal, and every entry is a cosine."""
    ops = _ops()
    a = _rand(9728, 256, seed=52)
    s = ops.sim_matrix(a, a)
    assert (s.diagonal() - 1).abs().max() < 1e-5
    assert (s - s.t()).abs().max() < 1e-6
    assert s.abs().max() <= 1 + 1e-5


def test_box_ops_bit_exact():
    ops = _ops()
    g = torch.Generator().manual_seed(60)
    def rb(k):
        return torch.cat([0.2 + 0.6 * torch.rand(k, 2, generator=g), 0.02 + 0.35 * torch.rand(k, 2, generator=g)], -1)
    p, t = rb(2560), rb(512)
    t[0] = p[3]
    t[1, 2:] = 0
    pc, tc = p.cuda(), t.cuda()
    pxy = ops.box_convert(pc, True)
    assert torch.equal(pxy.cpu(), O.box_cxcywh_to_xyxy(p))
    assert torch.equal(ops.box_convert(pxy, False).cpu(), O.box_xyxy_to_cxcywh(O.box_cxcywh_to_xyxy(p)))
    iou, uni, giou = ops.box_pairwise(pxy, ops.box_convert(tc, True))
    riou, runi = O.box_iou(O.box_cxcywh_to_xyxy(p), O.box_cxcywh_to_xyxy(t))
    rg = O.generalized_box_iou(O.box_cxcywh_to_xyxy(p), O.box_cxcywh_to_xyxy(t))
    assert torch.equal(iou.cpu(), riou) and torch.equal(uni.cpu(), runi)
    assert torch.equal(giou.cpu(), rg)
    cost = ops.box_match_cost(pc, tc)
    _close(cost, O.matcher_cost(p, t).cuda(), 1e-6, 1e-6, "matcher cost")   # cdist's summation order is unspecified
    assert ops.box_convert(torch.empty(0, 4).cuda(), True).shape == (0, 4)   # empty input


def test_hungarian_indices_from_gpu_cost_match_reference_cost():
    """'box index outputs exact': scipy's assignment on our cost equals the assignment on the oracle's cost."""
    from scipy.optimize import linear_sum_assignment
    ops = _ops()
    g = torch.Generator().manual_seed(61)
    for trial in range(20):
        nq, nt = 10, int(torch.randint(1, 5, (1,), generator=g))
        p = torch.cat([0.2 + 0.6 * torch.rand(nq, 2, generator=g), 0.05 + 0.3 * torch.rand(nq, 2, generator=g)], -1)
        t = torch.cat([0.2 + 0.6 * torch.rand(nt, 2, generator=g), 0.05 + 0.3 * torch.rand(nt, 2, generator=g)], -1)
        mine = linear_sum_assignment(ops.box_match_cost(p.cuda(), t.cuda()).cpu().numpy())
        ref = linear_sum_assignment(O.matcher_cost(p, t).numpy())
        assert (mine[0] == ref[0]).all() and (mine[1] == ref[1]).all()


def test_sharded_sim_matrix_single_process():
    """World size 1: the sharded similarity is the plain device scoring kernel (multi-rank host logic: gloo tests)."""
    from helping_hand_for_egocentric_videos_b200 import parallel
    a, b = _rand(9, 256, seed=70), _rand(14, 256, seed=71)
    _close(parallel.sharded_sim_matrix(a, b), O.sim_matrix(a, b), 1e-5, 1e-6, "sharded sim")
