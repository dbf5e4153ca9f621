"""GPU parity tests of the individual sm_100a kernels, each called THROUGH THE C ABI
(libsome_b200.so via ctypes) and compared with a plain fp32 torch restatement of the same op on the
same (bf16-rounded) inputs.  Tolerances are written at each comparison."""
import ctypes as C

import numpy as np
import pytest
import torch

from some_b200 import _lib

pytestmark = pytest.mark.gpu

DEV = 'cuda'


@pytest.fixture(scope='module')
def lib():
    if not torch.cuda.is_available():
        pytest.skip('needs a CUDA device')
    return _lib.load()


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def bf16_round(t):
    return t.to(torch.bfloat16).float()


def run_gemm(lib, A, W, bias, out, resid, epi, alpha=1.0, ld_out=None):
    """A, W, bias, out, resid: lists (1 or 2 groups) of tensors."""
    g = _lib.GemmArgs()
    groups = len(A)
    g.A, g.W = _lib.pair(*A), _lib.pair(*W)
    g.bias = _lib.pair(*bias) if bias is not None else (C.c_void_p * 2)()
    g.out = _lib.pair(*out)
    g.resid = _lib.pair(*resid) if resid is not None else (C.c_void_p * 2)()
    g.groups, g.M, g.K = groups, A[0].shape[0], A[0].shape[1]
    g.N = W[0].shape[0]
    g.lda = A[0].stride(0)
    g.ld_out = ld_out if ld_out is not None else out[0].stride(0)
    g.epilogue, g.alpha = epi, alpha
    _lib.check(lib.some_gemm(C.byref(g), stream()), 'some_gemm')
    torch.cuda.synchronize()


def glu_unpack_cols(y):
    """inverse of weights.glu_pack_rows on the output columns: [M, 2C] packed -> (out [M, C], gate [M, C])"""
    m, n = y.shape
    y = y.reshape(m, n // 32, 2, 16)
    return y[:, :, 0].reshape(m, n // 2), y[:, :, 1].reshape(m, n // 2)


@pytest.mark.parametrize('m,n,k', [(128, 256, 64), (300, 512, 512), (1000, 2048, 512), (257, 512, 2048),
                                   (4321, 1536, 512), (129, 512, 80)])
def test_gemm_store_bf16(lib, m, n, k):
    torch.manual_seed(m + n + k)
    A = torch.randn(m, k, device=DEV).to(torch.bfloat16)
    W = (torch.randn(n, k, device=DEV) / k ** 0.5).to(torch.bfloat16)
    out = torch.full((m, n), float('nan'), device=DEV, dtype=torch.bfloat16)
    run_gemm(lib, [A], [W], None, [out], None, _lib.EPI_STORE_BF16)
    ref = A.float() @ W.float().t()
    # bf16 output rounding (2^-9 relative) on O(1) values
    torch.testing.assert_close(out.float(), ref, atol=2e-2, rtol=2e-2)


def test_gemm_two_groups_bias_silu(lib):
    torch.manual_seed(1)
    m, n, k = 777, 2048, 512
    A = [torch.randn(m, k, device=DEV).to(torch.bfloat16) for _ in range(2)]
    W = [(torch.randn(n, k, device=DEV) / k ** 0.5).to(torch.bfloat16) for _ in range(2)]
    b = [torch.randn(n, device=DEV) for _ in range(2)]
    out = [torch.full((m, n), float('nan'), device=DEV, dtype=torch.bfloat16) for _ in range(2)]
    run_gemm(lib, A, W, b, out, None, _lib.EPI_SILU_BF16)
    for i in range(2):
        ref = torch.nn.functional.silu(A[i].float() @ W[i].float().t() + b[i])
        torch.testing.assert_close(out[i].float(), ref, atol=2e-2, rtol=2e-2)


def test_gemm_resid_f32_inplace(lib):
    torch.manual_seed(2)
    m, n, k = 515, 512, 2048
    A = [torch.randn(m, k, device=DEV).to(torch.bfloat16) for _ in range(2)]
    W = [(torch.randn(n, k, device=DEV) / k ** 0.5).to(torch.bfloat16) for _ in range(2)]
    b = [torch.randn(n, device=DEV) for _ in range(2)]
    x = [torch.randn(m, n, device=DEV) for _ in range(2)]
    ref = [0.5 * (A[i].float() @ W[i].float().t() + b[i]) + x[i] for i in range(2)]
    run_gemm(lib, A, W, b, x, x, _lib.EPI_RESID_F32, alpha=0.5)
    for i in range(2):
        # fp32 accumulate of bf16 products: only summation-order noise
        torch.testing.assert_close(x[i], ref[i], atol=2e-4, rtol=1e-4)


def test_gemm_glu_epilogues(lib):
    from some_b200.weights import glu_pack_rows
    torch.manual_seed(3)
    m, c, k = 391, 512, 512
    A = torch.randn(m, k, device=DEV).to(torch.bfloat16)
    W = (torch.randn(2 * c, k, device=DEV) / k ** 0.5).to(torch.bfloat16)
    b = torch.randn(2 * c, device=DEV)
    y = A.float() @ W.float().t() + b
    ref = y[:, :c] * torch.sigmoid(y[:, c:])
    Wp, bp = glu_pack_rows(W).contiguous(), glu_pack_rows(b).contiguous()
    out = torch.full((m, c), float('nan'), device=DEV, dtype=torch.bfloat16)
    run_gemm(lib, [A], [Wp], [bp], [out], None, _lib.EPI_GLU_BF16)
    torch.testing.assert_close(out.float(), ref, atol=2e-2, rtol=2e-2)
    x = torch.randn(m, c, device=DEV)
    ref2 = x + ref
    run_gemm(lib, [A], [Wp], [bp], [x], [x], _lib.EPI_GLU_RESID_F32)
    # sigmoid through tanh.approx (~2^-11 relative)
    torch.testing.assert_close(x, ref2, atol=3e-3, rtol=1e-3)


def test_gemm_resid_out_of_place_and_ragged_rows(lib):
    """TMA residual epilogue: resid != out, M not a multiple of 32 (clipped rows must stay untouched)."""
    torch.manual_seed(21)
    m, n, k = 1001, 512, 512
    A = torch.randn(m, k, device=DEV).to(torch.bfloat16)
    W = (torch.randn(n, k, device=DEV) / k ** 0.5).to(torch.bfloat16)
    b = torch.randn(n, device=DEV)
    x = torch.randn(m, n, device=DEV)
    out = torch.full((m + 40, n), 7.0, device=DEV)           # 40 guard rows behind the tensor
    run_gemm(lib, [A], [W], [b], [out[:m]], [x], _lib.EPI_RESID_F32)
    torch.testing.assert_close(out[:m], A.float() @ W.float().t() + b + x, atol=2e-4, rtol=1e-4)
    assert bool((out[m:] == 7.0).all()), 'rows beyond M were written'


def run_gemm_ln(lib, A, W, bias, out, epi, ln_s=None, stats=None, parts=0, resid=None, out_bf16=None, alpha=1.0):
    g = _lib.GemmArgs()
    g.A, g.W, g.bias, g.out = _lib.pair(*A), _lib.pair(*W), _lib.pair(*bias), _lib.pair(*out)
    g.resid = _lib.pair(*resid) if resid is not None else (C.c_void_p * 2)()
    g.ln_s = _lib.pair(*ln_s) if ln_s is not None else (C.c_void_p * 2)()
    g.ln_stats = _lib.pair(*stats) if stats is not None else (C.c_void_p * 2)()
    g.out_bf16 = _lib.pair(*out_bf16) if out_bf16 is not None else (C.c_void_p * 2)()
    g.ln_parts = parts
    g.groups, g.M, g.K, g.N = len(A), A[0].shape[0], A[0].shape[1], W[0].shape[0]
    g.lda, g.ld_out, g.epilogue, g.alpha = A[0].stride(0), out[0].stride(0), epi, alpha
    _lib.check(lib.some_gemm(C.byref(g), stream()), 'some_gemm')
    torch.cuda.synchronize()


@pytest.mark.parametrize('glu', [False, True])
def test_gemm_ln_producer(lib, glu):
    """SOME_EPI_RESID_F32_LN / SOME_EPI_GLU_RESID_F32_LN: same out as the plain residual epilogue + bf16(out) + per-row partial
    (sum x, sum x^2) in the slots of ln_stats (4 slots for N = 512, 8 for the GLU mix)."""
    from some_b200.weights import glu_pack_rows
    torch.manual_seed(22 + glu)
    m, c, k = 777, 512, 512
    groups = 2
    A = [torch.randn(m, k, device=DEV).to(torch.bfloat16) for _ in range(groups)]
    n = 2 * c if glu else c
    W = [(torch.randn(n, k, device=DEV) / k ** 0.5).to(torch.bfloat16) for _ in range(groups)]
    b = [torch.randn(n, device=DEV) for _ in range(groups)]
    x = [torch.randn(m, c, device=DEV) * 2 + 0.7 for _ in range(groups)]
    ref = []
    for i in range(groups):
        y = A[i].float() @ W[i].float().t() + b[i]
        ref.append(x[i] + (y[:, :c] * torch.sigmoid(y[:, c:]) if glu else 0.5 * y))
    Wk = [glu_pack_rows(w).contiguous() for w in W] if glu else W
    bk = [glu_pack_rows(v).contiguous() for v in b] if glu else b
    xb = [torch.full((m, c), float('nan'), device=DEV, dtype=torch.bfloat16) for _ in range(groups)]
    stats = [torch.full((m, _lib.LN_SLOTS, 2), float('nan'), device=DEV) for _ in range(groups)]
    run_gemm_ln(lib, A, Wk, bk, x, _lib.EPI_GLU_RESID_F32_LN if glu else _lib.EPI_RESID_F32_LN, stats=stats, resid=x,
                out_bf16=xb, alpha=1.0 if glu else 0.5)
    parts = 8 if glu else 4
    for i in range(groups):
        torch.testing.assert_close(x[i], ref[i], atol=3e-3 if glu else 2e-4, rtol=1e-3)
        assert torch.equal(xb[i], x[i].to(torch.bfloat16)), 'out_bf16 is not the bf16 rounding of out'
        st = stats[i][:, :parts]
        assert not torch.isnan(st).any()
        width = c // parts
        cols = x[i].reshape(m, parts, width)
        torch.testing.assert_close(st[:, :, 0], cols.sum(-1), atol=1e-3, rtol=1e-5)
        torch.testing.assert_close(st[:, :, 1], (cols * cols).sum(-1), atol=1e-2, rtol=1e-5)


@pytest.mark.parametrize('kind,parts', [('store', 4), ('silu', 1), ('glu', 8)])
def test_gemm_ln_consumer(lib, kind, parts):
    """SOME_EPI_LN_*: LayerNorm(x) . W^T + bias evaluated from bf16(x), W' = W * gamma, ln_s, b' and the partial row sums."""
    from some_b200.weights import glu_pack_rows
    torch.manual_seed(30 + parts)
    m, k = 1000, 512
    n = {'store': 1536, 'silu': 2048, 'glu': 1024}[kind]
    x = [torch.randn(m, k, device=DEV) * 1.7 + 0.4 for _ in range(2)]
    gamma = [torch.rand(k, device=DEV) * 0.4 + 0.8 for _ in range(2)]
    beta = [torch.randn(k, device=DEV) * 0.05 for _ in range(2)]
    W = [torch.randn(n, k, device=DEV) / k ** 0.5 for _ in range(2)]
    b = [torch.randn(n, device=DEV) for _ in range(2)]
    pack = glu_pack_rows if kind == 'glu' else (lambda t: t)
    xb, Wf, s, bf, stats, ref = [], [], [], [], [], []
    for i in range(2):
        xb.append(x[i].to(torch.bfloat16))
        wf = pack(W[i] * gamma[i][None, :]).to(torch.bfloat16).contiguous()
        Wf.append(wf)
        s.append(wf.double().sum(1).float().contiguous())
        bf.append(pack((W[i].double() @ beta[i].double() + b[i].double()).float()).contiguous())
        st = torch.full((m, _lib.LN_SLOTS, 2), float('nan'), device=DEV)
        cols = x[i].reshape(m, parts, k // parts)
        st[:, :parts, 0], st[:, :parts, 1] = cols.sum(-1), (cols * cols).sum(-1)
        stats.append(st)
        y = torch.nn.functional.layer_norm(x[i], (k,), gamma[i], beta[i], 1e-5) @ W[i].t() + b[i]
        ref.append({'store': y, 'silu': torch.nn.functional.silu(y), 'glu': y[:, :n // 2] * torch.sigmoid(y[:, n // 2:])}[kind])
    nout = n // 2 if kind == 'glu' else n
    out = [torch.full((m, nout), float('nan'), device=DEV, dtype=torch.bfloat16) for _ in range(2)]
    epi = {'store': _lib.EPI_LN_STORE_BF16, 'silu': _lib.EPI_LN_SILU_BF16, 'glu': _lib.EPI_LN_GLU_BF16}[kind]
    run_gemm_ln(lib, xb, Wf, bf, out, epi, ln_s=s, stats=stats, parts=parts)
    for i in range(2):
        # bf16 operands (x and W * gamma) + bf16 output against the fp32 LayerNorm -> Linear: ~1e-2 on O(1) values
        torch.testing.assert_close(out[i].float(), ref[i], atol=4e-2, rtol=3e-2)
        assert float((out[i].float() - ref[i]).abs().mean()) < 6e-3


def test_row_stats(lib):
    torch.manual_seed(40)
    m = 1003
    x = [torch.randn(m, 512, device=DEV) * 2 - 0.3 for _ in range(2)]
    xb = [torch.empty(m, 512, device=DEV, dtype=torch.bfloat16) for _ in range(2)]
    st = [torch.full((m, _lib.LN_SLOTS, 2), float('nan'), device=DEV) for _ in range(2)]
    a = _lib.RowStatsArgs()
    a.x, a.out_bf16, a.ln_stats, a.groups, a.M = _lib.pair(*x), _lib.pair(*xb), _lib.pair(*st), 2, m
    _lib.check(lib.some_row_stats(C.byref(a), stream()), 'some_row_stats')
    torch.cuda.synchronize()
    for i in range(2):
        assert torch.equal(xb[i], x[i].to(torch.bfloat16))
        torch.testing.assert_close(st[i][:, 0, 0], x[i].sum(1), atol=1e-3, rtol=1e-5)
        torch.testing.assert_close(st[i][:, 0, 1], (x[i] * x[i]).sum(1), atol=1e-2, rtol=1e-5)


@pytest.mark.parametrize('normalised', [False, True])
def test_col_means(lib, normalised):
    """some_col_means (load-time bias calibration): column means of a bf16 operand with a row pitch, optionally of the rows
    normalised by LayerNorm statistics split over two slots, against float64 torch; bit-identical from launch to launch."""
    torch.manual_seed(41)
    m, k, lda = 1003, 2048, 2048 + 64
    a = (torch.randn(m, lda, device=DEV) * 2 - 0.3).to(torch.bfloat16)
    x = a[:, :k].double()
    stats = None
    if normalised:
        stats = torch.zeros(m, _lib.LN_SLOTS, 2, device=DEV)
        for s, cols in enumerate((slice(0, k // 2), slice(k // 2, k))):
            stats[:, s, 0] = a[:, cols].float().sum(1)
            stats[:, s, 1] = (a[:, cols].float() ** 2).sum(1)
        mean = x.mean(1, keepdim=True)
        x = (x - mean) * torch.rsqrt((x * x).mean(1, keepdim=True) - mean * mean + 1e-5)
    outs = []
    for _ in range(2):
        out = torch.full((k,), float('nan'), device=DEV)
        _lib.check(lib.some_col_means(a.data_ptr(), m, k, lda, _lib.ptr(stats), 2, out.data_ptr(), stream()), 'some_col_means')
        outs.append(out)
    torch.cuda.synchronize()
    assert torch.equal(outs[0], outs[1])
    torch.testing.assert_close(outs[0].double(), x.mean(0), atol=1e-6, rtol=1e-5)      # fp32 sums of 1003 O(1) values


@pytest.mark.parametrize('n,epi', [(128, 'sigmoid'), (129, 'softmax'), (128, 'logits'), (129, 'logits')])
def test_gemm_heads(lib, n, epi):
    torch.manual_seed(4)
    m, k = 333, 512
    A = torch.randn(m, k, device=DEV).to(torch.bfloat16)
    W = (torch.randn(n, k, device=DEV) / k ** 0.5).to(torch.bfloat16)
    b = torch.randn(n, device=DEV)
    bpad = torch.cat([b, b.new_zeros((-n) % 32)])
    out = torch.full((m, n), float('nan'), device=DEV)
    code = {'sigmoid': _lib.EPI_SIGMOID_F32, 'softmax': _lib.EPI_SOFTMAX_F32, 'logits': _lib.EPI_BIAS_F32}[epi]
    run_gemm(lib, [A], [W], [bpad], [out], None, code)
    y = A.float() @ W.float().t() + b
    ref = {'sigmoid': torch.sigmoid(y), 'softmax': torch.softmax(y, -1), 'logits': y}[epi]
    torch.testing.assert_close(out, ref, atol=2e-4, rtol=2e-4)


def test_layernorm_and_bound_head(lib):
    torch.manual_seed(5)
    m = 1003
    x = [torch.randn(m, 512, device=DEV) * 3 + 1.5 for _ in range(2)]
    g = [torch.rand(512, device=DEV) + 0.5 for _ in range(2)]
    b = [torch.randn(512, device=DEV) * 0.1 for _ in range(2)]
    ob = [torch.empty(m, 512, device=DEV, dtype=torch.bfloat16) for _ in range(2)]
    of = [torch.empty(m, 512, device=DEV) for _ in range(2)]
    a = _lib.LnArgs()
    a.x, a.gamma, a.beta = _lib.pair(*x), _lib.pair(*g), _lib.pair(*b)
    a.out_bf16, a.out_f32, a.groups, a.M = _lib.pair(*ob), _lib.pair(*of), 2, m
    _lib.check(lib.some_layernorm(C.byref(a), stream()))
    torch.cuda.synchronize()
    for i in range(2):
        ref = torch.nn.functional.layer_norm(x[i], (512,), g[i], b[i], 1e-5)
        torch.testing.assert_close(of[i], ref, atol=1e-5, rtol=1e-5)
        torch.testing.assert_close(ob[i].float(), ref, atol=2e-2, rtol=1e-2)   # bf16 rounding
    w = torch.randn(512, device=DEV) / 512 ** 0.5
    bounds = torch.empty(m, device=DEV)
    _lib.check(lib.some_bound_head(x[0].data_ptr(), g[0].data_ptr(), b[0].data_ptr(), w.data_ptr(), 0.3, m,
                                   bounds.data_ptr(), stream()))
    torch.cuda.synchronize()
    ref = torch.sigmoid(torch.nn.functional.layer_norm(x[0], (512,), g[0], b[0], 1e-5) @ w + 0.3)
    torch.testing.assert_close(bounds, ref, atol=1e-5, rtol=1e-5)


def _cu(frames):
    cu = np.zeros(len(frames) + 1, dtype=np.int32)
    np.cumsum(frames, out=cu[1:])
    return torch.from_numpy(cu).to(DEV)


def test_dwconv_bn_silu(lib):
    torch.manual_seed(6)
    frames = [1, 17, 128, 129, 300, 31]
    cu = _cu(frames)
    m = int(cu[-1])
    x = [torch.randn(m, 512, device=DEV).to(torch.bfloat16) for _ in range(2)]
    w = [torch.randn(31, 512, device=DEV) * 0.2 for _ in range(2)]
    b = [torch.randn(512, device=DEV) * 0.1 for _ in range(2)]
    out = [torch.full((m, 512), float('nan'), device=DEV, dtype=torch.bfloat16) for _ in range(2)]
    a = _lib.DwconvArgs()
    a.x, a.w, a.b, a.out = _lib.pair(*x), _lib.pair(*w), _lib.pair(*b), _lib.pair(*out)
    a.groups, a.B, a.cu_frames, a.max_frames = 2, len(frames), cu.data_ptr(), max(frames)
    _lib.check(lib.some_dwconv_bn_silu(C.byref(a), stream()))
    torch.cuda.synchronize()
    for i in range(2):
        r0 = 0
        for t in frames:
            xi = x[i][r0:r0 + t].float().t().unsqueeze(0)                       # [1, 512, t]
            wi = w[i].t().unsqueeze(1)                                          # [512, 1, 31]
            ref = torch.nn.functional.silu(torch.nn.functional.conv1d(xi, wi, b[i], padding=15, groups=512))[0].t()
            torch.testing.assert_close(out[i][r0:r0 + t].float(), ref, atol=3e-2, rtol=2e-2)   # bf16 out
            r0 += t


@pytest.mark.parametrize('impl', ['some_attention_varlen'])
@pytest.mark.parametrize('frames', [[1], [64, 65, 127, 128, 129], [700, 3, 259], [2584]])
def test_attention_varlen(lib, frames, impl):
    torch.manual_seed(7)
    cu = _cu(frames)
    m = int(cu[-1])
    qkv = [(torch.randn(m, 1536, device=DEV) * 1.5).to(torch.bfloat16) for _ in range(2)]
    out = [torch.full((m, 512), float('nan'), device=DEV, dtype=torch.bfloat16) for _ in range(2)]
    a = _lib.AttnArgs()
    a.qkv, a.out = _lib.pair(*qkv), _lib.pair(*out)
    a.groups, a.B, a.M, a.cu_frames, a.max_frames = 2, len(frames), m, cu.data_ptr(), max(frames)
    _lib.check(getattr(lib, impl)(C.byref(a), stream()), impl)
    torch.cuda.synchronize()
    for i in range(2):
        r0 = 0
        for t in frames:
            z = qkv[i][r0:r0 + t].float()
            q, k, v = (z[:, j * 512:(j + 1) * 512].reshape(t, 8, 64).transpose(0, 1) for j in range(3))
            ref = torch.nn.functional.scaled_dot_product_attention(q[None], k[None], v[None])[0]
            ref = ref.transpose(0, 1).reshape(t, 512)
            # P is rounded to bf16 before P.V, output rounded to bf16
            torch.testing.assert_close(out[i][r0:r0 + t].float(), ref, atol=2e-2, rtol=2e-2)
            r0 += t


def test_attention_growing_max_forces_rescale(lib):
    """Scores whose row maximum jumps by far more than 2^8 from one key tile to the next: exercises the lazy
    O-rescale path of the tcgen05 kernel on every tile (a race there shows up as wrong rows)."""
    torch.manual_seed(8)
    frames = [1500, 333]
    cu = _cu(frames)
    m = int(cu[-1])
    qkv = torch.randn(m, 1536, device=DEV) * 0.5
    ramp = torch.cat([torch.arange(t, device=DEV, dtype=torch.float32) / 64.0 for t in frames])   # grows with the key index
    qkv[:, 512:1024] += ramp[:, None] * torch.sign(torch.randn(1, 512, device=DEV))
    qkv[:, :512] = qkv[:, :512].abs() * torch.sign(qkv[0:1, 512:1024] - 0.0 + 1e-3) * 2.0
    qkv = qkv.to(torch.bfloat16)
    out = torch.full((m, 512), float('nan'), device=DEV, dtype=torch.bfloat16)
    a = _lib.AttnArgs()
    a.qkv, a.out = _lib.pair(qkv), _lib.pair(out)
    a.groups, a.B, a.M, a.cu_frames, a.max_frames = 1, len(frames), m, cu.data_ptr(), max(frames)
    for _ in range(3):      # repeat: the failure mode is timing dependent
        out.fill_(float('nan'))
        _lib.check(lib.some_attention_varlen(C.byref(a), stream()))
        torch.cuda.synchronize()
        r0 = 0
        for t in frames:
            z = qkv[r0:r0 + t].float()
            q, k, v = (z[:, j * 512:(j + 1) * 512].reshape(t, 8, 64).transpose(0, 1) for j in range(3))
            ref = torch.nn.functional.scaled_dot_product_attention(q[None], k[None], v[None])[0]
            ref = ref.transpose(0, 1).reshape(t, 512)
            torch.testing.assert_close(out[r0:r0 + t].float(), ref, atol=3e-2, rtol=3e-2)
            r0 += t


@pytest.mark.parametrize('outlier', [200, 206, 519, 1023])
def test_attention_outlier_key_after_the_first_tile(lib, outlier):
    """The exp pass runs against the group's stale reference maximum and a tile is redone only when its row sum gives an
    overflow away (attention_tc.cu).  One key far above everything seen so far -- by more than 2^127 in the exponent, so the
    first attempt produces +inf -- placed in a tile other than a group's first one, at a position handled by the MUFU path
    (key index % 8 < 6) or by the polynomial path (% 8 in {6, 7}, which must clamp instead of wrapping around)."""
    torch.manual_seed(9)
    t = 1100
    cu = _cu([t])
    qkv = torch.randn(t, 1536, device=DEV) * 0.5
    qkv[:, :512] = qkv[:, :512].abs()                         # q > 0, so a key of all + LARGE scores high against every query
    qkv[outlier, 512:1024] = 40.0                             # score ~ 64 * 0.4 * 40 = 1000  ->  1000 / 8 * log2(e) = 180 > 127
    qkv = qkv.to(torch.bfloat16)
    out = torch.full((t, 512), float('nan'), device=DEV, dtype=torch.bfloat16)
    a = _lib.AttnArgs()
    a.qkv, a.out = _lib.pair(qkv), _lib.pair(out)
    a.groups, a.B, a.M, a.cu_frames, a.max_frames = 1, 1, t, cu.data_ptr(), t
    _lib.check(lib.some_attention_varlen(C.byref(a), stream()))
    torch.cuda.synchronize()
    z = qkv.float()
    q, k, v = (z[:, j * 512:(j + 1) * 512].reshape(t, 8, 64).transpose(0, 1) for j in range(3))
    ref = torch.nn.functional.scaled_dot_product_attention(q[None], k[None], v[None])[0].transpose(0, 1).reshape(t, 512)
    assert torch.isfinite(out.float()).all()
    torch.testing.assert_close(out.float(), ref, atol=2e-2, rtol=2e-2)     # every row is (almost) exactly v[outlier]


def test_mel_matches_torch_stft(lib):
    from some_b200 import synth
    from some_b200.engine import Engine
    from some_b200.weights import mel_tables
    cfg = synth.named_config('two_head')
    tabs = mel_tables(cfg, DEV)
    clips = list(synth.edge_case_waveforms().values()) + [synth.synth_waveform(5, seconds=2.0)]
    eng = Engine.__new__(Engine)
    eng.lib, eng.device, eng.mel, eng.launches, eng.prof = lib, torch.device(DEV), tabs, 0, None
    host, tables, cu = Engine.pack(eng, clips)
    b, m = len(clips), int(cu[-1])
    out = torch.full((m, 80), float('nan'), device=DEV)
    outb = torch.empty((m, 80), device=DEV, dtype=torch.bfloat16)
    td = tables.to(DEV)
    eng.run_mel(host.to(DEV), td[:b], td[b:], torch.from_numpy(cu).to(DEV), b, int(np.diff(cu).max()), out, outb)
    torch.cuda.synchronize()
    basis = torch.from_numpy(tabs['bank']).to(DEV)
    for i, w in enumerate(clips):
        wav = torch.from_numpy(w).to(DEV)[None]
        pad = torch.nn.functional.pad(wav, (1024, 1024))
        spec = torch.stft(pad, 2048, 512, 2048, torch.hann_window(2048, device=DEV), center=False, return_complex=True)
        lin = (basis @ spec.abs())[0].t()                                       # [T, 80] linear mel
        got = out[int(cu[i]):int(cu[i + 1])]
        assert got.shape == lin.shape
        # compare in the linear domain relative to the frame's largest band (fp32 FFT round-off), and in the
        # log domain where the band is not buried under the round-off floor
        glin = got.exp()
        scale = lin.max(dim=1, keepdim=True).values.clamp_min(1e-5)
        assert ((glin - lin.clamp_min(1e-5)).abs() / scale).max().item() < 2e-5
        big = lin > 1e-3 * scale
        assert (got - lin.clamp_min(1e-5).log())[big].abs().max().item() < 1e-3 if big.any() else True
        torch.testing.assert_close(outb[int(cu[i]):int(cu[i + 1])].float(), got, atol=4e-2, rtol=1e-2)


def test_decode_matches_oracle(lib, golden_dir):
    """Integer outputs bit-exact, float outputs within 1e-4 of the oracle on identical probs / bounds."""
    from oracle import decode as od
    from some_b200 import synth
    from some_b200.engine import Engine
    gen = torch.Generator().manual_seed(99)
    rb = (torch.rand(4, 700, generator=gen) ** 3)
    rp = (torch.rand(4, 700, 128, generator=gen) ** 6)
    frames = [700, 700, 700, 700, 1, 37]
    probs = torch.cat([rp.reshape(-1, 128), torch.rand(38, 128, generator=gen) * 0.5]).contiguous()
    bounds = torch.cat([rb.reshape(-1), torch.rand(38, generator=gen)]).contiguous()
    cu = _cu(frames)
    m = int(cu[-1])
    cfg = synth.named_config('two_head')
    eng = Engine.__new__(Engine)
    eng.lib, eng.device, eng.config, eng.outdim, eng.launches, eng.prof = lib, torch.device(DEV), cfg, 128, 0, None
    eng.timestep = 512 / 44100
    from some_b200.engine import _Workspace
    ws = _Workspace(m, 128, DEV)
    nc = torch.empty(len(frames), dtype=torch.int32, device=DEV)
    dbg = {}
    eng.run_decode(ws, m, len(frames), cu, nc, False, dbg, probs=probs.to(DEV), bounds=bounds.to(DEV))
    torch.cuda.synchronize()
    g = np.load(golden_dir / 'decode_kat.npz')
    cu_h = cu.cpu().numpy()
    for i, t in enumerate(frames):
        r0 = int(cu_h[i])
        p_i, b_i = probs[r0:r0 + t].numpy(), bounds[r0:r0 + t].numpy()
        f2i = od.decode_bounds_to_alignment(b_i)
        vals, rest = od.decode_gaussian_blurred_probs(p_i, 0, 127, 1.0, 0.1)
        np.testing.assert_array_equal(dbg['frame2item'][r0:r0 + t].cpu().numpy(), f2i)
        np.testing.assert_array_equal(dbg['rest'][r0:r0 + t].cpu().numpy().astype(bool), rest)
        np.testing.assert_allclose(dbg['values'][r0:r0 + t].cpu().numpy(), vals, rtol=0, atol=1e-4)
        if i < 4:   # the reference's own outputs for these inputs (golden)
            np.testing.assert_array_equal(f2i, g['rnd_frame2item'][i])
        nm, nd, nk = od.decode_note_sequence(f2i, dbg['values'][r0:r0 + t].cpu().numpy(), ~rest)
        n = int(nc[i])
        assert n == len(nd)
        np.testing.assert_array_equal(ws.note_dur[r0:r0 + n].cpu().numpy(), nd)
        np.testing.assert_array_equal(ws.note_rest[r0:r0 + n].cpu().numpy().astype(bool), ~nk)
        np.testing.assert_allclose(ws.note_midi[r0:r0 + n].cpu().numpy(), nm, rtol=0, atol=1e-4)
        if i < 4:
            np.testing.assert_array_equal(nd, g[f'rnd_note_dur_{i}'])


def test_decode_quantized_matches_reference_exactly(lib, golden_dir):
    """A18, inference/me_quant_infer.py:21-38: argmax over 129 softmax bins, rest = bin 128, values clip(0, 127); the
    per-note mode / mean run on integers.  Every output of the kernel must equal the oracle AND the reference's own
    postprocess outputs (tests/golden/decode_quant_kat.npz) exactly, including note_midi (integer sums / counts in fp32)."""
    from oracle import decode as od
    from some_b200 import synth
    from some_b200.engine import Engine, _Workspace
    g = np.load(golden_dir / 'decode_quant_kat.npz')
    gen = torch.Generator().manual_seed(77)
    frames = [700, 700, 1, 37]
    probs_l, bounds_l = [], []
    for t in frames:
        logits = torch.randn(1, t, 129, generator=gen) * 2.0
        logits[..., 128] += 1.0
        probs_l.append(torch.softmax(logits, dim=-1)[0])
        bounds_l.append((torch.rand(1, t, generator=gen) ** 3)[0])
    probs, bounds = torch.cat(probs_l).contiguous(), torch.cat(bounds_l).contiguous()
    cu = _cu(frames)
    m = int(cu[-1])
    cfg = synth.named_config('quant_two_head')
    eng = Engine.__new__(Engine)
    eng.lib, eng.device, eng.config, eng.outdim, eng.launches, eng.prof = lib, torch.device(DEV), cfg, 129, 0, None
    eng.timestep = 512 / 44100
    ws = _Workspace(m, 129, DEV)
    nc = torch.empty(len(frames), dtype=torch.int32, device=DEV)
    dbg = {}
    eng.run_decode(ws, m, len(frames), cu, nc, True, dbg, probs=probs.to(DEV), bounds=bounds.to(DEV))
    torch.cuda.synchronize()
    cu_h = cu.cpu().numpy()
    for i, t in enumerate(frames):
        r0 = int(cu_h[i])
        p_i, b_i = probs[r0:r0 + t].numpy(), bounds[r0:r0 + t].numpy()
        midi = p_i.argmax(-1).astype(np.int64)
        f2i = od.decode_bounds_to_alignment(b_i)
        np.testing.assert_array_equal(dbg['frame2item'][r0:r0 + t].cpu().numpy(), f2i)
        np.testing.assert_array_equal(dbg['rest'][r0:r0 + t].cpu().numpy().astype(bool), midi == 128)
        np.testing.assert_array_equal(dbg['values'][r0:r0 + t].cpu().numpy(), np.clip(midi, 0, 127).astype(np.float32))
        nm, nd, nk = od.decode_note_sequence(f2i, np.clip(midi, 0, 127), midi != 128)
        n = int(nc[i])
        assert n == len(nd) == len(g[f'q{i}_note_midi'])
        got_midi = ws.note_midi[r0:r0 + n].cpu().numpy()
        got_dur = ws.note_dur[r0:r0 + n].cpu().numpy()
        got_rest = ws.note_rest[r0:r0 + n].cpu().numpy().astype(bool)
        np.testing.assert_array_equal(got_dur, nd)
        np.testing.assert_array_equal(got_rest, ~nk)
        np.testing.assert_array_equal(got_midi, nm)
        # the unmodified reference's outputs for the same inputs
        np.testing.assert_array_equal(got_midi, g[f'q{i}_note_midi'])
        np.testing.assert_array_equal(got_dur.astype(np.int64) * (512 / 44100), g[f'q{i}_note_dur'])
        np.testing.assert_array_equal(got_rest, g[f'q{i}_note_rest'])


def test_keyshift_mel_matches_reference_golden(golden_dir):
    """some_b200.spec.MelSpectrogram (drop-in for modules/rmvpe/spec.py) on the key-shift / speed / center=False paths
    (direct-DFT kernel some_mel_logmel_keyshift) against the outputs of the unmodified reference (tests/golden/keyshift.npz);
    keyshift = 0 goes through the fused FFT kernel."""
    if not torch.cuda.is_available():
        pytest.skip('needs a CUDA device')
    from some_b200 import synth
    from some_b200.spec import MelSpectrogram
    g = np.load(golden_dir / 'keyshift.npz')
    audio = torch.from_numpy(synth.synth_waveform(int(g['seed']), seconds=float(g['seconds']))).to(DEV)
    mel = MelSpectrogram(80, 44100, 2048, 512, mel_fmin=40, mel_fmax=8000)
    assert np.array_equal(mel.mel_basis.numpy(), np.load(golden_dir / 'mel.npz')['mel_basis'])
    cases = [(f'ks_{k}', dict(keyshift=k)) for k in range(-5, 6)]
    cases += [('ks_frac_2.37', dict(keyshift=2.37)), ('speed_1.25', dict(speed=1.25)), ('nocenter_ks3', dict(keyshift=3, center=False))]
    for key, kw in cases:
        got = mel(audio.unsqueeze(0), **kw)[0].cpu().numpy()
        assert got.shape == g[key].shape, (key, got.shape, g[key].shape)
        # fp32 DFT over <= 2734 terms against torch's FFT; log() amplifies relative errors of near-clamp bands
        err = float(np.abs(got - g[key]).max())
        assert err < 1e-3, (key, err)
    # batched call == per-clip calls
    two = torch.stack([audio, audio.flip(0)])
    b = mel(two, keyshift=-3)
    assert torch.equal(b[0], mel(audio.unsqueeze(0), keyshift=-3)[0])
    assert torch.equal(b[1], mel(audio.flip(0).unsqueeze(0), keyshift=-3)[0])
