"""GPU: block-scaled FP8 forward (csrc/gemm_fp8.cu) — act_quant and fp8_gemm against the
reference's own compiled Triton kernels (oracle/_ref/, launched by oracle/ref_cubin.py), the CPU
restatement (oracle/fp8_gemm_oracle.py) and exact integer-grid products; the fp8 branches of the
linear modules; a tiny-Llama perplexity against the reference kernels' own self-divergence."""
import json
import os

import pytest
import torch

from oracle import fp8_gemm_oracle as fo
from oracle import ref_cubin

pytestmark = pytest.mark.gpu

needs_ref = pytest.mark.skipif(not ref_cubin.available(),
                               reason='oracle/_ref/ missing: build() compiles the reference kernels '
                                      'only where an llmc checkout and Triton exist')


def _report(name, doc):
    """Measured agreement figures (PARITY.md) go to $LLMC_B200_REPORT_DIR when it is set."""
    out = os.environ.get('LLMC_B200_REPORT_DIR')
    if out:
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, f'fp8_gemm_{name}.json'), 'w') as fh:
            json.dump(doc, fh, indent=1, default=str)


def _act_input(shape, dtype, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(*shape, generator=g) * torch.exp(torch.randn(*shape, generator=g) * 2)
    flat = x.view(-1, 128)
    flat[0::7] *= 3e4           # large blocks
    flat[3::7] *= 1e-4          # tiny blocks
    flat[1] = 0.0               # one all-zero block: s = 0, NaN codes
    return x.to(dtype)


ACT_CASES = [(torch.bfloat16, (64, 1024)), (torch.float16, (4, 33, 512)), (torch.float32, (2, 7, 768))]


@pytest.mark.parametrize('dtype,shape', ACT_CASES)
def test_act_quant_against_ieee_oracle(dtype, shape):
    from llmc_b200.kernel import act_quant
    x = _act_input(shape, dtype, 1)
    y, s = act_quant(x.cuda())
    yo, so = fo.act_quant(x)
    assert y.shape == x.shape and y.dtype == torch.float8_e4m3fn
    assert s.shape == (*shape[:-1], shape[-1] // 128) and s.dtype == torch.float32
    s, y = s.cpu(), y.cpu()
    # scales within 2 ulp of IEEE division, the NaN pattern identical
    assert torch.equal(s == 0, so == 0)
    si, soi = s.view(torch.int32).long(), so.view(torch.int32).long()
    assert (si - soi).abs().max().item() <= 2
    yn, yon = y.float().isnan(), yo.float().isnan()
    assert torch.equal(yn, yon) and yn.any()
    # codes within one e4m3 step (same sign, adjacent magnitudes)
    yb, yob = y.view(torch.uint8).long(), yo.view(torch.uint8).long()
    ok = ~yn
    assert ((yb[ok] - yob[ok]).abs() <= 1).all()
    _report(f'act_quant_vs_ieee_{str(dtype)[6:]}', {
        'blocks': s.numel(), 'scales_differing': int((si != soi).sum()),
        'codes': int(ok.sum()), 'codes_differing': int((yb[ok] != yob[ok]).sum())})


@needs_ref
@pytest.mark.parametrize('dtype,shape', ACT_CASES)
def test_act_quant_bit_identical_to_reference(dtype, shape):
    from llmc_b200.kernel import act_quant
    x = _act_input(shape, dtype, 2).cuda()
    y, s = act_quant(x)
    yr, sr = ref_cubin.act_quant(x)
    assert torch.equal(s.view(torch.int32), sr.view(torch.int32))
    assert torch.equal(y.view(torch.uint8), yr.view(torch.uint8))
    assert y.float().isnan().any()


def test_act_quant_block_size_must_be_128():
    from llmc_b200.kernel import act_quant
    with pytest.raises(NotImplementedError):
        act_quant(torch.zeros(2, 256, device='cuda', dtype=torch.bfloat16), 64)


def _grid_operands(M, N, K, seed):
    """Small-integer fp8 values and power-of-two scales: every partial sum is an fp32 integer
    multiple of a power of two below 2^24, so any summation order gives the same exact result."""
    g = torch.Generator().manual_seed(seed)
    a = torch.randint(-4, 5, (M, K), generator=g).float().to(torch.float8_e4m3fn)
    b = torch.randint(-4, 5, (N, K), generator=g).float().to(torch.float8_e4m3fn)
    a_s = torch.pow(2.0, torch.randint(-3, 4, (M, K // 128), generator=g).float())
    b_s = torch.pow(2.0, torch.randint(-3, 4, (-(-N // 128), K // 128), generator=g).float())
    return a, a_s, b, b_s


@pytest.mark.parametrize('M,N,K', [(1, 576, 256), (77, 200, 384), (300, 576, 512), (256, 256, 128),
                                   (129, 1536, 1024), (1000, 130, 640)])
def test_fp8_gemm_exact_on_integer_grid(M, N, K):
    from llmc_b200.kernel import fp8_gemm_out
    a, a_s, b, b_s = _grid_operands(M, N, K, M + N + K)
    exact, _ = fo.fp8_gemm_exact(a, a_s, b, b_s)
    ref = exact.float()
    assert torch.equal(ref.double(), exact)               # representable
    args = [t.cuda() for t in (a, a_s, b, b_s)]
    for dt in (torch.float32, torch.bfloat16, torch.float16):
        c = fp8_gemm_out(*args, dt)
        assert c.dtype == dt and c.shape == (M, N)
        assert torch.equal(c.cpu(), ref.to(dt)), dt


def _random_operands(M, N, K, seed):
    g = torch.Generator().manual_seed(seed)
    x = (torch.randn(M, K, generator=g) * torch.exp(torch.randn(K, generator=g))).bfloat16()
    w = torch.randn(N, K, generator=g) * 0.02
    from oracle import fp8_oracle
    wq, ws = fp8_oracle.block_quant(w, 'e4m3', 128)
    a, a_s = fo.act_quant(x)
    return a, a_s, wq, ws


GEMM_SHAPES = [(256, 576, 7168), (512, 1536, 7168), (77, 200, 384)]


@pytest.mark.parametrize('M,N,K', GEMM_SHAPES)
def test_fp8_gemm_within_fp64_bound(M, N, K):
    from llmc_b200.kernel import fp8_gemm
    a, a_s, b, b_s = _random_operands(M, N, K, 5)
    c = fp8_gemm(*[t.cuda() for t in (a, a_s, b, b_s)]).cpu()
    exact, bound = fo.fp8_gemm_exact(a, a_s, b, b_s)
    assert c.dtype == torch.float32
    assert ((c.double() - exact).abs() <= bound).all()
    c32 = fo.fp8_gemm(a, a_s, b, b_s)
    assert ((c32.double() - exact).abs() <= bound).all()


@needs_ref
@pytest.mark.parametrize('M,N,K', GEMM_SHAPES)
def test_fp8_gemm_within_reference_config_spread(M, N, K):
    from llmc_b200.kernel import fp8_gemm
    a, a_s, b, b_s = [t.cuda() for t in _random_operands(M, N, K, 6)]
    c = fp8_gemm(a, a_s, b, b_s)
    refs = {cfg[0]: (ref_cubin.fp8_gemm(a, a_s, b, b_s, cfg[0]), cfg[4])
            for cfg in ref_cubin.gemm_configs(N, K)}
    assert len(refs) == 36
    stack = torch.stack([r for r, _ in refs.values()])
    spread = (stack.max(0).values - stack.min(0).values).max().item()
    worst = max((c - r).abs().max().item() for r, _ in refs.values())
    tc = [r for r, kind in refs.values() if kind == 'tcgen05']
    same_tc = [torch.equal(c, r) for r in tc]
    frac_tc = [(c == r).float().mean().item() for r in tc]
    _report(f'gemm_vs_ref_{M}x{N}x{K}', {
        'spread_max_over_configs': spread, 'ours_max_dev_from_any_config': worst,
        'tcgen05_configs': len(tc), 'tcgen05_configs_bit_identical': sum(same_tc),
        'fraction_bit_identical_per_tcgen05_config': frac_tc,
        'mma_sync_configs': sum(1 for _, k in refs.values() if k == 'mma.sync')})
    assert spread > 0.0
    assert worst <= spread, (worst, spread)
    # same per-K-block promotion as the reference's tcgen05 code: bit-identical to every such config
    assert len(tc) == 12 and all(same_tc)
    exact, bound = fo.fp8_gemm_exact(a.cpu(), a_s.cpu(), b.cpu(), b_s.cpu())
    assert ((c.cpu().double() - exact).abs() <= bound).all()


@pytest.mark.parametrize('bias_dtype', [None, torch.float32, torch.bfloat16])
def test_bf16_and_bias_epilogue(bias_dtype):
    from llmc_b200.kernel import fp8_gemm_out
    M, N, K = 200, 576, 1024
    a, a_s, b, b_s = [t.cuda() for t in _random_operands(M, N, K, 8)]
    bias = None
    if bias_dtype is not None:
        bias = torch.randn(N, generator=torch.Generator().manual_seed(9)).to(bias_dtype).cuda()
    y = fp8_gemm_out(a, a_s, b, b_s, torch.bfloat16, bias)
    y_ref = fp8_gemm_out(a, a_s, b, b_s, torch.float32).to(torch.bfloat16)
    if bias is not None:
        y_ref += bias
    assert y.dtype == torch.bfloat16 and torch.equal(y, y_ref)


@needs_ref
def test_bias_epilogue_matches_reference_composition():
    from llmc_b200.kernel import fp8_gemm_out
    M, N, K = 512, 1536, 7168
    a, a_s, b, b_s = [t.cuda() for t in _random_operands(M, N, K, 10)]
    bias = torch.randn(N, generator=torch.Generator().manual_seed(11)).cuda()
    y = fp8_gemm_out(a, a_s, b, b_s, torch.bfloat16, bias)
    c = fp8_gemm_out(a, a_s, b, b_s, torch.float32)
    tc = [n for n, *_, kind in ref_cubin.gemm_configs(N, K) if kind == 'tcgen05']
    r = ref_cubin.fp8_gemm(a, a_s, b, b_s, tc[0])
    y_r = r.to(torch.bfloat16)
    y_r += bias
    # same composition: wherever the fp32 results agree, the bf16 + bias outputs agree bit for bit
    same = c == r
    assert torch.equal(y[same], y_r[same])


def test_argument_errors():
    from llmc_b200 import _lib
    from llmc_b200.kernel import fp8_gemm, fp8_gemm_out
    a = torch.zeros(4, 200, device='cuda', dtype=torch.float8_e4m3fn)
    with pytest.raises(_lib.LlmcB200Error, match='multiple of 128'):
        fp8_gemm(a, torch.ones(4, 1, device='cuda'), a, torch.ones(1, 1, device='cuda'))
    a = torch.zeros(4, 256, device='cuda', dtype=torch.float8_e4m3fn)
    s = torch.ones(4, 2, device='cuda')
    with pytest.raises(_lib.LlmcB200Error, match='bias needs a bf16 output'):
        fp8_gemm_out(a, s, a, s, torch.float32, torch.zeros(4, device='cuda'))


def _fp8_linear(N, K, bias, seed):
    from llmc_b200.module_utils import LlmcFp8Linear
    from llmc_b200.quant_float import weight_cast_to_fp8
    g = torch.Generator().manual_seed(seed)
    lin = torch.nn.Linear(K, N, bias=bias)
    m = LlmcFp8Linear.new(lin, 128).cuda()
    w = (torch.randn(N, K, generator=g) * 0.05).bfloat16().cuda()
    m.weight.data, m.weight_scale_inv.data = weight_cast_to_fp8(w, 128)
    if bias:
        m.bias.data = torch.randn(N, generator=g).cuda()
    return m


@pytest.mark.parametrize('bias', [False, True])
def test_llmc_fp8_linear_switch_on(monkeypatch, bias):
    from llmc_b200 import module_utils as mu
    monkeypatch.setattr(mu, 'USE_FP8GEMM_TRITON_KERNEL', True)
    m = _fp8_linear(576, 512, bias, 1)
    x = torch.randn(3, 40, 512, generator=torch.Generator().manual_seed(2)).bfloat16().cuda()
    y = m(x)
    assert m.weight.dtype == torch.float8_e4m3fn
    assert y.shape == (3, 40, 576) and y.dtype == torch.bfloat16
    assert torch.equal(y, mu.block_wise_fp8_forward_func(x, m.weight, m.weight_scale_inv, 128, m.bias))
    # block_wise_fp8_forward_func is the reference's composition of the two kernels
    from llmc_b200.kernel import act_quant, fp8_gemm
    xq, xs = act_quant(x)
    y2 = fp8_gemm(xq, xs, m.weight, m.weight_scale_inv).to(torch.bfloat16)
    if bias:
        y2 += m.bias
    assert torch.equal(y, y2)
    assert 'use_fp8gemm_triton_kernel=True' in repr(m)


def test_wrappers_take_the_fp8_forward():
    from llmc_b200 import module_utils as mu
    m = _fp8_linear(256, 384, True, 3)
    x = torch.randn(2, 16, 384, generator=torch.Generator().manual_seed(4)).bfloat16().cuda()
    want = mu.block_wise_fp8_forward_func(x, m.weight, m.weight_scale_inv, 128, m.bias)
    calls = []

    def w_qdq(module):
        calls.append(1)
        return module.weight.data

    for new in (lambda: mu.OriginFloatLinear.new(m),
                lambda: mu.FakeQuantLinear.new(m, w_qdq, None),
                lambda: mu.EffcientFakeQuantLinear.new(m, w_qdq, None)):
        calls.clear()
        q = new()
        assert q.fp8_forward and q.block_size == 128
        assert q.weight_scale_inv is m.weight_scale_inv
        assert torch.equal(q(x), want)
        assert torch.equal(q(x), want)
        if isinstance(q, mu.FakeQuantLinear):
            assert len(calls) == 1 and q.tmp_weight is not None     # evaluated once, then ignored
        if not isinstance(q, mu.FakeQuantLinear):
            assert 'fp8_forward=True' in repr(q)


@needs_ref
def test_tiny_llama_ppl_within_reference_self_divergence(monkeypatch):
    """Every decoder linear of the tiny Llama as an LlmcFp8Linear (weights from weight_cast_to_fp8),
    switch on; PPL through our kernels vs the same model on the reference cubins of one tcgen05
    config (cfgA) and one mma.sync config (cfgB)."""
    from llmc_b200 import module_utils as mu
    from llmc_b200.quant_float import weight_cast_to_fp8
    from llmc_b200.synth import SynthModel, perplexity
    monkeypatch.setattr(mu, 'USE_FP8GEMM_TRITON_KERNEL', True)
    model = SynthModel('tiny-llama', seed=0, device='cuda')
    for block in model.get_blocks():
        for name, lin in list(model.get_block_linears(block).items()):
            new = mu.LlmcFp8Linear.new(lin, 128).cuda()
            new.weight.data, new.weight_scale_inv.data = weight_cast_to_fp8(lin.weight.data.contiguous(), 128)
            model._set(block, name, new)
    tokens = torch.randint(0, 512, (1, 64 * 8), generator=torch.Generator().manual_seed(4))
    ppl = perplexity(model, tokens, 64, ce_dtype=torch.float32)

    def with_ref(kind):
        def fwd(x, w, w_scale, block_size, bias):
            xq, xs = ref_cubin.act_quant(x)
            N, K = w.shape
            name = [c[0] for c in ref_cubin.gemm_configs(N, K) if c[4] == kind][0]
            y = ref_cubin.fp8_gemm(xq, xs, w, w_scale, name).to(torch.bfloat16)
            if bias is not None:
                y += bias
            return y
        monkeypatch.setattr(mu, 'block_wise_fp8_forward_func', fwd)
        return perplexity(model, tokens, 64, ce_dtype=torch.float32)

    ppl_a, ppl_b = with_ref('tcgen05'), with_ref('mma.sync')
    bar = max(abs(ppl_a - ppl_b), 1e-4 * ppl_a)
    _report('tiny_llama_ppl', {'ours': ppl, 'ref_tcgen05': ppl_a, 'ref_mma_sync': ppl_b, 'bar': bar})
    assert abs(ppl - ppl_a) <= bar, (ppl, ppl_a, ppl_b)
