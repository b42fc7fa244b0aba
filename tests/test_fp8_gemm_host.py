"""CPU: the block-scaled FP8 forward's argument checks (C ABI and Python), the fp32 oracle against
the reference's fp8_gemm_kernel run under Triton's interpreter (tests/golden/fp8_gemm_kat.pt), and,
where oracle/_ref/ was built, the instructions the reference's compiled act_quant uses."""
import ctypes
import os

import pytest
import torch

from oracle import fp8_gemm_oracle as fo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_c_abi_rejects_bad_arguments_before_any_cuda_call():
    from llmc_b200 import _lib
    lib = _lib.load()
    p, null = ctypes.c_void_p(256), ctypes.c_void_p(0)

    def last():
        return lib.llmc_b200_last_error().decode()

    assert lib.llmc_fp8_gemm(p, p, p, p, null, 0, p, 0, 64, 64, 200, null) == -1
    assert 'K=200 must be a multiple of 128' in last()
    assert lib.llmc_fp8_gemm(p, null, p, p, null, 0, p, 0, 64, 64, 256, null) == -1
    assert 'null pointer' in last()
    assert lib.llmc_fp8_gemm(p, p, p, p, p, 0, p, 0, 64, 64, 256, null) == -1
    assert 'bias needs a bf16 output' in last()
    assert lib.llmc_fp8_gemm(p, p, p, p, p, 1, p, 2, 64, 64, 256, null) == -1
    assert 'bias_dtype' in last()
    assert lib.llmc_fp8_gemm(p, p, p, p, null, 0, p, 7, 64, 64, 256, null) == -1
    assert 'out_dtype' in last()
    assert lib.llmc_fp8_gemm(null, null, null, null, null, 0, null, 0, 0, 64, 256, null) == 0
    assert lib.llmc_fp8_act_quant(p, 4, 100, 2, p, p, null) == -1
    assert 'K=100 must be a multiple of 128' in last()
    assert lib.llmc_fp8_act_quant(null, 4, 128, 2, p, p, null) == -1
    assert 'null pointer' in last()
    assert lib.llmc_fp8_act_quant(p, 4, 128, 5, p, p, null) == -1
    assert lib.llmc_fp8_act_quant(null, 0, 128, 2, null, null, null) == 0


def test_python_entry_points_follow_the_reference_asserts():
    from llmc_b200.kernel import act_quant, fp8_gemm
    with pytest.raises(NotImplementedError, match='only 128'):
        act_quant(torch.zeros(2, 256, dtype=torch.bfloat16), 64)
    with pytest.raises(AssertionError, match='divisible by block_size'):
        act_quant(torch.zeros(2, 200, dtype=torch.bfloat16))
    with pytest.raises(AssertionError, match='contiguous'):
        act_quant(torch.zeros(256, 2, dtype=torch.bfloat16).t())
    a = torch.zeros(256, 4, dtype=torch.float8_e4m3fn).t()
    with pytest.raises(AssertionError, match='contiguous'):
        fp8_gemm(a, torch.ones(4, 2), torch.zeros(8, 256, dtype=torch.float8_e4m3fn), torch.ones(1, 2))


def test_oracle_matches_reference_interpreter_golden():
    kat = torch.load(os.path.join(ROOT, 'tests', 'golden', 'fp8_gemm_kat.pt'))
    assert len(kat['cases']) >= 3
    for case in kat['cases']:
        a = case['a'].view(torch.float8_e4m3fn)
        b = case['b'].view(torch.float8_e4m3fn)
        exact, bound = fo.fp8_gemm_exact(a, case['a_s'], b, case['b_s'])
        ours = fo.fp8_gemm(a, case['a_s'], b, case['b_s'])
        assert ((ours.double() - exact).abs() <= bound).all()
        for cfg, c in case['c'].items():
            assert c.shape == (case['M'], case['N'])
            assert ((c.double() - exact).abs() <= bound).all(), cfg
            # a summation-order difference only: a few fp32 ulps of the promoted sum
            assert ((c - ours).abs() <= 8 * torch.finfo(torch.float32).eps * exact.abs().float()
                    + bound.float()).all(), cfg


def test_oracle_act_quant_zero_block_and_saturation():
    x = torch.randn(2, 256)
    x[0, :128] = 0
    y, s = fo.act_quant(x)
    assert s[0, 0] == 0 and y[0, :128].float().isnan().all()
    assert y.float().abs().nan_to_num(0).max() <= 448


def test_reference_act_quant_ptx_uses_div_full_and_satfinite_cvt():
    from oracle import ref_cubin
    if not ref_cubin.available():
        pytest.skip('oracle/_ref/ not built (needs an llmc checkout and Triton)')
    m = ref_cubin.manifest()
    for dt in ('bf16', 'fp16', 'fp32'):
        with open(os.path.join(ref_cubin.REF_DIR, f'act_quant_{dt}.ptx')) as fh:
            ptx = fh.read()
        assert 'div.full.f32' in ptx and 'cvt.rn.satfinite.e4m3x2.f32' in ptx, dt
        assert len(m[f'act_quant_{dt}']['params']) == 5
    kinds = {v['mma'] for v in m.values() if 'N' in v}
    assert kinds == {'tcgen05', 'mma.sync'}
