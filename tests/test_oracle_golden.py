"""CPU: the oracle restatement (oracle/*.py) against fixtures produced by the reference's own
code (oracle/gen_golden.py).  Bit-exact wherever the reference is elementwise/integer."""
import os

import pytest
import torch

from oracle import gptq_oracle as go
from oracle import quant_oracle as qo


def _load(golden_dir, name):
    return torch.load(os.path.join(golden_dir, name), weights_only=False)


def _eq(a, b):
    if a is None or b is None:
        return a is None and b is None
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(a, b)


def test_quant_dynamic_matches_reference(golden_dir):
    kat = _load(golden_dir, 'quant_kat.pt')
    assert len(kat['dynamic']) >= 70
    for c in kat['dynamic']:
        gran, gs = c['granularity'], c['group_size']
        _, s, z, qmax, qmin = qo.tensor_qparams(c['w'], c['bit'], c['sym'], gran, gs)
        assert _eq(s, c['scales']), c
        assert torch.equal(z.float(), c['zeros'].float())
        codes, rs, rz = qo.real_quant_dynamic(c['w'], c['bit'], c['sym'], gran, gs)
        assert _eq(codes, c['codes'])
        assert _eq(rs, c['real_scales'])
        assert _eq(rz, c['real_zeros'])
        assert _eq(qo.fake_quant_dynamic(c['w'], c['bit'], c['sym'], gran, gs), c['qdq'])


def test_quant_survey_kat(golden_dir):
    """SURVEY.md Appendix B first two bullets, as literal numbers."""
    w = torch.tensor([[0.1234, -0.5678, 0.9, -0.0001, 0.3333, 0.25, -0.75, 0.5]],
                     dtype=torch.float16)
    codes, s, z = qo.real_quant_dynamic(w, 4, False, 'per_group', 8)
    assert codes.tolist() == [[8, 2, 15, 7, 10, 9, 0, 12]]
    assert float(s) == 0.11004638671875 and int(z) == 7
    codes, s, z = qo.real_quant_dynamic(w, 4, True, 'per_group', 8)
    assert codes.tolist() == [[1, -4, 7, 0, 3, 2, -6, 4]]
    assert float(s) == 0.1285400390625 and z is None


def test_quant_static_and_act(golden_dir):
    kat = _load(golden_dir, 'quant_kat.pt')
    for c in kat['static']:
        qdq = qo.fake_quant_static(c['w'], c['scales'], c['zeros'], c['qmax'], c['qmin'],
                                   'per_group', c['group_size'])
        assert _eq(qdq, c['qdq'])
        codes, rs, rz = qo.real_quant_static(c['w'], c['scales'], c['zeros'], c['qmax'],
                                             c['qmin'], c['bit'], c['sym'], 'per_group',
                                             c['group_size'])
        assert _eq(codes, c['codes']) and _eq(rz, c['real_zeros'])
    for c in kat['acts']:
        assert _eq(qo.fake_quant_dynamic(c['x'], c['bit'], c['sym'], 'per_token'), c['qdq'])


def test_pack_vllm_and_awq(golden_dir):
    kat = _load(golden_dir, 'pack_kat.pt')
    for c in kat['vllm']:
        codes, s, _ = qo.real_quant_dynamic(c['w'], c['bit'], c['sym'], c['granularity'],
                                            c['group_size'])
        packed, scales = qo.pack_vllm(codes, s, c['bit'])
        assert _eq(packed, c['packed']) and _eq(scales, c['scales'])
    # literal words of SURVEY.md Appendix B
    p0 = kat['vllm'][0]['packed']
    assert [[x & 0xffffffff for x in r] for r in p0.tolist()] == \
        [[0x44332211, 0x76544321], [0xfedcba98, 0xffeeddcc]]
    for c in kat['awq']:
        _, s, z = qo.real_quant_dynamic(c['w'], 4, False, 'per_group', c['group_size'])
        qweight, scales, qzeros = qo.pack_awq(c['w'], s, z, c['group_size'])
        assert _eq(qweight, c['qweight']) and _eq(scales, c['scales']) and _eq(qzeros, c['qzeros'])
    k0 = kat['awq'][0]
    assert (int(k0['qweight'][0, 0]) & 0xffffffff) == 0x7cbf8bd0
    assert [int(x) & 0xffffffff for x in k0['qzeros'][0]] == \
        [0x79687779, 0x77778888, 0x68888777, 0x77798888]


def _close(a, b, rel):
    """GEMM / LAPACK derived values: MKL's summation order depends on the core count, so these are
    compared to `rel` of the tensor's largest magnitude (bit-equality holds only on the machine
    that generated the fixture)."""
    a, b = a.double(), b.double()
    return a.shape == b.shape and float((a - b).abs().max()) <= rel * max(float(b.abs().max()), 1e-30)


@pytest.mark.parametrize('idx', [0, 1, 2, 3])
def test_gptq_layer(golden_dir, idx):
    """Each stage starts from the REFERENCE's output of the previous stage, so a last-bit
    difference in a BLAS call cannot cascade into a different permutation or rounding."""
    c = _load(golden_dir, 'gptq_kat.pt')[idx]
    wkw, sp = c['weight_kwargs'], c['special']
    C = c['W'].shape[1]
    H, n = go.hessian(c['batches'], C)
    assert n == len(c['batches'])
    assert _close(H, c['H'], 1e-5)               # SGEMM: summation order only
    # permutation / gather / damping are exact given the reference's H; the factor is LAPACK
    Wp, Hinv, perm = go.prepare(c['W'], c['H'], sp['actorder'], 0.01)
    if sp['actorder']:
        d = torch.diag(c['H'])
        assert torch.equal(d[perm], d[c['perm']])          # equal up to ties (SURVEY 8a G3)
        if not torch.equal(perm, c['perm']):
            Wp, Hinv, _ = go.prepare(c['W'][:, c['perm']], c['H'][c['perm']][:, c['perm']], False, 0.01)
            perm = c['perm']
    assert torch.equal(Wp, c['Wp'])
    assert _close(Hinv, c['Hinv'], 1e-5)
    gran, gs = wkw['granularity'], wkw.get('group_size')
    static = None
    if gran == 'per_group' and sp['static_groups']:
        ng = C // gs
        s = c['rtn']['scales'].reshape(-1, ng).t()
        z = c['rtn']['zeros']
        z = z.reshape(-1, ng).t() if z.numel() > 1 else None
        static = ([s[i].reshape(-1, 1) for i in range(ng)],
                  [z[i].reshape(-1, 1) if z is not None else torch.tensor(0.0) for i in range(ng)])
    elif gran == 'per_channel':
        static = (c['rtn']['scales'], c['rtn']['zeros'])
    tmp, Losses, groups = go.weight_transform(c['Wp'], c['Hinv'], wkw['bit'], wkw['symmetric'], gran, gs,
                                              static_qparams=static, perm=perm)
    # the first 128-column block has no reduction in it (rank-1 updates are K=1 products): exact
    assert torch.equal(tmp[:, :128], c['tmp_perm'][:, :128])
    # later blocks go through `Err1 @ Hinv[i1:i2, i2:]` (K=128 SGEMM): summation order
    bad = ((tmp - c['tmp_perm']).abs() > 1e-5 * c['tmp_perm'].abs().max()).float().mean().item()
    assert bad <= 1e-3, bad
    assert Losses.sum().item() == pytest.approx(c['losses_sum'], rel=1e-4)
    assert _close(Losses.sum(1), c['losses_rows'], 1e-3)
    if gran == 'per_group' and not sp['static_groups']:
        # merge / qdq are elementwise: exact when fed the reference's own sweep result
        bs, bz = go.merged_group_qparams(groups)
        assert torch.equal(bs[:: C // gs], c['buf_scales'][:: C // gs])     # group 0 of every row
        assert _close(bs, c['buf_scales'], 1e-4)
        assert float((bz != c['buf_zeros']).float().mean()) <= 1e-3
        invperm = torch.argsort(perm) if perm is not None else None
        qdq = go.w_qdq(c['new_weight'], c['buf_scales'], c['buf_zeros'], wkw['bit'], wkw['symmetric'],
                       gs, perm if sp['actorder'] else None, invperm, c['dtype'])
        assert _eq(qdq, c['qdq'])


def _ulp_close(a, b, ulps=2):
    """Reductions (`mean` over tokens / rows) evaluated in another order may land on a
    neighbouring fp16/bf16 value."""
    eps = torch.finfo(b.dtype).eps
    return a.shape == b.shape and a.dtype == b.dtype and bool(
        ((a.double() - b.double()).abs() <= ulps * eps * b.double().abs().clamp(min=1e-30)).all())


def test_awq_search_and_clip(golden_dir):
    """awq.py:48-253 and auto_clip.py:83-211 restated vs the reference run."""
    import torch.nn.functional as F
    from oracle import awq_oracle as ao
    kat = _load(golden_dir, 'awq_kat.pt')
    for c in kat['search']:
        wkw = c['weight_kwargs']
        gran, gs = wkw['granularity'], wkw.get('group_size')
        W = c['W']
        subset = [W['gate_proj.weight'], W['up_proj.weight']]
        w_max = ao.weight_scale(subset, gran, gs)
        assert _ulp_close(w_max, c['w_max'])
        assert _ulp_close(ao.act_scale(c['x']), c['x_mean'])
        assert _ulp_close(ao.get_scales(c['x'], c['w_max'], 0.25, c['version']), c['scales_r025'], 4)

        def forward(ws, x, down=W['down_proj.weight']):
            return F.linear(F.silu(F.linear(x, ws[0])) * F.linear(x, ws[1]), down)
        best, losses = ao.search_scale(subset, c['x'], forward, wkw['bit'], wkw['symmetric'], gran, gs,
                                       c['version'])
        # three chained GEMMs in fp16/bf16 per grid point: MKL blocking differs with the core count
        assert losses == pytest.approx(c['losses'], rel=1e-3)
        ref = torch.tensor(c['losses'])
        order = torch.argsort(ref)
        if float(ref[order[1]] - ref[order[0]]) > 2e-3 * float(ref[order[0]]):
            assert int(torch.tensor(losses).argmin()) == int(order[0])
            assert _ulp_close(best, c['best_scales'], 4)
    for c in kat['clip']:
        wkw = c['weight_kwargs']
        mx, mn = ao.auto_clip_layer(c['w'], c['x'], wkw['bit'], wkw['symmetric'], wkw['granularity'],
                                    wkw.get('group_size'), clip_sym=c['clip_sym'], n_sample_token=64)
        # arg-min over 10 shrink levels of a reduction: identical up to near-ties
        assert float((mx != c['best_max']).float().mean()) <= 0.01
        assert float((mn != c['best_min']).float().mean()) <= 0.01
        assert _eq(ao.apply_clip(c['w'], c['best_max'], c['clip_sym'], c['best_min']), c['clipped'])


def test_block_oracle_reproduces_reference_pipeline(golden_dir):
    """oracle/block_oracle.py (the five-forward GPTQ schedule of one decoder block, also the CPU
    arm of bench.py) against the reference's own end-to-end run on the tiny Llama (inputs:
    tests/golden/e2e_gptq_llama.pt): per-layer Losses.sum() of BOTH blocks — block 1 only matches
    if block 0's quantised output (the quant_out pass) is right.

    bf16 CPU GEMMs round differently between CPU builds and thread counts, and GPTQ carries that
    from block 0 into block 1 at the 1e-2 level (as far as the reference's sdpa and eager runs
    differ).  The expected losses (tests/golden/e2e_gptq_llama_cpu_losses.json) therefore come from
    a CPU run of the reference at a recorded thread count, and the oracle runs at that count."""
    import json
    from oracle import block_oracle as bo
    d = _load(golden_dir, 'e2e_gptq_llama.pt')
    with open(os.path.join(golden_dir, 'e2e_gptq_llama_cpu_losses.json')) as fh:
        ref_run = json.load(fh)
    sd = _load(golden_dir, d['init'])['sd0']
    x = [torch.nn.functional.embedding(d['calib_ids'][i:i + 1], sd['model.embed_tokens.weight'])
         for i in range(d['calib_ids'].shape[0])]
    threads = torch.get_num_threads()
    torch.set_num_threads(ref_run['threads'])
    try:
        for blk in range(2):
            W = {n: sd[f'model.layers.{blk}.{"self_attn" if "proj" in n and n[0] in "qkvo" else "mlp"}.{n}.weight']
                 for n in bo.LINEARS}
            W['ln1'] = sd[f'model.layers.{blk}.input_layernorm.weight']
            W['ln2'] = sd[f'model.layers.{blk}.post_attention_layernorm.weight']
            x, _, info = bo.gptq_block(W, x, heads=4, kv_heads=2)
            for n in bo.LINEARS:
                mod = 'self_attn' if n in ('q_proj', 'k_proj', 'v_proj', 'o_proj') else 'mlp'
                ref = ref_run['losses'][f'{blk}.{mod}.{n}']
                assert info[n]['loss'] == pytest.approx(ref, rel=2e-3), (blk, n, info[n]['loss'], ref)
    finally:
        torch.set_num_threads(threads)


def test_range_oracle_matches_reference(golden_dir):
    """calib_algo mse (quant.py:145-203, incl. the aliased running range), per_head / per_block
    (:612-658) and the static histogram observer (:265-522) restated in oracle/quant_oracle.py."""
    kat = _load(golden_dir, 'range_kat.pt')
    for c in kat['mse']:
        qdq, s, z, mn, mx = qo.fake_quant_mse(c['w'], c['bit'], c['sym'], c['granularity'], c['group_size'])
        assert _close(mn, c['min'], 1e-6) and _close(mx, c['max'], 1e-6)
        assert float((mn != c['min']).float().mean()) <= 0.02           # pow / sum rounding near-ties
        assert _close(s, c['scales'], 1e-6)
        assert float((qdq != c['qdq']).float().mean()) <= 0.02
    for c in kat['gran']:
        qdq, _, _ = qo.fake_quant_dynamic_any(c['w'], c['bit'], c['sym'], c['kind'], **c['kwargs'])
        assert _eq(qdq, c['qdq']), c['kind']
    for c in kat['hist']:
        lo, hi = qo.static_hist_range([a for a in c['acts']])
        assert float(lo) == pytest.approx(float(c['hist_min']), rel=1e-6)
        assert float(hi) == pytest.approx(float(c['hist_max']), rel=1e-6)


def test_hist_observer_host_logic_matches_reference(golden_dir):
    """The product's static_hist bookkeeping (llmc_b200/quant.py: re-binning, merge, quantile walk)
    is host arithmetic; with the two device pieces (min/max, histc) replaced by their torch
    equivalents it must reproduce the reference's range and scale on CPU."""
    from llmc_b200.quant import IntegerQuantizer

    class _CpuHist(IntegerQuantizer):
        def _histc(self, tensor, lo, hi):
            return torch.histc(tensor.float(), self.bins, min=lo, max=hi)

        def get_minmax_range(self, tensor):
            return (tensor.min(), tensor.max())
    kat = _load(golden_dir, 'range_kat.pt')
    for c in kat['hist']:
        q = _CpuHist(8, True, 'per_tensor', calib_algo='static_hist')
        sc, zs, qmin, qmax = q.get_batch_tensors_qparams([a.clone() for a in c['acts']])
        assert len(sc) == 1
        assert float(sc[0]) == pytest.approx(float(c['hist_scale']), rel=1e-6)


# ---- SpQR (SURVEY 8(f)-3) ---------------------------------------------------------------------------------
def _spqr_cfg(c, so):
    thr = so.threshold_of(c['Wp'], c['Hinv'], c['special']['relative_threshold'])
    return so.make_cfg(c['weight_kwargs'], c['special'], c['level2'], c['level2'], thr)


def test_spqr_oracle_matches_reference(golden_dir):
    """oracle/spqr_oracle.py against layers the reference's own SpQR produced
    (oracle/gen_spqr_golden.py): leave-one-out outlier search, bilevel qparams, outlier mask,
    `inf` threshold, simplified outliers, round_zp on and off.
      * first 128-column block (elementwise arithmetic + sums over one group only): EXACT;
      * whole sweep (one fp32 GEMM per block in between, MKL summation order): <= 1e-5;
      * from (W, H) through LAPACK's Cholesky triple: <= 1e-3 on the loss, masks >= 99 % equal;
      * w_qdq on the reference's own buffers: exact."""
    from oracle import spqr_oracle as so
    kat = _load(golden_dir, 'spqr_kat.pt')
    assert len(kat) == 5
    for c in kat:
        cfg = _spqr_cfg(c, so)
        gs = cfg['gs']
        cnt = min(128, c['Wp'].shape[1])
        t, e, m, s, z, l = so.row_block(c['Wp'][:, :cnt], c['Hinv'][:cnt, :cnt], cfg)
        R = t.shape[0]
        ng = c['Wp'].shape[1] // gs
        assert torch.equal(t, c['tmp_perm'][:, :cnt]), c['name']
        assert torch.equal(m.bool(), c['mask_perm'][:, :cnt]), c['name']
        assert torch.equal(s, c['buf_scales'].reshape(R, ng)[:, :cnt // gs]), c['name']
        assert torch.equal(z, c['buf_zeros'].reshape(R, ng)[:, :cnt // gs]), c['name']
        tmp, mask, S, Z, losses = so.weight_transform(c['Wp'], c['Hinv'], cfg)
        assert _close(tmp, c['tmp_perm'], 1e-5), c['name']
        assert float((mask.bool() == c['mask_perm']).float().mean()) >= 0.999
        assert _close(S.reshape(-1, 1), c['buf_scales'], 1e-5) and _close(Z.reshape(-1, 1), c['buf_zeros'], 1e-4)
        assert abs(float(losses.sum()) - c['losses_sum']) <= 1e-5 * c['losses_sum']
        full = so.layer_transform(c['W'], c['H'], c['weight_kwargs'], c['special'], c['level2'], c['level2'])
        assert abs(float(full['losses_rows'].sum()) - c['losses_sum']) <= 1e-3 * c['losses_sum'], c['name']
        assert float((full['buf_mask'] == c['buf_mask']).float().mean()) >= 0.99
        if c['perm'] is not None:
            assert float((full['perm'] == c['perm']).float().mean()) >= 0.95
        q = so.w_qdq(c['new_weight'], c['buf_scales'], c['buf_zeros'], c['buf_mask'], c['perm'],
                     c['weight_kwargs'], torch.bfloat16)
        assert torch.equal(q, c['qdq']), c['name']
    assert sum(int(c['mask_perm'].sum()) for c in kat) > 100          # the outlier paths are exercised


def _build_spqr_host(tmp_path):
    import shutil
    import subprocess
    cxx = shutil.which('g++') or shutil.which('c++')
    if cxx is None:
        pytest.skip('no host C++ compiler')
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    so_path = os.path.join(str(tmp_path), 'spqr_row_host.so')
    subprocess.check_call([cxx, '-O2', '-ffp-contract=off', '-shared', '-fPIC',
                           '-I', os.path.join(root, 'llmc_b200', 'csrc'),
                           os.path.join(root, 'tests', 'host', 'spqr_row_host.cpp'), '-o', so_path])
    import ctypes
    return ctypes.CDLL(so_path)


def _spqr_host_block(lib, Wb, Hb, wk, l2s, l2z, thr, simplified, lanes=0):
    import ctypes
    P = ctypes.c_void_p
    R, cnt = Wb.shape
    gs = wk['group_size']
    ng = cnt // gs
    W = Wb.contiguous().clone()
    Hb = Hb.contiguous()
    err, mask = torch.zeros(R, cnt), torch.zeros(R, cnt, dtype=torch.uint8)
    S, Z, loss = torch.zeros(R, ng), torch.zeros(R, ng), torch.zeros(R)
    head = (P(W.data_ptr()), P(Hb.data_ptr()), R, cnt, gs, wk['bit'], int(wk['symmetric']),
            int(wk.get('round_zp', True)), l2s['bit'], int(l2s['symmetric']), int(l2s.get('round_zp', True)),
            l2z['bit'], int(l2z['symmetric']), int(l2z.get('round_zp', True)), ctypes.c_float(thr),
            int(simplified))
    tail = (P(err.data_ptr()), P(mask.data_ptr()), P(S.data_ptr()), P(Z.data_ptr()), P(loss.data_ptr()))
    if lanes:
        # lock-step emulation of the lane-parallel kernel (spqr_row.cuh: lanes_*)
        lib.spqr_row_block_lanes_host(*head, int(lanes), *tail)
    else:
        lib.spqr_row_block_host(*head, *tail)
    return W, err, mask, S, Z, loss


def test_spqr_device_row_code_on_the_host_matches_oracle(golden_dir, tmp_path):
    """llmc_b200/csrc/spqr_row.cuh is the arithmetic of the CUDA kernel spqr_inblock_kernel.  Built
    for the HOST (tests/host/spqr_row_host.cpp, -ffp-contract=off) it must agree bit for bit with
    the oracle — on the reference-generated layers and on a seeded 128-column block with other
    second-level configurations — so the device code is pinned without a GPU.  `lanes`: the
    lane-parallel form the kernel actually runs (16 lanes per row), emulated in lock step."""
    from oracle import spqr_oracle as so
    lib = _build_spqr_host(tmp_path)
    kat = _load(golden_dir, 'spqr_kat.pt')
    for c in kat:
        cfg = _spqr_cfg(c, so)
        cnt = min(128, c['Wp'].shape[1])
        ref = so.row_block(c['Wp'][:, :cnt], c['Hinv'][:cnt, :cnt], cfg)
        for lanes in (0, 16, 8):
            got = _spqr_host_block(lib, c['Wp'][:, :cnt], c['Hinv'][:cnt, :cnt], c['weight_kwargs'],
                                   c['level2'], c['level2'], cfg['thr'], c['special']['simplified_outliers'],
                                   lanes=lanes)
            for a, b in zip(got, ref):
                assert torch.equal(a, b), (c['name'], lanes)
    g = torch.Generator().manual_seed(77)
    for (bit, gs, l2s, l2z, rel) in [
            (4, 16, dict(bit=3, symmetric=False, round_zp=False), dict(bit=3, symmetric=False, round_zp=False), 0.2),
            (3, 32, dict(bit=4, symmetric=True, round_zp=True), dict(bit=3, symmetric=False, round_zp=True), 0.05),
            (2, 64, dict(bit=8, symmetric=False, round_zp=True), dict(bit=8, symmetric=True, round_zp=False), 0.5),
            (4, 128, dict(bit=3, symmetric=False, round_zp=False), dict(bit=3, symmetric=False, round_zp=False), 0.2)]:
        R, cnt = 48, 128
        W = torch.randn(R, cnt, generator=g) * 0.02
        W[torch.rand(R, cnt, generator=g) < 0.02] *= 6
        A = torch.randn(cnt, cnt, generator=g)
        Hinv = torch.linalg.cholesky(A @ A.T / cnt + 0.5 * torch.eye(cnt), upper=True)
        wk = dict(bit=bit, symmetric=False, group_size=gs, round_zp=bool(bit % 2 == 0))
        sp = dict(simplified_outliers=False, relative_threshold=rel)
        thr = so.threshold_of(W, Hinv, rel)
        cfg = so.make_cfg(wk, sp, l2s, l2z, thr)
        ref = so.row_block(W, Hinv, cfg)
        for lanes in (0, 16):
            got = _spqr_host_block(lib, W, Hinv, wk, l2s, l2z, thr, False, lanes=lanes)
            for a, b in zip(got, ref):
                assert torch.equal(a, b), (bit, gs, lanes)
        assert int(ref[2].sum()) > 0
