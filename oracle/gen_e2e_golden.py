"""Generate tests/golden/e2e_*.pt by running the REFERENCE's whole pipeline on CPU:
`GPTQ(...).run_block_loop()` / `Awq(...).run_block_loop()` -> `deploy('fake_quant')` -> PPL
(eval/eval_ppl.py:15-58), on a tiny random-init HF Llama (SURVEY.md Appendix D recipe,
oracle/ref_harness.py).  Build container only (needs /root/reference):

    python oracle/gen_e2e_golden.py

The fixtures hold the initial weights, token ids and the reference's results, so the `-m gpu`
tests (tests/test_gpu_e2e.py) can run the B200 pipeline on the same inputs.
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, '..'))
from oracle import ref_harness as rh  # noqa: E402

OUT = os.path.join(HERE, '..', 'tests', 'golden')

TINY = dict(hidden_size=256, intermediate_size=512, num_hidden_layers=2, num_attention_heads=4,
            num_key_value_heads=2, vocab_size=512, rms_norm_eps=1e-5, max_position_embeddings=4096,
            tie_word_embeddings=False, attention_bias=False, mlp_bias=False, rope_theta=500000.0)

GPTQ_QUANT = {'method': 'GPTQ', 'quant_out': True,
              'weight': {'bit': 4, 'symmetric': False, 'granularity': 'per_group', 'group_size': 128},
              'special': {'actorder': True, 'static_groups': False, 'percdamp': 0.01, 'blocksize': 128,
                          'true_sequential': True}}
AWQ_QUANT = {'method': 'Awq',
             'weight': {'bit': 4, 'symmetric': True, 'granularity': 'per_group', 'group_size': 128},
             'special': {'trans': True, 'trans_version': 'v2', 'weight_clip': True, 'clip_sym': True,
                         'save_scale': True, 'save_clip': True, 'scale_path': '/tmp', 'clip_path': '/tmp'}}
SQ_QUANT = {'method': 'SmoothQuant',
            'weight': {'bit': 8, 'symmetric': True, 'granularity': 'per_channel'},
            'act': {'bit': 8, 'symmetric': True, 'granularity': 'per_token'},
            'special': {'alpha': 0.8}}
HQQ_QUANT = {'method': 'HQQ',
             'weight': {'bit': 4, 'symmetric': False, 'granularity': 'per_group', 'group_size': 64, 'round_zp': False},
             'special': {'axis': 0, 'lp_norm': 0.7, 'beta': 10, 'kappa': 1.01, 'iters': 20}}
SPQR_QUANT = {'method': 'SpQR', 'quant_out': True,
              'weight': {'bit': 4, 'symmetric': False, 'granularity': 'per_group', 'group_size': 16,
                         'round_zp': False},
              'special': {'actorder': True, 'percdamp': 1, 'blocksize': 128, 'true_sequential': True,
                          'relative_threshold': 0.2, 'simplified_outliers': False,
                          'scale': {'bit': 3, 'symmetric': False, 'granularity': 'per_group',
                                    'group_size': 16, 'round_zp': False},
                          'zero': {'bit': 3, 'symmetric': False, 'granularity': 'per_group',
                                   'group_size': 16, 'round_zp': False}}}
RTN_QUANT = {'method': 'RTN',
             'weight': {'bit': 4, 'symmetric': False, 'granularity': 'per_group', 'group_size': 128}}


def check_shape_model_equivalence(hf_model, sd):
    """The shape model of llmc_b200/synth.py must compute the same function as the HF model the
    reference runs on (fp32, CPU) — otherwise the end-to-end comparison would be meaningless."""
    from llmc_b200.synth import SynthModel
    sm = SynthModel('tiny-llama', device='cpu')
    sm.model = sm.model.float()
    sm.torch_dtype = torch.float32
    sm.load_hf_state_dict({k: v.float() for k, v in sd.items()})
    ids = torch.randint(0, 512, (2, 48), generator=torch.Generator().manual_seed(9))
    ours = sm.logits(ids, device='cpu')
    ref = hf_model.float()(ids).logits
    err = (ours - ref).abs().max().item() / ref.abs().max().item()
    assert err < 1e-5, err
    return err


def run_case(name, quant, dtype, n_calib, calib_len, bs, n_eval, eval_len, seed=0, attn=None, save=True):
    from transformers import LlamaConfig
    rh.setup()
    hf_cfg = LlamaConfig(**TINY)
    model = rh.shape_llama(hf_cfg, dtype, seed=seed, attn=attn)
    sd0 = {k: v.detach().clone() for k, v in model.model.state_dict().items()}
    import copy
    arch_err = check_shape_model_equivalence(copy.deepcopy(model.model), sd0)
    g = torch.Generator().manual_seed(seed + 1)
    calib = torch.randint(0, TINY['vocab_size'], (n_calib, calib_len), generator=g)
    evalt = torch.randint(0, TINY['vocab_size'], (1, n_eval * eval_len), generator=g)
    ppl_fp = rh.perplexity(model.model, evalt, eval_len)
    ppl_fp_f32 = rh.perplexity(model.model, evalt, eval_len, ce_dtype=torch.float32)
    init_path = os.path.join(OUT, 'e2e_init_llama.pt')
    if not save:
        pass
    elif not os.path.exists(init_path) or name.startswith('gptq'):
        torch.save(dict(hf_config=TINY, dtype=dtype, seed=seed, sd0=sd0), init_path)
    else:
        ref0 = torch.load(init_path, weights_only=False)['sd0']
        assert all(torch.equal(ref0[k], sd0[k]) for k in sd0)
    logits_fp = model.model(evalt[:, :eval_len]).logits[0].float()
    rec = {'losses': {}, 'awq_losses': {}}
    if quant['method'] == 'GPTQ':
        from llmc.compression.quantization.gptq import GPTQ
        orig_wt = GPTQ.weight_transform
        orig_lt = GPTQ.layer_transform

        def lt(self, layer, name):
            rec['cur'] = f'{self.block_idx}.{name}'
            return orig_lt(self, layer, name)

        def wt(self, W, Hinv, Losses, tmp):
            r = orig_wt(self, W, Hinv, Losses, tmp)
            rec['losses'][rec['cur']] = float(Losses.sum().item())
            return r
        GPTQ.layer_transform, GPTQ.weight_transform = lt, wt
    if quant['method'] == 'SpQR':
        from llmc.compression.quantization.spqr import SpQR
        orig_swt = SpQR.weight_transform
        orig_slt = SpQR.layer_transform

        def slt(self, layer, name):
            rec['cur'] = f'{self.block_idx}.{name}'
            return orig_slt(self, layer, name)

        def swt(self, W, Hinv, Losses, tmp, mask):
            r = orig_swt(self, W, Hinv, Losses, tmp, mask)
            rec['losses'][rec['cur']] = float(Losses.sum().item())
            rec.setdefault('outliers', {})[rec['cur']] = int(mask.sum().item())
            return r
        SpQR.layer_transform, SpQR.weight_transform = slt, swt
    if quant['method'] == 'Awq':
        from llmc.compression.quantization.awq import Awq
        orig_ss = Awq.search_scale_subset

        def ss(self, prev_op, layers_dict, input, inspect_module, is_gqa, subset_kwargs):
            losses = []
            orig_cl = self.calculate_loss

            def cl(o, x):
                v = orig_cl(o, x)
                losses.append(v)
                return v
            self.calculate_loss = cl
            try:
                r = orig_ss(self, prev_op, layers_dict, input, inspect_module, is_gqa, subset_kwargs)
            finally:
                self.calculate_loss = orig_cl
            rec['awq_losses'][f'{self.block_idx}.{next(iter(layers_dict))}'] = losses
            return r
        Awq.search_scale_subset = ss
    algo = rh.run_algo(model, quant, calib, bs=bs, seq_len=calib_len)
    if quant['method'] == 'GPTQ':
        GPTQ.layer_transform, GPTQ.weight_transform = orig_lt, orig_wt
    if quant['method'] == 'Awq':
        Awq.search_scale_subset = orig_ss
    if quant['method'] == 'SpQR':
        SpQR.layer_transform, SpQR.weight_transform = orig_slt, orig_swt
    # GPTQ leaves fp32 compensated weights here (gptq.py:193); AWQ the scaled + clipped ones
    transformed = {k: v.detach().clone() for k, v in model.model.state_dict().items()
                   if 'buf_' not in k and 'layers' in k} if quant['method'] in ('Awq', 'SmoothQuant') else {}
    bufs = {k: (v.to_dense().bool() if v.is_sparse else v).detach().clone()      # SpQR's sparse buf_mask -> bool
            for k, v in model.model.state_dict().items() if 'buf_' in k}
    algo.deploy('fake_quant')
    deployed = {k: v.detach().clone() for k, v in model.model.state_dict().items()
                if 'layers' in k and k.endswith('weight') and 'norm' not in k}
    ppl_q = rh.perplexity(model.model, evalt, eval_len)
    ppl_q_f32 = rh.perplexity(model.model, evalt, eval_len, ce_dtype=torch.float32)
    logits_q = model.model(evalt[:, :eval_len]).logits[0].float()
    out = dict(name=name, hf_config=TINY, quant=quant, dtype=dtype, init='e2e_init_llama.pt', calib_ids=calib,
               bs=bs, eval_ids=evalt, eval_len=eval_len, ppl_fp=ppl_fp, ppl_q=ppl_q,
               ppl_fp_f32=ppl_fp_f32, ppl_q_f32=ppl_q_f32,
               logits_fp=logits_fp.half(), logits_q=logits_q.half(), losses=rec['losses'],
               awq_losses=rec['awq_losses'], outliers=rec.get('outliers', {}), deployed=deployed, transformed=transformed, bufs=bufs,
               arch_check_rel_err=arch_err,
               act_scales={k: v.clone() for k, v in getattr(algo, 'act_scales', {}).items()},
               weight_clips={k: {kk: vv.clone() for kk, vv in v.items()} if isinstance(v, dict) else v
                             for k, v in getattr(getattr(algo, 'auto_clipper', None), 'weight_clips', {}).items()})
    if not save:
        return out
    if quant['method'] in ('GPTQ', 'Awq', 'SpQR'):
        # The reference against ITSELF: the same pipeline with HF's 'eager' attention instead of
        # 'sdpa' — the same mathematics in another floating-point evaluation order.  GPTQ / AWQ
        # amplify bf16-level input differences (act-order permutations, group membership, arg-min
        # near-ties), so this is the yardstick for what "matches the reference" can mean end to end.
        alt = run_case(name, quant, dtype, n_calib, calib_len, bs, n_eval, eval_len, seed, attn='eager',
                       save=False)
        out['self_divergence'] = dict(
            what="reference run with attn_implementation='eager' vs the default 'sdpa' run above",
            loss_rel_dev={k: abs(alt['losses'][k] - v) / v for k, v in out['losses'].items()},
            identical_weight_frac={k: float((alt['deployed'][k] == v).float().mean())
                                   for k, v in out['deployed'].items()},
            awq_curve_rel_dev={k: float(((torch.tensor(alt['awq_losses'][k]) - torch.tensor(v)).abs()
                                         / torch.tensor(v)).max()) for k, v in out['awq_losses'].items()},
            ppl_q=alt['ppl_q'], ppl_q_f32=alt['ppl_q_f32'])
        sd = out['self_divergence']
        print('  self-divergence: max loss dev', max(sd['loss_rel_dev'].values(), default=0),
              'min identical frac', min(sd['identical_weight_frac'].values()), 'ppl_f32', sd['ppl_q_f32'])
    torch.save(out, os.path.join(OUT, f'e2e_{name}.pt'))
    print(f'e2e_{name}: ppl_fp {ppl_fp:.4f} ({ppl_fp_f32:.4f}) ppl_q {ppl_q:.4f} ({ppl_q_f32:.4f}) layers {len(rec["losses"])} '
          f'size {os.path.getsize(os.path.join(OUT, f"e2e_{name}.pt")) / 1e6:.1f} MB')


CPU_THREADS = 8


def gptq_cpu_losses():
    """The reference's per-layer GPTQ Losses.sum() on the e2e_gptq_llama inputs, run on this host's
    CPU torch build with CPU_THREADS threads -> e2e_gptq_llama_cpu_losses.json, the expected values
    of tests/test_oracle_golden.py::test_block_oracle_reproduces_reference_pipeline.  bf16 CPU GEMMs
    round differently between CPU builds and thread counts, and GPTQ carries that from block 0's
    quantised output into block 1, so the file records the build and thread count it came from."""
    import json
    torch.set_num_threads(CPU_THREADS)
    out = run_case('gptq_llama', GPTQ_QUANT, torch.bfloat16, 16, 128, 1, 8, 128, save=False)
    stored = torch.load(os.path.join(OUT, 'e2e_gptq_llama.pt'), weights_only=False)
    assert torch.equal(out['calib_ids'], stored['calib_ids'])
    doc = dict(what='reference GPTQ run_block_loop on the e2e_gptq_llama inputs, CPU: per-layer Losses.sum()',
               torch=torch.__version__, cpu_capability=torch.backends.cpu.get_cpu_capability(),
               threads=CPU_THREADS, losses=out['losses'])
    path = os.path.join(OUT, 'e2e_gptq_llama_cpu_losses.json')
    with open(path, 'w') as fh:
        json.dump(doc, fh, indent=1)
    print(path, len(out['losses']), 'layers')


if __name__ == '__main__':
    which = sys.argv[1:] or ['gptq', 'awq', 'awq_gqa', 'rtn', 'sq', 'hqq', 'spqr', 'gptq_cpu']
    if 'hqq' in which:
        run_case('hqq_llama', HQQ_QUANT, torch.bfloat16, 4, 64, 1, 8, 128)
    if 'sq' in which:
        run_case('sq_llama', SQ_QUANT, torch.bfloat16, 8, 64, 1, 8, 128)
    if 'gptq' in which:
        run_case('gptq_llama', GPTQ_QUANT, torch.bfloat16, 16, 128, 1, 8, 128)
    if 'awq' in which:
        run_case('awq_llama', AWQ_QUANT, torch.bfloat16, 16, 128, -1, 8, 128)
    if 'awq_gqa' in which:
        # base_bq.py:591-594, 678-685 / awq.py:343-348: v_proj -> o_proj migration on the GQA model
        import copy
        q = copy.deepcopy(AWQ_QUANT)
        q['special']['do_gqa_trans'] = True
        run_case('awq_gqa_llama', q, torch.bfloat16, 16, 128, -1, 8, 128)
    if 'spqr' in which:
        run_case('spqr_llama', SPQR_QUANT, torch.bfloat16, 16, 128, 1, 8, 128)
    if 'rtn' in which:
        run_case('rtn_llama', RTN_QUANT, torch.bfloat16, 4, 64, 1, 8, 128)
    if 'gptq_cpu' in which:
        gptq_cpu_losses()
