""""configs/quantization/*.yml run unchanged" (north_star, VERDICT r1 weak-8).

tests/golden/ref_yamls.json is a snapshot of every shipped reference YAML whose method is RTN /
GPTQ / Awq / SpQR / HQQ / SmoothQuant (oracle/gen_yaml_fixture.py parses the reference's configs/quantization/**.yml).  The
CPU test feeds each file's `quant` section to the algorithm classes' own config parsing; the GPU
test runs shipped files end to end through `python -m llmc_b200`'s main() on the tiny Llama with only
model.path / dataset names / sizes overridden (llmc_b200.__main__.adapt_reference_config)."""
import json
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# shipped YAMLs the library refuses with NotImplementedError, and why (everything else must parse)
UNSUPPORTED = {
    'methods/FP_Quant/awq_we2m1a16_g128.yml': 'e2m1',
    'methods/FP_Quant/gptq_we2m1a16_g128.yml': 'e2m1',
    'methods/FP_Quant/rtn_we2m1a16_g128.yml': 'use_qtorch',
    'methods/FP_Quant/rtn_we2m1ae2m1.yml': 'use_qtorch',
    'methods/FP_Quant/rtn_we4m3ae4m3.yml': 'use_qtorch',
    'methods/FP_Quant/rtn_we5m2ae5m2.yml': 'use_qtorch',
    'methods/GPTQ/gptq_owq_w_only.yml': 'OWQ',
    'methods/KVQuant/rtn_w_a_kivi_quant_kv.yml': 'KV-cache',
    'methods/KVQuant/rtn_w_a_naive_quant_kv.yml': 'KV-cache',
    'methods/KVQuant/rtn_w_a_pertensor_static_naive_quant_kv.yml': 'KV-cache',
    'methods/RTN/rtn_w_a_kv.yml': 'KV-cache',
    'methods/RTN/rtn_w_a_wint4afp8.yml': 'Weight48',
    'methods/RTN/rtn_w_a_wint4aint8.yml': 'Weight48',
}


def _docs():
    with open(os.path.join(ROOT, 'tests', 'golden', 'ref_yamls.json')) as fh:
        return json.load(fh)


def _quant_section(cfg):
    q = cfg.quant
    if 'method' in q:
        return q
    return q.get('language') or next(v for v in q.values() if isinstance(v, dict) and 'method' in v)


def test_fixture_matches_the_reference_yamls():
    """Every snapshot entry parses to what the reference's file parsed to when the snapshot was
    taken (tests/golden/ref_yamls_sha256.json), and no shipped hot-path file is missing."""
    from oracle.gen_yaml_fixture import doc_sha256
    docs = _docs()
    with open(os.path.join(ROOT, 'tests', 'golden', 'ref_yamls_sha256.json')) as fh:
        digests = json.load(fh)
    assert len(digests) >= 80
    assert set(docs) == set(digests)
    for rel, doc in docs.items():
        assert doc_sha256(doc) == digests[rel], rel


def test_every_shipped_hot_path_yaml_parses():
    import llmc_b200.awq  # noqa: F401
    import llmc_b200.gptq  # noqa: F401
    import llmc_b200.hqq  # noqa: F401
    import llmc_b200.rtn  # noqa: F401
    import llmc_b200.smoothquant  # noqa: F401
    import llmc_b200.spqr  # noqa: F401
    from llmc_b200.blockwise import AttrDict
    from llmc_b200.registry import ALGO_REGISTRY

    class _M:
        block_name_prefix = 'model.layers'
    refused = {}
    for rel, doc in _docs().items():
        cfg = AttrDict.wrap(doc)
        q = _quant_section(cfg)
        cls = ALGO_REGISTRY[q.method]
        o = cls.__new__(cls)
        o.quant_config, o.config, o.model = q, cfg, _M()
        try:
            o.set_quant_config()
            if q.method in ('GPTQ', 'SpQR'):
                o.add_quant_config()
        except NotImplementedError as e:
            refused[rel] = str(e)
    assert set(refused) == set(UNSUPPORTED), (sorted(set(refused) ^ set(UNSUPPORTED)))
    for rel, why in UNSUPPORTED.items():
        assert why.lower() in refused[rel].lower(), (rel, refused[rel])


RUN = ['methods/GPTQ/gptq_w_only.yml', 'methods/Awq/awq_w_only.yml', 'methods/RTN/rtn_w_only.yml',
       'methods/RTN/rtn_w_a.yml', 'backend/vllm/gptq_w4a16.yml', 'backend/vllm/awq_w4a16.yml',
       'backend/vllm/rtn_w8a16.yml', 'backend/autoawq/awq_w4a16.yml', 'backend/sglang/rtn_w8a8.yml']


@pytest.mark.gpu
@pytest.mark.parametrize('rel', RUN)
def test_shipped_yaml_runs_end_to_end(rel, tmp_path):
    import torch
    from llmc_b200.__main__ import adapt_reference_config, main
    docs = _docs()
    if rel not in docs:
        pytest.skip(f'{rel} not shipped by this reference revision')
    cfg = adapt_reference_config(docs[rel], 'tiny-llama', n_samples=8, seq_len=128, eval_seq_len=128,
                                 save_path=str(tmp_path))
    assert cfg['quant'] == docs[rel]['quant']            # the quant section is used as shipped
    algo, model, report = main(cfg, quiet=True)
    torch.cuda.synchronize()
    if 'ppl_fake_quant' in report:
        assert report['ppl_fake_quant'] == report['ppl_fake_quant'] and report['ppl_fake_quant'] < 1e4
    if any(k.startswith('save_') and v is True for k, v in (docs[rel].get('save') or {}).items()
           if k not in ('save_trans', 'save_fake')):
        assert 'saved' in report and os.path.exists(os.path.join(report['saved'], 'config.json'))
