"""Snapshot the reference's shipped quantisation YAMLs that use a hot-path method (RTN / GPTQ / Awq,
plus the built 8(f)-3 siblings SpQR / HQQ / SmoothQuant;
SURVEY.md Appendix F: 91 of 132 files) as parsed dicts -> tests/golden/ref_yamls.json, so that
"configs/quantization/*.yml run unchanged" can be tested without the reference checkout, and the
SHA-256 of each parsed file -> tests/golden/ref_yamls_sha256.json, which pins the snapshot to the
files it was taken from.

    python oracle/gen_yaml_fixture.py <reference checkout>
"""
import glob
import hashlib
import json
import os
import sys

import yaml

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', 'tests', 'golden')
OUT = os.path.join(GOLDEN, 'ref_yamls.json')
DIGESTS = os.path.join(GOLDEN, 'ref_yamls_sha256.json')


def doc_sha256(doc):
    """Digest of a parsed YAML document, independent of key order and JSON formatting."""
    return hashlib.sha256(json.dumps(doc, sort_keys=True).encode()).hexdigest()


def main(reference):
    ref = os.path.join(reference, 'configs', 'quantization')
    out = {}
    for p in sorted(glob.glob(os.path.join(ref, '**', '*.yml'), recursive=True)):
        with open(p) as fh:
            try:
                doc = yaml.safe_load(fh)
            except yaml.YAMLError:
                continue
        q = (doc or {}).get('quant') or {}
        methods = {q.get('method')} | {v.get('method') for v in q.values() if isinstance(v, dict)}
        if methods & {'RTN', 'GPTQ', 'Awq', 'SpQR', 'HQQ', 'SmoothQuant'}:
            out[os.path.relpath(p, ref)] = doc
    with open(OUT, 'w') as fh:
        json.dump(out, fh, indent=0, sort_keys=True)
    with open(DIGESTS, 'w') as fh:
        json.dump({rel: doc_sha256(doc) for rel, doc in out.items()}, fh, indent=0, sort_keys=True)
    print(len(out), 'yamls ->', OUT, os.path.getsize(OUT), 'bytes')


if __name__ == '__main__':
    main(sys.argv[1])
