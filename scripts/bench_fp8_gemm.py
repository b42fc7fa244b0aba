"""K7-fp8 benchmark: the block-scaled FP8 forward (act_quant + fp8_gemm, csrc/gemm_fp8.cu) against
the reference's own Triton kernels compiled for sm_100a (oracle/_ref/, best of its 36 autotune
configurations per shape, i.e. what its autotuner would pick) and, for context, the
dequantise-once bf16 GEMM (llmc_gemm_bf16 on the pre-dequantised weight).

Shapes are DeepSeek-V3 layers at hidden size 7168 (q_a_proj, kv_a_proj, q_b_proj, o_proj, dense
MLP up / down, one routed expert), each at M = 128, 4096 and 16384 tokens.  Every timed call is
preceded by a 256 MB write that evicts the 126 MB L2, and timed alone with CUDA events; the
figure is the median.  Ours and the reference's best config are timed alternately in the same
process.  TFLOP/s counts 2*M*N*K; the share is of the data-sheet dense FP8 rate (4500 TFLOP/s at
1000 W, not reached as such).

    python scripts/bench_fp8_gemm.py [--iters 10] [--out profiles/r03_bench_fp8_gemm.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

SHAPES = [('q_a_proj', 1536, 7168), ('kv_a_proj', 576, 7168), ('q_b_proj', 24576, 1536),
          ('o_proj', 7168, 16384), ('mlp_up', 18432, 7168), ('mlp_down', 7168, 18432),
          ('expert', 2048, 7168)]
MS = [128, 4096, 16384]
PEAK_FP8 = 4500e12


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm',
                              '--format=csv,noheader'], capture_output=True, text=True, timeout=30)
        return out.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f'nvidia-smi unavailable ({e})'


class Timer:
    def __init__(self):
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')

    def __call__(self, fn, iters):
        ts = []
        for _ in range(iters):
            self.flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e-3)
        return statistics.median(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=10)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--out', default=None)
    ap.add_argument('--quick', action='store_true', help='M = 4096 only, 2 shapes')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('bench_fp8_gemm: needs a CUDA device')
    from llmc_b200.kernel import act_quant, fp8_gemm_out
    from llmc_b200.module_utils import block_wise_fp8_forward_func, linear_forward
    from llmc_b200.quant_float import weight_cast_to_bf16, weight_cast_to_fp8
    from oracle import ref_cubin
    have_ref = ref_cubin.available()
    info = card()
    print('card:', info, flush=True)
    timer = Timer()
    rows = []
    shapes, ms = (SHAPES[:2], [4096]) if args.quick else (SHAPES, MS)
    for name, N, K in shapes:
        g = torch.Generator(device='cuda').manual_seed(N + K)
        w = (torch.randn(N, K, generator=g, device='cuda') * 0.02).bfloat16()
        wq, ws = weight_cast_to_fp8(w, 128)
        w_deq = weight_cast_to_bf16(wq, ws, 128)
        del w
        for M in ms:
            x = torch.randn(M, K, generator=g, device='cuda').bfloat16()
            xq, xs = act_quant(x)
            flops = 2.0 * M * N * K
            row = {'layer': name, 'M': M, 'N': N, 'K': K}
            # warm-up every arm
            fp8_gemm_out(xq, xs, wq, ws, torch.bfloat16)
            block_wise_fp8_forward_func(x, wq, ws, 128, None)
            linear_forward(x, w_deq)
            best = None
            if have_ref:
                cands = []
                for cfg in ref_cubin.gemm_configs(N, K):
                    ref_cubin.fp8_gemm(xq, xs, wq, ws, cfg[0])
                    cands.append((timer(lambda: ref_cubin.fp8_gemm(xq, xs, wq, ws, cfg[0]), 2), cfg))
                best = min(cands)[1]
                row['ref_best_config'] = {'name': best[0], 'BLOCK_M': best[1], 'BLOCK_N': best[2],
                                          'num_stages': best[3], 'mma': best[4]}
            t_ours, t_ref = [], []
            for _ in range(args.rounds):           # alternate the two arms
                t_ours.append(timer(lambda: fp8_gemm_out(xq, xs, wq, ws, torch.bfloat16), args.iters))
                if best is not None:
                    t_ref.append(timer(lambda: ref_cubin.fp8_gemm(xq, xs, wq, ws, best[0]), args.iters))
            row['ours_gemm_s'] = statistics.median(t_ours)
            row['ours_gemm_rounds_s'] = t_ours
            row['ours_act_quant_s'] = timer(lambda: act_quant(x), args.iters)
            row['ours_act_quant_GBps'] = M * K * 3.0 / row['ours_act_quant_s'] / 1e9
            row['ours_fused_s'] = timer(lambda: block_wise_fp8_forward_func(x, wq, ws, 128, None), args.iters)
            row['dequant_once_bf16_s'] = timer(lambda: linear_forward(x, w_deq), args.iters)
            row['ours_gemm_TFLOPs'] = flops / row['ours_gemm_s'] / 1e12
            row['ours_gemm_share_of_4500'] = row['ours_gemm_TFLOPs'] * 1e12 / PEAK_FP8
            row['dequant_once_TFLOPs'] = flops / row['dequant_once_bf16_s'] / 1e12
            if best is not None:
                row['ref_gemm_s'] = statistics.median(t_ref)
                row['ref_gemm_rounds_s'] = t_ref
                row['ref_gemm_TFLOPs'] = flops / row['ref_gemm_s'] / 1e12
                row['speedup_vs_ref'] = row['ref_gemm_s'] / row['ours_gemm_s']
                c = fp8_gemm_out(xq, xs, wq, ws, torch.float32)
                r = ref_cubin.fp8_gemm(xq, xs, wq, ws, best[0])
                row['max_abs_dev_vs_ref_best'] = (c - r).abs().max().item()
                row['bit_identical_fraction_vs_ref_best'] = (c == r).float().mean().item()
            rows.append(row)
            print(json.dumps({k: (round(v, 7) if isinstance(v, float) else v) for k, v in row.items()
                              if not k.endswith('rounds_s')}), flush=True)
            del x, xq, xs
        del wq, ws, w_deq
        torch.cuda.empty_cache()
    doc = {'card': info, 'timing': 'CUDA events, one call per timing, L2 evicted by a 256 MB write '
                                   'before each call; median of --iters calls, ours and ref alternated '
                                   'for --rounds rounds', 'iters': args.iters, 'rows': rows}
    if args.out:
        with open(args.out, 'w') as fh:
            json.dump(doc, fh, indent=1)


if __name__ == '__main__':
    main()
