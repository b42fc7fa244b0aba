#!/usr/bin/env python
"""bench.py — GPTQ-W4 layers/sec (BASELINE.json metric), Llama-3-8B shape, 128 x 2048 synthetic
calibration tokens (configs[1]; YAML = configs/gptq_w_only.yml, the schema of the reference's
configs/quantization/methods/GPTQ/gptq_w_only.yml).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A STEP = GPTQ calibration of ONE decoder block (7 linears: RTN seed qparams, Hessians over the
full calibration set, Cholesky, column sweep, fake-quant forward that feeds the next block).
Steps walk consecutive blocks of the model exactly like run_block_loop (block i+1 consumes the
quantised output of block i); the default W=3, K=29 is the complete 32-block model with the first
three blocks as warm-up.  value = 7*K / t.

Two timed regions, both bracketed by barrier + cuda synchronize, timed with CUDA events, max
over ranks:
  value : weights and activations resident in HBM when the region starts;
  e2e   : every step copies its block's weights host(pinned) -> device and the calibrated block
          (fp32 compensated weights + group scales/zeros + per-layer loss) device -> host, like
          the reference's block.cuda() ... block.cpu() (base_blockwise_quantization.py:397,418).
N > 1 (torchrun): data-parallel over calibration samples — the reference's own multi-GPU mode
(base_dataset.py:170-172) — with ONE NCCL all-reduce of H per distinct input (gptq.py:292
does it per batch); total work fixed => "scaling": "strong".

--impl reference: the reference's CPU path (oracle port; the Python reference cannot travel to
the GPU box) on the host cores: every step is the same workload — one decoder block through the
reference's schedule at the real shapes — on a bounded sample (see REF_SAMPLE), and the reported
value is extrapolated to the full calibration set with stated rules.

--dump-outputs DIR: after the timed steps, write what the last device-resident step produced
(block_outputs) to DIR/<name>.npy, so that two builds can be compared output for output on the
same seeded inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODEL = 'llama-3-8b'
N_SAMPLES, SEQ_LEN = 128, 2048
LINEARS_PER_BLOCK = 7


def workload_name(args):
    """The same string in both arms' `config.workload`."""
    return (f'GPTQ W4A16 g128 asym act-order true_sequential quant_out, {args.model} shape, '
            f'{args.samples}x{args.seq_len} synthetic tokens (BASELINE.json configs[1]); '
            f'step = one decoder block (7 linears)')


METRIC = 'GPTQ-W4 layers/sec (Llama-3-8B shape, 128 calib samples)'
DATA = 'synthetic (random-init N(0,0.02^2) weights, uniform random token ids)'


def bench_config(args, world):
    """`config` of the JSON line — the SAME dict in both arms (the driver compares them)."""
    return {'workload': workload_name(args), 'yaml': 'configs/gptq_w_only.yml',
            'l2': 'inputs (>=2 GiB activations per step) exceed the 126 MB L2',
            'parallelism': (f'dp{world} over calibration samples, 1 NCCL all-reduce of H per distinct input'
                            if world > 1 else 'single GPU')}


def load_yaml_config():
    import yaml
    with open(os.path.join(ROOT, 'configs', 'gptq_w_only.yml')) as fh:
        return yaml.safe_load(fh)


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json'))), 'measured'
    except Exception:
        return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0}, 'fallback'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.nvml_thread, self.nvml_stop = None, threading.Event()

    def _nvml_loop(self, pynvml, h):
        # in-process NVML polling: the same counters nvidia-smi prints, without a second process
        # hammering the driver during the timed region
        R = pynvml
        bits = (('hw_slowdown', R.nvmlClocksEventReasonHwSlowdown),
                ('hw_thermal_slowdown', R.nvmlClocksEventReasonHwThermalSlowdown),
                ('sw_thermal_slowdown', R.nvmlClocksEventReasonSwThermalSlowdown),
                ('sw_power_cap', R.nvmlClocksEventReasonSwPowerCap))
        while not self.nvml_stop.wait(0.1):
            try:
                sm = R.nvmlDeviceGetClockInfo(h, R.NVML_CLOCK_SM)
                mx = R.nvmlDeviceGetMaxClockInfo(h, R.NVML_CLOCK_SM)
                pw = R.nvmlDeviceGetPowerUsage(h) / 1e3
                mask = R.nvmlDeviceGetCurrentClocksEventReasons(h)
                self.rows.append([str(sm), str(mx), str(pw)] +
                                 ['Active' if (mask & b) else 'Not Active' for _, b in bits])
            except Exception:
                break

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical GPUs; map through CUDA_VISIBLE_DEVICES when it is numeric
            vis = os.environ.get('CUDA_VISIBLE_DEVICES', '')
            ids = [int(v) for v in vis.split(',')] if vis and all(v.strip().isdigit() for v in vis.split(',')) else None
            phys = ids[self.index] if ids and self.index < len(ids) else self.index
            h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
            self.proc = 'nvml'
            self.nvml_thread = threading.Thread(target=self._nvml_loop, args=(pynvml, h), daemon=True)
            self.nvml_thread.start()
            return
        except Exception:
            self.proc = None
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}',
                 '--format=csv,noheader,nounits', '-lms', '200'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
        if self.proc == 'nvml':
            self.nvml_stop.set()
            self.nvml_thread.join(timeout=2)
        else:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except Exception:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        sm.sort()
        # under load = upper half of the samples (the region also contains idle host gaps)
        load = sm[len(sm) // 2:] or sm
        med = load[len(load) // 2] if load else None
        return {'sm_mhz': med, 'sm_max_mhz': mx, 'reasons': sorted(reasons), 'samples': len(sm)}


def dist_setup(n_gpus):
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    return rank, world, local


def barrier(world):
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()


def max_over_ranks(ms, world):
    if world == 1:
        return ms
    t = torch.tensor([ms], device='cuda', dtype=torch.float64)
    torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    return float(t.item())


def make_algo(cfg, model, first_input):
    from llmc_b200.blockwise import AttrDict
    from llmc_b200.gptq import GPTQ

    class BenchGPTQ(GPTQ):
        """Seed qparams are collected per block inside the step (the metric counts
        collect_model_qparams, SURVEY.md 8d) instead of for the whole model up front."""

        def collect_model_qparams(self):
            # GPTQ.block_opt collects a pending block's seeds on entry (the same code path a
            # host-resident model takes)
            self._qparams_pending = set(range(len(self.blocks)))

    c = AttrDict.wrap(cfg)
    return BenchGPTQ(model, c.quant, first_input, None, c)


def run_ours(args):
    from llmc_b200 import _lib
    from llmc_b200.prof import TIMER
    from llmc_b200.synth import SynthModel
    rank, world, local = dist_setup(args.gpus)
    dev = torch.device('cuda', local)
    torch.cuda.set_device(dev)
    cfg = load_yaml_config()
    W, K = args.warmup, args.steps
    n_blocks = W + K
    lib = _lib.load()
    pk, pk_src = peaks()

    def build_model():
        torch.manual_seed(0)
        m = SynthModel(args.model, n_layers=n_blocks, seed=0, device='cuda', with_head=False,
                       init='device')
        return m

    def first_input(model):
        # rank r calibrates on samples r::world (data/dataset/base_dataset.py:170-172)
        inp = model.first_block_input(args.samples, args.seq_len, bs=1, seed=1, device='cuda')
        if world > 1:
            inp = {'data': inp['data'][rank::world], 'kwargs': inp['kwargs'][rank::world]}
        # one contiguous [n, S, hidden] tensor viewed as a list (whole-batch kernels, no cat)
        x = torch.cat(inp['data'], dim=0)
        inp['data'] = list(torch.split(x, 1, dim=0))
        inp['stacked'] = x
        return inp

    out = {}
    # ------------------------------------------------------------------ region 1: device resident
    model = build_model()
    algo = make_algo(cfg, model, first_input(model))
    blocks = algo.blocks
    for i in range(W):
        algo.block_idx = i
        algo.block_opt(blocks[i])
    barrier(world)
    sampler = ClockSampler(local)
    if os.environ.get('LLMC_BENCH_SAMPLER', '1') == '1':     # diagnosis switch, default on
        sampler.start()
    TIMER.enabled = os.environ.get('LLMC_BENCH_TIMER', '1') == '1'
    TIMER.reset()
    step_sync = os.environ.get('LLMC_BENCH_STEP_SYNC', '0') == '1'
    l0 = lib.llmc_b200_launch_count()
    ms0 = torch.cuda.memory_stats(dev)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    t_host = time.perf_counter()
    for i in range(W, W + K):
        algo.block_idx = i
        algo.block_opt(blocks[i])
        if step_sync:
            algo.layer_loss(f'{i}.mlp.down_proj')
    host_enqueue_ms = (time.perf_counter() - t_host) * 1e3     # host time to enqueue the K steps
    e.record()
    ms1 = torch.cuda.memory_stats(dev)
    # cudaMalloc / cudaFree inside the timed region synchronise the device (allocator churn)
    alloc_diag = {k: int(ms1.get(k, 0) - ms0.get(k, 0))
                  for k in ('num_device_alloc', 'num_device_free', 'num_alloc_retries')}
    barrier(world)
    ms_dev = max_over_ranks(s.elapsed_time(e), world)
    launches = lib.llmc_b200_launch_count() - l0
    kern = TIMER.summary()
    TIMER.enabled = False
    clocks = sampler.stop()
    loss_probe = algo.layer_loss(f'{W}.self_attn.q_proj') if K > 0 else None
    dump = None
    if args.dump_outputs and rank == 0 and K > 0:
        dump = block_outputs(algo, model, blocks[W + K - 1], W + K - 1)
    del algo, model, blocks
    torch.cuda.empty_cache()

    # ------------------------------------------------------------------ region 2: end to end
    model = build_model()
    inp = first_input(model)
    # The model lives in pinned host memory, as in the reference (whose run_block_loop does
    # block.cuda() / block.cpu() around every block); the public API is
    # run_block_loop(first, last, streamer): every step's weights go host->device and its
    # results (calibrated fp32 weights + qparam buffers) device->host inside the timed region,
    # and the per-layer loss of the step is read back on the host.
    from llmc_b200.blockwise import BlockStreamer
    # N > 1: every rank streams the (replicated) weights in; the calibrated block is identical on
    # all ranks and is written back by rank 0 only, like the reference's rank-0 save
    streamer = BlockStreamer(model.get_blocks(), dev, writeback=(rank == 0))
    streamer.offload()
    algo = make_algo(cfg, model, inp)
    host_losses = []
    pending = []          # (pinned fp64 scalar, event) of steps whose loss is still travelling

    def drain(keep):
        while len(pending) > keep:
            h, ev = pending.pop(0)
            ev.synchronize()
            host_losses.append(float(h))

    def read_loss(i):
        # Host read of the step's result, pipelined by one step: the loss of block i is copied to
        # pinned memory asynchronously and consumed while block i+1 is being enqueued, so the host
        # keeps its lead over the GPU (a blocking .item() per step made N > 1 runs host bound).
        st = torch.cuda.current_stream(dev)
        t = algo.losses[f'{i}.mlp.down_proj'].double().sum()
        h = torch.empty((), dtype=torch.float64, pin_memory=True)
        h.copy_(t, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(st)
        pending.append((h, ev))
        drain(1)

    algo.run_block_loop(0, W, streamer, on_block_done=read_loss)
    drain(0)
    if W > 0:
        streamer.preallocate_results(0, range(W, W + K))               # pinning is setup, not a step
    torch.cuda.synchronize()
    h2d0, d2h0 = streamer.h2d_bytes, streamer.d2h_bytes
    barrier(world)
    s2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s2.record()
    algo.run_block_loop(W, W + K, streamer, on_block_done=read_loss)
    drain(0)                                                          # every step's loss is on the host
    torch.cuda.current_stream().wait_stream(streamer.d2h)             # the last write-back is timed too
    e2.record()
    barrier(world)
    ms_e2e = max_over_ranks(s2.elapsed_time(e2), world)
    h2d = (streamer.h2d_bytes - h2d0) // max(K, 1)
    d2h_holder = {'bytes': (streamer.d2h_bytes - d2h0) // max(K, 1) + 8}

    # ------------------------------------------------------------------ report (rank 0)
    if rank != 0:
        return
    layers = LINEARS_PER_BLOCK * K
    if not kern:                       # LLMC_BENCH_TIMER=0 (diagnosis): no per-kernel spans
        kern = {'untimed': dict(calls=1, ms=ms_dev, flops=0.0, bytes=0.0)}
    total_kernel_ms = sum(v['ms'] for v in kern.values()) or 1.0
    dom = max(kern, key=lambda k: kern[k]['ms'])
    # the roofline object describes the dominant TENSOR kernel by time among our kernels
    # Spans are grouped by the device kernel behind them: 'gemm' (fake-quant forward) and 'syrk'
    # (Hessian) are the two instantiations of csrc/gemm.cu:umma_gemm_kernel.
    own = {k: v for k, v in kern.items() if 'cusolver' not in k}
    umma = {'ms': 0.0, 'calls': 0, 'flops': 0.0, 'bytes': 0.0}
    for k in ('gemm', 'syrk'):
        if k in own:
            for f in umma:
                umma[f] += own[k][f]
    dom_own = max(own, key=lambda k: own[k]['ms'])
    d = own[dom_own]
    ncu = {}
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'profiles', 'roofline_traffic.json')) as f:
            ncu = json.load(f)
    except (OSError, ValueError):
        pass
    if umma['ms'] >= d['ms'] and umma['flops'] > 0:
        # one launch = one 16-sample chunk GEMM or one SYRK; algorithmic flops = 2MNK (GEMM),
        # T*C*(C+1) (SYRK, unique entries only); DESIGN.md section 4
        ach = umma['flops'] / umma['ms'] / 1e9
        peak_tf = pk['bf16_tflops']
        roof = {'kernel': 'umma_gemm_kernel (spans gemm+syrk)', 'bound': 'tensor', 'achieved': round(ach, 1),
                'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': round(ach / peak_tf, 4),
                'traffic': ncu.get('umma_gemm_kernel', {}).get('dram_bytes_per_launch'),
                'traffic_note': ncu.get('umma_gemm_kernel', {}).get('note'),
                'peak_source': f'{pk_src} bf16_tflops (cuBLAS burst); sustained figure: '
                               f'{pk.get("bf16_tflops_sustained")}',
                'avg_launch_ms': round(umma['ms'] / umma['calls'], 4), 'launches': umma['calls'],
                'algorithmic_flops_per_launch': round(umma['flops'] / umma['calls'], 1)}
    else:
        ach = d['bytes'] / d['ms'] / 1e6
        roof = {'kernel': dom_own, 'bound': 'hbm', 'achieved': round(ach, 1), 'peak': pk['hbm_gbs'],
                'unit': 'GB/s', 'frac': round(ach / pk['hbm_gbs'], 4), 'traffic': None,
                'peak_source': f'{pk_src} hbm_gbs', 'avg_launch_ms': round(d['ms'] / d['calls'], 4),
                'launches': d['calls']}
    breakdown = {k: {'calls': v['calls'], 'ms': round(v['ms'], 2),
                     'share': round(v['ms'] / total_kernel_ms, 4),
                     **({'tflops': round(v['flops'] / v['ms'] / 1e9, 1)} if v['flops'] else {}),
                     **({'gbs': round(v['bytes'] / v['ms'] / 1e6, 1)} if v['bytes'] else {})}
                 for k, v in sorted(kern.items(), key=lambda kv: -kv[1]['ms'])}
    cpu = cpu_baseline_sample(args)
    line = {
        'metric': METRIC,
        'value': round(layers / (ms_dev / 1e3), 3), 'unit': 'layers/s', 'n_gpus': world,
        'steps': K, 'warmup': W, 'ms_per_step': round(ms_dev / K, 2), 'higher_is_better': True,
        'scaling': 'strong', 'vs_baseline': None, 'dtype': 'bf16 activations/weights, fp32 Hessian+GPTQ',
        'data': DATA,
        'config': bench_config(args, world),
        'e2e': {'value': round(layers / (ms_e2e / 1e3), 3), 'unit': 'layers/s',
                'ms_per_step': round(ms_e2e / K, 2), 'h2d_bytes_per_step': h2d,
                'd2h_bytes_per_step': d2h_holder['bytes']},
        'gpu_launches': int(launches),
        'host_enqueue_ms_per_step': round(host_enqueue_ms / max(K, 1), 2),
        'allocator_in_timed_region': alloc_diag,
        'clocks': clocks,
        'roofline': roof,
        'kernels': breakdown,
        'cpu_baseline': cpu,
        'check': {'q_proj_loss_first_timed_block': loss_probe, 'dominant_span': dom},
    }
    if dump is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in dump.items():
            np.save(os.path.join(args.dump_outputs, f'{name}.npy'), arr)
    emit(line)


DUMP_BYTES = 64 << 20            # all arrays of --dump-outputs together
DUMP_MAX_ELEMS = 1 << 19         # per array; larger arrays are reduced to a seeded sample


def block_outputs(algo, model, block, idx):
    """What block_opt hands its caller for block `idx`, as host float arrays: per linear the
    GPTQ-compensated fp32 weight, the fake-quant weight the next forward uses, the group scales /
    zeros, the act-order permutation and the per-row losses; and the block's output, which is the
    next block's calibration input.  An array above the per-array share of DUMP_BYTES is reduced
    to the same seeded choice of elements in every run (integers go to float64, exact; the rest to
    float32)."""
    arrays = {}
    for name, m in model.get_block_linears(block).items():
        for buf in ('weight', 'tmp_weight', 'buf_scales', 'buf_zeros', 'buf_perm'):
            t = getattr(m, buf, None)
            if torch.is_tensor(t):
                arrays[f'{name}.{buf}'] = t
        arrays[f'{name}.losses'] = algo.losses[f'{idx}.{name}']
    x = algo.input.get('stacked')
    arrays['block_output'] = x if x is not None else torch.cat(algo.input['data'])
    share = DUMP_BYTES // len(arrays)
    out = {}
    for name, t in arrays.items():
        flat = t.detach().reshape(-1)
        dt = torch.float32 if t.is_floating_point() else torch.float64
        n = min(DUMP_MAX_ELEMS, share // dt.itemsize)
        if flat.numel() > n:
            g = torch.Generator().manual_seed(flat.numel())
            idx_s = torch.randint(flat.numel(), (n,), generator=g).sort().values
            flat = flat[idx_s.to(flat.device)]
        out[name] = flat.to(dt).cpu().numpy().reshape(t.shape if flat.numel() == t.numel() else -1)
    return out


# ---------------------------------------------------------------------------------- CPU baseline
# The reference's own algorithm on the host CPU (oracle/block_oracle.py, pinned against the
# reference's end-to-end run by tests/test_oracle_golden.py::test_block_oracle_...): ONE decoder
# block of the SAME workload through the reference's schedule — five block forwards, eleven
# per-linear Hessians, seven Cholesky triples and column sweeps at the real shapes — on a bounded
# SAMPLE, extrapolated to the full calibration set with the rules below.  BASELINE.md §3 planned
# "one block at the full calibration set" (25-30 min); a driver run cannot afford that.
REF_SAMPLE = dict(n_tok=256, sweep_cols=256, chol_cap=6144)
_THREADS = None


def _best_threads(cores):
    """Thread count per phase of the CPU arm, chosen by a short probe of each phase's dominant op:
    on a 100+ core host neither MKL nor the elementwise kernels are fastest with every core (the
    reference's column loop is ~15 tiny torch ops per column; bf16 GEMMs and LAPACK collapse under
    oversubscription) — the baseline gets the best setting found, not a handicap."""
    global _THREADS
    if _THREADS is not None:
        return _THREADS
    import torch.nn.functional as F
    from oracle import gptq_oracle as go
    from oracle import quant_oracle as qo
    g = torch.Generator().manual_seed(0)
    Wsw = torch.randn(1024, 128, generator=g) * 0.02
    Hinv = torch.triu(torch.rand(128, 128, generator=g) * 0.01) + torch.eye(128)
    xb = torch.randn(256, 4096, generator=g).bfloat16()
    wb = torch.randn(14336, 4096, generator=g).bfloat16()
    xf = torch.randn(4096, 256, generator=g)
    A = torch.randn(2048, 2048, generator=g)
    A = A @ A.t() + 2048 * torch.eye(2048)
    probes = {
        'sweep': lambda: go.weight_transform(Wsw, Hinv, 4, False, 'per_group', 128),
        'forward': lambda: F.linear(xb, wb),
        'hessian': lambda: xf.matmul(xf.t()),
        'cholesky': lambda: torch.cholesky_inverse(torch.linalg.cholesky(A)),
        'qparams': lambda: qo.tensor_qparams(wb[:4096], 4, False, 'per_group', 128),
    }
    cands = sorted({c for c in (1, 4, 8, 16, 32, 64) if c <= cores})
    out = {}
    for name, fn in probes.items():
        best, best_t = cands[0], float('inf')
        for n in cands:
            if name != 'sweep' and n < 4 and cores >= 4:
                continue
            torch.set_num_threads(n)
            fn()                                            # warm
            dt = float('inf')
            for _ in range(2):
                t0 = time.perf_counter()
                fn()
                dt = min(dt, time.perf_counter() - t0)
            if dt < best_t:
                best, best_t = n, dt
        out[name] = best
    torch.set_num_threads(cores)
    _THREADS = out
    return out


def reference_block_sample(args, seed=0):
    """One sampled step of the reference arm.  Returns (extrapolated seconds for ONE full block,
    wall seconds of the sample, detail dict).

    Extrapolation (each rule is exact in the operation count of the phase it scales):
      forward, hessian : x T / n_tok        (GEMM work is linear in tokens; T = samples * seq_len)
      hessian_fixed    : x samples          (the O(C^2) rescale / accumulate passes of add_batch run
                         once per calibration batch, bs = 1 sample; the sample step holds one batch)
      cholesky         : x (C / n)^3 per linear whose C exceeds chol_cap (LAPACK potrf/potri, O(C^3))
      sweep            : x C / sweep_cols per linear (per-column cost of the reference's loop is
                         launch/dispatch bound and flat in the column index)
      qparams          : measured in full."""
    from llmc_b200.synth import SHAPES
    from oracle import block_oracle as bo
    sh = SHAPES[args.model]
    cores = os.cpu_count() or 1
    threads = _best_threads(cores)
    T = args.samples * args.seq_len
    n_tok = min(REF_SAMPLE['n_tok'], args.seq_len)
    g = torch.Generator().manual_seed(1000 + seed)
    W = bo.make_block(sh['hidden'], sh['inter'], sh['heads'], sh['kv_heads'], sh['dtype'], seed=seed)
    x = [(torch.randn(1, n_tok, sh['hidden'], generator=g) * torch.exp(
        torch.randn(sh['hidden'], generator=g) * 0.5)).to(sh['dtype'])]
    t0 = time.perf_counter()
    _, t, info = bo.gptq_block(W, x, sh['heads'], sh['kv_heads'], sweep_cols=REF_SAMPLE['sweep_cols'],
                               chol_cap=REF_SAMPLE['chol_cap'], threads=threads)
    wall = time.perf_counter() - t0
    torch.set_num_threads(cores)
    tok = T / n_tok
    chol = sum(v['t_chol'] * (v['C'] / v['chol_n']) ** 3 for v in info.values())
    sweep = sum(v['t_sweep'] * (v['C'] / v['sweep_cols']) for v in info.values())
    full = dict(forward=t['forward'] * tok, hessian=t['hessian'] * tok,
                hessian_fixed=t['hessian_fixed'] * args.samples, cholesky=chol, sweep=sweep,
                qparams=t['qparams'])
    return sum(full.values()), wall, dict(measured_s={k: round(v, 3) for k, v in t.items()},
                                          extrapolated_block_s={k: round(v, 2) for k, v in full.items()},
                                          threads=threads)


def reference_sample_text(args, cores):
    return (f'oracle port of the reference (CPU torch, {cores} host threads; oracle/block_oracle.py): one '
            f'{args.model}-shaped decoder block through the reference schedule (5 block forwards, 11 per-linear '
            f'Hessians, 7 Cholesky triples + W4 asym g128 act-order column sweeps) on a sample of '
            f'{min(REF_SAMPLE["n_tok"], args.seq_len)} of {args.samples * args.seq_len} calibration tokens, Cholesky of '
            f'C > {REF_SAMPLE["chol_cap"]} on its leading {REF_SAMPLE["chol_cap"]}^2 block, sweeps on the first '
            f'{REF_SAMPLE["sweep_cols"]} columns; value = 7 linears / the block time extrapolated to the full '
            'workload (forward, Hessian GEMM x tokens; per-batch Hessian passes x samples; Cholesky x (C/n)^3; '
            'sweep x C/cols)')


def cpu_baseline_sample(args):
    cores = os.cpu_count() or 1
    est, wall, detail = reference_block_sample(args)
    return {'value': round(LINEARS_PER_BLOCK / est, 6), 'unit': 'layers/s', 'cores': cores, 'kind': 'port',
            'sample': reference_sample_text(args, cores), 'sample_wall_s': round(wall, 2),
            'extrapolated_block_s': round(est, 1), **detail}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    for i in range(args.warmup):
        reference_block_sample(args, seed=i)
    est_total, detail = 0.0, None
    t0 = time.perf_counter()
    for i in range(args.steps):
        est, _, detail = reference_block_sample(args, seed=args.warmup + i)
        est_total += est
    wall = time.perf_counter() - t0
    v = round(LINEARS_PER_BLOCK * args.steps / est_total, 6)
    world = int(os.environ.get('WORLD_SIZE', '1'))
    sample = reference_sample_text(args, cores)
    emit({
        'impl': 'reference', 'metric': METRIC,
        'value': v, 'unit': 'layers/s', 'n_gpus': world,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': round(est_total / args.steps * 1e3, 1),
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
        'dtype': 'bf16 activations/weights, fp32 Hessian+GPTQ', 'data': DATA,
        'config': bench_config(args, world),
        'note': 'value and ms_per_step are EXTRAPOLATED to the full workload from the per-step sample '
                '(cpu_baseline.sample); sample_ms_per_step is what a step actually took on the host',
        'sample_ms_per_step': round(wall / args.steps * 1e3, 1),
        'cpu_baseline': {'value': v, 'unit': 'layers/s', 'cores': cores, 'kind': 'port', 'sample': sample,
                         **(detail or {})},
        'e2e': {'value': v, 'unit': 'layers/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}})


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line of the contract, on the process's original stdout."""
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + '\n')
    out.flush()


def main():
    # Libraries print banners on fd 1 (e.g. "NCCL version ..." under torchrun); keep the real
    # stdout for the JSON line and send everything else to stderr.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), 'w')
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=29)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--model', default=MODEL)
    ap.add_argument('--samples', type=int, default=N_SAMPLES)
    ap.add_argument('--seq-len', dest='seq_len', type=int, default=SEQ_LEN)
    ap.add_argument('--dump-outputs', dest='dump_outputs', metavar='DIR', default=None,
                    help='write the last timed step\'s results to DIR/<name>.npy (at most 64 MiB)')
    args = ap.parse_args()
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs dumps the CUDA path; the reference arm runs a sampled CPU block')
    if args.impl == 'reference':
        return run_reference(args)
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device — llmc_b200 has no CPU path (use --impl reference '
                         'for the CPU baseline)')
    run_ours(args)
    if int(os.environ.get('WORLD_SIZE', '1')) > 1:
        torch.distributed.destroy_process_group()


if __name__ == '__main__':
    main()
