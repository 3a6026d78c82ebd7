#!/usr/bin/env python
"""Headline benchmark: pipelined ViT / BERT / DeiT inference throughput on N B200s (one stage per GPU).

    python bench.py --gpus 1 --steps 200 --warmup 20                       # N = 1
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W                             # N > 1, one rank per GPU
    python bench.py --impl reference --gpus N --steps K --warmup W         # the reference's CPU path

A STEP is one micro-batch through the whole pipeline (BASELINE.json: images/s or sequences/s per pipeline).
Default workload = BASELINE.json configs[1]'s model and micro-batch (google/vit-base-patch16-224, ubatch 8,
fp16 operands / fp32 accumulate) with the 48 sub-layers split evenly over the N stages ([1,24,25,48] at N=2).

Every N runs the same code: DistP2pContext (N > 1) + DistP2pPipelineStage on the native pipeline (one CUDA graph per
stage micro-batch, peer-memory links between the GPUs, `pipeedge_b200/comm/p2p/_native.py`); graphs are captured before
the warm-up, so the first timed micro-batch is already a replay.

One JSON line is printed by rank 0:
  value        whole-pipeline throughput with inputs already resident in HBM: device time (CUDA events) from the first
               graph launch to the last micro-batch leaving each rank / the last result reaching the data rank, max
               over ranks
  e2e          the same through the public API with pinned HOST inputs: H2D of every micro-batch and D2H of
               every result inside the (wall-clock, device-synchronised) timed region
  checksum     sum |logits| over the first 16 results: identical inputs at every N, so it must not depend on N
  roofline     N = 1: the dominant kernel (the FC1 tcgen05 GEMM): algorithmic FLOPs per launch / its CUDA-event
               duration, against MEASURED_PEAKS.json; N > 1: the bottleneck STAGE (its GEMM + attention FLOPs over its
               event-timed kernel sequence), per-rank breakdown under `stages`
  cpu_baseline the CPU oracle port (oracle/shards.py, torch fp32 on the host cores) on a bounded sample
`--impl reference` times that CPU port as the reference arm with the same thread calibration and the same `config`
(the reference is Python and cannot travel to the GPU box; see DESIGN.md).

`--steps K` is the number of timed micro-batches in every arm. `--dump-outputs DIR` writes what the timed path returned
for its last micro-batch (the logits) as `DIR/<name>.npy` in float32: inputs and weights are seeded, so two builds run
with the same arguments can be compared output for output.
"""
import argparse
import faulthandler
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from pipeedge_b200.synth import MODEL_SPECS, hf_config, synth_input, synth_weights  # noqa: E402

WORKLOADS = {
    # name: (model, ubatch, seq_len, quant bits per hop, metric, unit)
    'vit-base': ('google/vit-base-patch16-224', 8, 0, 0, 'images/sec per pipeline', 'images/s'),
    'vit-large': ('google/vit-large-patch16-224', 16, 0, 0, 'images/sec per pipeline', 'images/s'),
    'bert-base': ('textattack/bert-base-uncased-CoLA', 32, 128, 0, 'sequences/sec per pipeline', 'sequences/s'),
    'deit-base-q8': ('facebook/deit-base-distilled-patch16-224', 32, 0, 8, 'images/sec per pipeline', 'images/s'),
    'vit-base-b1': ('google/vit-base-patch16-224', 1, 0, 0, 'images/sec per pipeline', 'images/s'),   # BASELINE configs[0]
}
N_INPUTS = 16   # distinct resident micro-batches the timed loop rotates over
DUMP_LIMIT_BYTES = 64 << 20


def dump_output(out_dir: str, name: str, t: torch.Tensor) -> None:
    """Write `t` as `out_dir/<name>.npy` in float32. Beyond DUMP_LIMIT_BYTES only a fixed, seeded sample of its rows is
    written (the same rows in every run)."""
    os.makedirs(out_dir, exist_ok=True)
    a = t.detach().float().cpu()
    if a.numel() * 4 > DUMP_LIMIT_BYTES:
        rows = max(1, DUMP_LIMIT_BYTES // (4 * a[0].numel()))
        a = a[torch.randperm(a.shape[0], generator=torch.Generator().manual_seed(0))[:rows].sort().values]
    np.save(os.path.join(out_dir, f'{name}.npy'), a.numpy())


def even_partition(layers: int, n: int):
    """Split `layers` sub-layers into n contiguous 1-based inclusive ranges, as even as possible."""
    base, rem = divmod(layers, n)
    out, cur = [], 1
    for i in range(n):
        size = base + (1 if i < rem else 0)
        out.append((cur, cur + size - 1))
        cur += size
    return out


def flops_per_item(spec, seq: int) -> float:
    """GEMMs + QK^T/PV only (SURVEY.md 8d): L * [S*(2*H*3H + 2*H*H + 2*2*H*I) + 4*S^2*H]."""
    h, i = spec.hidden, spec.inter
    return spec.blocks * (seq * (2 * h * 3 * h + 2 * h * h + 4 * h * i) + 4 * seq * seq * h)


class ClockSampler:
    """Samples nvidia-smi SM clocks and throttle reasons while the timed region runs.

    nvidia-smi needs up to a second to start on an 8-GPU box - longer than a 20-step timed phase - so the sampler is
    started ahead of the warm-up (`wait_first`), every sample is time-stamped, and the summary uses the samples that fall
    into the marked window (`mark_start` .. `mark_end`: the second warm-up phase + the timed phase, the same load back to
    back), or the sample nearest to it."""
    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int, enabled: bool = True):
        self.index, self.proc, self.lines = index, None, []
        self.t_start = self.t_end = None
        self.enabled = enabled

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line))

    def __enter__(self):
        if not self.enabled:
            return self
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.QUERY}',
                                          '--format=csv,noheader,nounits', '-lms', '25'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None
        return self

    def wait_first(self, timeout: float = 8.0):
        """Block until the first sample has arrived (nvidia-smi is up), at most `timeout` seconds."""
        deadline = time.perf_counter() + timeout
        while self.proc is not None and not self.lines and time.perf_counter() < deadline:
            time.sleep(0.01)

    def mark_start(self):
        self.t_start = time.perf_counter()

    def mark_end(self):
        self.t_end = time.perf_counter()

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.06)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self) -> dict:
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        rows = []
        for stamp, line in list(self.lines):
            parts = [p.strip() for p in line.split(',')]
            if len(parts) < 6:
                continue
            try:
                rows.append((stamp, float(parts[0]), float(parts[1]),
                             [n for n, v in zip(names, parts[2:6]) if v.lower().startswith('active')]))
            except ValueError:
                continue
        window = rows
        if self.t_start is not None and self.t_end is not None and rows:
            window = [r for r in rows if self.t_start <= r[0] <= self.t_end + 0.05]
            if not window:   # shorter than one sampling period: the sample nearest to the window
                mid = 0.5 * (self.t_start + self.t_end)
                window = [min(rows, key=lambda r: abs(r[0] - mid))]
        sm = [r[1] for r in window]
        reasons = sorted({n for r in window for n in r[3]})
        return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': max((r[2] for r in window), default=None),
                'reasons': reasons, 'samples': len(sm), 'samples_total': len(rows)}


def load_peaks() -> dict:
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path, encoding='utf-8') as fh:
            peaks = json.load(fh)
        peaks['source'] = 'measured'
        return peaks
    # /opt/skills/guides/B200_PROFILING.md fallback
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0, 'source': 'fallback'}


# ---------------------------------------------------------------------------------------------------
# CPU arm: the oracle port, timed (cpu_baseline and --impl reference share every line of this)
# ---------------------------------------------------------------------------------------------------
def usable_cores() -> int:
    """Host threads this process may really use: affinity mask, capped by a cgroup CPU quota if one is set."""
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    try:
        with open('/sys/fs/cgroup/cpu.max', encoding='utf-8') as fh:
            quota, period = fh.read().split()
        if quota != 'max':
            cores = max(1, min(cores, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return cores


def cpu_forward_timer(spec, ubatch: int, seq: int):
    """Returns (callable running one micro-batch through the whole model on the CPU, threads used, calibration log).

    "All the host threads it can use": on a many-core shared box torch's fp32 GEMMs get SLOWER past a point, so the
    thread count is calibrated - median of 3 repetitions per candidate of the FULL model (of its first two blocks when
    a full forward takes more than 0.6 s), candidates {8, 16, 32, 64, 96, all usable}."""
    from oracle import shards as osh   # the one place bench.py may execute oracle/ (as the timed CPU baseline)
    weights = synth_weights(spec, seed=0)
    model = osh.PreparedShard(spec, weights, 1, spec.layers)
    x = synth_input(spec, ubatch, seed=1, seq_len=seq or 128)
    limit = usable_cores()
    torch.set_num_threads(min(16, limit))
    model.forward(x)                      # warm-up: thread pool, oneDNN primitive caches
    t0 = time.perf_counter()
    model.forward(x)
    probe = model if time.perf_counter() - t0 < 0.6 else osh.PreparedShard(spec, weights, 1, 8)
    log = {}
    for n in sorted({min(c, limit) for c in (8, 16, 32, 64, 96, limit)}):
        torch.set_num_threads(n)
        probe.forward(x)
        reps = []
        for _ in range(3):
            t0 = time.perf_counter()
            probe.forward(x)
            reps.append(time.perf_counter() - t0)
        log[n] = statistics.median(reps)
    best = min(log, key=log.get)
    torch.set_num_threads(best)
    return (lambda: model.forward(x)), best, {'host_cores': limit,
                                              'probe': 'full model' if probe is model else '2 blocks',
                                              'median_s_by_threads': {str(k): round(v, 4) for k, v in log.items()}}


def cpu_sample(spec, ubatch: int, seq: int, unit: str, steps: int) -> dict:
    """Time `steps` forwards of the CPU port; the same routine serves `cpu_baseline` and `--impl reference`."""
    fwd, cores, cal = cpu_forward_timer(spec, ubatch, seq)
    # Warm-up until the per-forward time has settled: the first forwards of a process run ~2x slower than its steady state
    # (the allocator still maps and unmaps the 10-100 MB temporaries of every layer; r02g: 0.31 s vs 0.14 s per
    # micro-batch), which is why a 20-step arm and a 64-step arm of the same code disagreed by 2x.
    t_w = time.perf_counter()
    warm, last = 0, float('inf')
    while warm < 40 and time.perf_counter() - t_w < 12.0:
        t1 = time.perf_counter()
        fwd()
        dt1 = time.perf_counter() - t1
        warm += 1
        if warm >= 5 and dt1 > 0.93 * last:     # no longer getting faster
            break
        last = min(last, dt1)
    cal['warmup_forwards'] = warm
    t0 = time.perf_counter()
    for _ in range(steps):
        logits = fwd()
    dt = time.perf_counter() - t0
    return {'value': steps * ubatch / dt, 'unit': unit, 'cores': cores, 'kind': 'port', 'steps': steps, 'seconds': dt,
            'calibration': cal, 'logits': logits,
            'sample': f"{steps} micro-batches of {ubatch} through all {spec.layers} sub-layers, torch fp32 CPU "
                      f"({dt:.1f} s), 1 process x {cores} threads of {cal['host_cores']} usable host cores "
                      "(median-of-3 thread calibration)"}


def cpu_baseline_child(args) -> dict:
    """`cpu_baseline` of the GPU arm = the reference arm's own command in a child process.

    The CPU port's speed depends on the state of the process it runs in: on the B200 hosts (2 x Xeon 8562Y+, 16-CPU
    quota) a fresh process needs 0.30 s per ViT-B micro-batch, forward after forward, while the same code at the end of
    the GPU arm's process needed 0.14 s (scripts/cpu_arm_trajectory.py, profiles/r02_cpu_arm_trajectory.txt; neither a
    CUDA context created first nor NUMA pinning reproduces the fast regime reliably). Round 1's two CPU numbers differed by
    2-3x for that reason. Both arms now run the SAME command in the SAME kind of process, so they agree; the faster regime
    is documented in DESIGN.md section 7 and would halve every GPU / CPU ratio."""
    cmd = [sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--workload', args.workload, '--steps', '24',
           '--warmup', '2', '--gpus', '1']
    if args.ubatch:
        cmd += ['--ubatch', str(args.ubatch)]
    env = {k: v for k, v in os.environ.items() if k not in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK')}
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env, check=False)
    for line in res.stdout.splitlines():
        if line.startswith('{'):
            base = json.loads(line)['cpu_baseline']
            base['how'] = 'the reference arm (`bench.py --impl reference`) run as a child process of this one'
            return base
    return {'value': None, 'unit': None, 'cores': None, 'kind': 'port', 'sample': 'the child process failed: ' + res.stderr[-300:]}


def make_config(workload, spec, ubatch, seq_eff, parts, qbit, world) -> dict:
    """The `config` object: identical for both arms."""
    return {'workload': workload, 'model': spec.name, 'ubatch': ubatch, 'seq_len': seq_eff,
            'partition': [list(p) for p in parts], 'quant': [qbit] * (world - 1) + [0], 'n_stages': world,
            'inputs': f"{N_INPUTS} distinct synthetic micro-batches rotated (seeds 100..{100 + N_INPUTS - 1}); weights seed 0"}


def run_reference_arm(args, spec, ubatch, seq, qbit, metric, unit, workload):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return   # the CPU arm is a single process using the host cores; other ranks have no work
    world = int(os.environ.get('WORLD_SIZE', str(args.gpus)))
    res = cpu_sample(spec, ubatch, seq, unit, args.steps)
    if args.dump_outputs:
        dump_output(args.dump_outputs, 'logits', res['logits'])
    print(json.dumps({
        'impl': 'reference', 'metric': metric, 'value': res['value'], 'unit': unit, 'n_gpus': args.gpus,
        'steps': res['steps'], 'warmup': args.warmup, 'ms_per_step': res['seconds'] / res['steps'] * 1e3,
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': make_config(workload, spec, ubatch, seq or spec.tokens, even_partition(spec.layers, max(1, world)),
                              qbit, max(1, world)),
        'note': "CPU port of the reference path (oracle/shards.py) in ONE process on the host cores; the reference "
                "package is Python and cannot travel to the GPU box, and its N-rank Gloo pipeline is not what is timed",
        'cpu_baseline': {k: res[k] for k in ('value', 'unit', 'cores', 'kind', 'sample', 'calibration')},
        'e2e': {'value': res['value'], 'unit': unit, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }))


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------
def make_shard(spec, weights, layer_start, layer_end):
    from pipeedge_b200.models import ModuleShardConfig
    from pipeedge_b200.models.transformers import bert, deit, vit
    classes = {'vit': vit.ViTShardForImageClassification, 'deit': deit.DeiTShardForImageClassification,
               'bert': bert.BertShardForSequenceClassification}
    cfg = ModuleShardConfig(layer_start=layer_start, layer_end=layer_end, is_first=layer_start == 1,
                            is_last=layer_end == spec.layers)
    return classes[spec.family](hf_config(spec), cfg, weights)


def dominant_kernel_us(spec, ubatch, seq, dev) -> float:
    """Average launch duration (us) of the dominant kernel - the FC1 GEMM with its GELU epilogue - as it runs inside a
    step: back-to-back launches in a CUDA graph (as in the stage's graph), each on a different weight copy so that the
    weights stream from HBM like in a forward (copies total > 126 MB L2), CUDA events on the launching stream."""
    from pipeedge_b200 import _lib, ops
    m, n, k = ubatch * seq, spec.inter, spec.hidden
    copies = max(8, int(200e6 // (n * k * 2)) + 1)
    gen = torch.Generator(device=dev).manual_seed(7)
    a = (torch.randn(m, k, device=dev, generator=gen)).half()
    ws = [(torch.randn(n, k, device=dev, generator=gen) * 0.02).half() for _ in range(copies)]
    bias = torch.zeros(n, device=dev)
    out = torch.empty(m, n, device=dev, dtype=torch.float16)
    side = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(side):
        for i in range(3):
            ops.linear(a, ws[i], bias, _lib.PE_EPI_GELU_F16, out=out, static_w=True)
        side.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            for w in ws:
                ops.linear(a, w, bias, _lib.PE_EPI_GELU_F16, out=out, static_w=True)
        for _ in range(3):
            graph.replay()
        reps = 10
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record(side)
        for _ in range(reps):
            graph.replay()
        end.record(side)
        side.synchronize()
    return start.elapsed_time(end) * 1e3 / (reps * copies)


def roofline_from_profile(shard, sample, spec, ubatch, seq, peaks, step_ms=None) -> dict:
    """Per-kernel CUDA-event times of live eager forwards -> roofline of the dominant kernel (FC1 GEMM)."""
    stage = shard.stage
    acc = {}
    for _ in range(3):
        for kind, ms in stage.profile(sample):
            acc.setdefault(kind, []).append(ms)
    m = ubatch * seq
    h, i = spec.hidden, spec.inter
    flops = {'gemm_qkv': 2.0 * m * 3 * h * h, 'gemm_out': 2.0 * m * h * h, 'gemm_fc1': 2.0 * m * i * h,
             'gemm_fc2': 2.0 * m * h * i, 'attention': 4.0 * ubatch * seq * seq * h}
    breakdown = {}
    for kind, vals in acc.items():
        avg_ms = sum(vals) / len(vals)
        entry = {'launches_per_forward': len(vals) // 3, 'avg_us': avg_ms * 1e3}
        if kind in flops:
            entry['tflops'] = flops[kind] / (avg_ms * 1e-3) / 1e12
        breakdown[kind] = entry
    total_ms = sum(sum(v) for v in acc.values()) / 3
    dom = 'gemm_fc1'
    # The per-kernel times above are bracketed by events, which serialise the launches (no programmatic-dependent-launch
    # overlap) and add event latency to every kernel: they are upper bounds, good for shares. The dominant kernel's
    # launch duration proper is measured back to back in a graph, as it runs in the step.
    dom_us = dominant_kernel_us(spec, ubatch, seq, sample.device)
    achieved = flops[dom] / (dom_us * 1e-6) / 1e12
    peak = peaks['bf16_tflops_sustained']   # timed inside a long step
    launches = breakdown[dom]['launches_per_forward']
    traffic = None   # DRAM bytes per launch of this kernel from the committed `ncu --set full` capture
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'profiles', 'ncu_traffic.json')) as f:
            traffic = json.load(f)['dram_bytes_per_launch']
    except (OSError, KeyError, ValueError):
        pass
    return {'bound': 'tensor', 'kernel': 'gemm_tcgen05_kernel<PE_EPI_GELU_F16> (FC1)', 'achieved': achieved,
            'peak': peak, 'unit': 'TFLOP/s', 'frac': achieved / peak, 'traffic': traffic,
            'peak_source': f"{peaks['source']} bf16_tflops_sustained (MEASURED_PEAKS.json)",
            'flops_per_launch': flops[dom], 'avg_launch_us': dom_us,
            'method': 'CUDA events around a graph of back-to-back launches on distinct weight copies (> L2)',
            'share_of_step': (launches * dom_us * 1e-3 / step_ms) if step_ms else sum(acc[dom]) / 3 / total_ms,
            'share_of_step_event_bracketed': sum(acc[dom]) / 3 / total_ms,
            'all_gemm_tflops': sum(flops[k] * breakdown[k]['launches_per_forward'] for k in flops if k in breakdown
                                   and k.startswith('gemm')) / (sum(sum(acc[k]) for k in acc if k.startswith('gemm'))
                                                                / 3 * 1e-3) / 1e12,
            'breakdown': breakdown, 'eager_forward_ms': total_ms}


def stage_roofline(shard, spec, ubatch, seq, parts_rank, dev) -> dict:
    """This rank's stage, kernel by kernel (CUDA events around every launch of eager forwards: upper bounds, launch
    overlap is lost): GEMM + attention FLOPs of its sub-layers over the sum of its kernel times."""
    stage = shard.stage
    lo, hi = parts_rank
    if stage.in_is_tuple:
        width = stage.inter if stage.first_sub == 3 else stage.hidden
        sample = (torch.randn(ubatch, seq, width, device=dev), torch.randn(ubatch, seq, stage.hidden, device=dev))
    else:
        sample = torch.randn(ubatch, seq, stage.hidden, device=dev)
    acc = {}
    reps = 3
    for _ in range(reps):
        for kind, ms in stage.profile(sample):
            acc[kind] = acc.get(kind, 0.0) + ms
    m, h, i = ubatch * seq, spec.hidden, spec.inter
    per_sub = {0: 2.0 * m * 3 * h * h + 4.0 * ubatch * seq * seq * h, 1: 2.0 * m * h * h, 2: 2.0 * m * i * h,
               3: 2.0 * m * h * i}
    flops = sum(per_sub[(layer - 1) % 4] for layer in range(lo, hi + 1))
    total_ms = sum(acc.values()) / reps
    return {'layers': [lo, hi], 'flops': flops, 'eager_ms': total_ms, 'tflops': flops / (total_ms * 1e-3) / 1e12,
            'kernel_ms': {k: round(v / reps, 4) for k, v in acc.items()}}


def run_gpu(args, spec, ubatch, seq, qbit, metric, unit, workload):
    """All N: one stage per rank through DistP2pContext / DistP2pPipelineStage (the runtime.py path)."""
    import contextlib
    import torch.distributed as dist
    from pipeedge_b200.comm.p2p import DistP2pContext, DistP2pPipelineStage
    import runtime as rt
    rank, world = int(os.environ.get('RANK', '0')), int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', rank)) % torch.cuda.device_count()
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    os.environ.setdefault('PIPEEDGE_MAX_UBATCH', str(max(ubatch, 8)))
    parts = even_partition(spec.layers, world)
    weights = synth_weights(spec, seed=0)
    shard = make_shard(spec, weights, *parts[rank])
    del weights
    steps, warmup = args.steps, max(3, args.warmup)
    seq_eff = seq or spec.tokens
    dim1 = seq_eff if spec.family == 'bert' else 0
    last = world - 1
    # the same module hooks runtime.py installs; the native pipeline performs them inside its link kernels
    shard.register_buffer('quant_bit', torch.tensor(qbit if rank != last else 0), persistent=False)
    if rank != last:
        shard.register_forward_hook(rt.forward_hook_quant_encode)
    if rank != 0:
        shard.register_forward_pre_hook(rt.forward_pre_hook_quant_decode)

    got = []
    res_done = threading.Event()
    target = {'n': 0}

    def results_cb(t):
        got.append(t)
        if len(got) >= target['n']:
            res_done.set()

    phase_q = []
    phase_evt = threading.Event()
    stop = threading.Event()

    def handle_cmd(cmd, tensors):
        if cmd == 0:
            stop.set()
        elif cmd == 2:     # phase boundary: [kind]
            phase_q.append(int(tensors[0][0]))
            phase_evt.set()

    def wait_cmd():
        assert phase_evt.wait(900), "no phase command from rank 0"
        kind = phase_q.pop(0)
        if not phase_q:
            phase_evt.clear()
        return kind

    def allmax(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    def allsum(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t[0])

    def barrier():
        if world > 1:
            dist.barrier()

    out = None
    ctx_mgr = DistP2pContext(('gloo',), {'world_size': world, 'rank': rank}, handle_cmd) if world > 1 \
        else contextlib.nullcontext()
    with ctx_mgr as ctx:
        src = None if world == 1 else (last if rank == 0 else rank - 1)
        dst = None if world == 1 else (0 if rank == last else rank + 1)
        with DistP2pPipelineStage(src, dst, shard, results_cb if rank == 0 else None) as stage_ctx:
            native = stage_ctx.native
            if native is None:
                raise SystemExit("bench.py: the native pipeline was not selected (PIPEEDGE_NATIVE=0 or a rank without a "
                                 "B200 shard?)")
            stage_ctx.prepare(ubatch, dim1)          # graph capture happens here, before any timed or warm-up step
            inputs_host = inputs_dev = None
            if rank == 0:
                inputs_host = [synth_input(spec, ubatch, seed=100 + i, seq_len=seq or 128).pin_memory()
                               for i in range(N_INPUTS)]
                inputs_dev = [x.to(dev) for x in inputs_host]
            torch.cuda.synchronize()
            barrier()

            def run_phase(n, host):
                """Rank 0 feeds n micro-batches and collects n results; every rank times its device window."""
                native.timing_reset()
                barrier()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                if rank == 0:
                    got.clear()
                    res_done.clear()
                    target['n'] = n
                    src_list = inputs_host if host else inputs_dev
                    for i in range(n):
                        stage_ctx.enqueue_tensor(src_list[i % N_INPUTS])
                    assert res_done.wait(900), "pipeline results did not arrive"
                    native.sync()
                    torch.cuda.synchronize()
                    wall = time.perf_counter() - t0
                    if world > 1:
                        ctx.cmd_broadcast(2, (torch.tensor([1]),))     # every result is back: the phase is over
                else:
                    wait_cmd()
                    native.sync()
                    wall = time.perf_counter() - t0
                stage_ctx.check_workers()
                tim = native.timing()
                barrier()
                return wall, tim

            sampler = ClockSampler(local, enabled=rank == 0)   # the line reports the data rank's GPU
            sampler.__enter__()
            sampler.wait_first()
            wall_w, _ = run_phase(warmup, False)
            # ... and keep going (untimed) until the GPU has been busy for ~0.3 s: W micro-batches are a few ms of
            # work, not enough for the clocks to leave their idle state
            extra = 0
            if rank == 0:
                per_step = max(wall_w / warmup, 1e-4)
                extra = int(min(2000, max(0.0, 0.3 - wall_w) / per_step))
            # the clock sampler spans the second warm-up phase too: a 20-step timed phase lasts ~10 ms, less than one
            # nvidia-smi sampling period, and both phases run the same load back to back
            clocks = sampler
            clocks.mark_start()
            run_phase(max(extra, 1), False)
            _, tim = run_phase(steps, False)
            clocks.mark_end()
            clocks.__exit__(None, None, None)
            ms_rank = max(tim['compute_ms'], tim['results_ms'])
            ms = allmax(ms_rank)
            kernels = allsum(float(tim['kernels'])) + steps     # + the data rank's results-get kernel per micro-batch
            checksum = None
            if rank == 0:
                checksum = float(sum(t.double().abs().sum() for t in got[:N_INPUTS]))
                if args.dump_outputs:
                    dump_output(args.dump_outputs, 'logits', got[-1])
            run_phase(warmup, True)
            e2e_wall, _ = run_phase(steps, True)
            e2e_wall = allmax(e2e_wall) if world > 1 else e2e_wall
            e2e_checksum = float(sum(t.double().abs().sum() for t in got[:N_INPUTS])) if rank == 0 else None
            # per-stage kernel roofline (eager, event-bracketed) after the timed phases
            with torch.cuda.stream(torch.cuda.Stream(device=dev)):
                mine = stage_roofline(shard, spec, ubatch, seq_eff, parts[rank], dev)
                torch.cuda.current_stream().synchronize()
            stages = [mine]
            if world > 1:
                stages = [None] * world
                dist.all_gather_object(stages, mine)
            if rank == 0:
                peaks = load_peaks()
                value = steps * ubatch / (ms * 1e-3)
                total_flops = flops_per_item(spec, seq_eff)
                h2d = inputs_host[0].numel() * inputs_host[0].element_size()
                d2h = got[0].numel() * got[0].element_size()
                cfg = make_config(workload, spec, ubatch, seq_eff, parts, qbit, world)
                hop_bytes = ubatch * seq_eff * spec.hidden * (1 if qbit == 8 else 4) if world > 1 else 0
                out = {
                    'metric': metric, 'value': value, 'unit': unit, 'n_gpus': world, 'steps': steps, 'warmup': warmup,
                    'ms_per_step': ms / steps, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
                    'dtype': 'f16', 'data': 'synthetic', 'config': cfg,
                    'pipeline': {'impl': 'native: one CUDA graph per stage micro-batch, peer-memory links (cudaIpc rings, '
                                         'device-polled flags)' + (f', {qbit}-bit QuantPipe fused into the send kernel' if qbit else ''),
                                 'graph_kernels_per_microbatch': native.graph_kernels.get((ubatch, dim1)),
                                 'hop_bytes_per_microbatch': hop_bytes,
                                 'l2': f"timed loop rotates over {N_INPUTS} distinct resident micro-batches"
                                       + ("; the stage's fp16 weights "
                                          f"({spec.blocks * (4 * spec.hidden ** 2 + 2 * spec.hidden * spec.inter) * 2 / 1e6:.0f} MB) "
                                          "exceed the 126 MB L2 and stream from HBM every step" if world == 1 else
                                          "; per-stage weights may be L2-resident, as in steady-state serving")},
                    'clocks': clocks.summary(),
                    'e2e': {'value': steps * ubatch / e2e_wall, 'unit': unit, 'h2d_bytes_per_step': h2d,
                            'd2h_bytes_per_step': d2h, 'ms_per_step': e2e_wall / steps * 1e3},
                    'gpu_launches': int(kernels),
                    'checksum': checksum, 'checksum_e2e': e2e_checksum,
                    'model_tflops': value * total_flops / 1e12,
                    'model_frac_of_sustained_peak_per_gpu': value * total_flops / 1e12 / world / peaks['bf16_tflops_sustained'],
                    'stages': stages,
                }
                if world == 1:
                    with torch.cuda.stream(torch.cuda.Stream(device=dev)):
                        inner = shard.vit if spec.family != 'bert' else shard.bert
                        emb = inner._embed(inputs_dev[0])   # noqa: protected access - the stage's input
                        out['roofline'] = roofline_from_profile(shard, emb, spec, ubatch, seq_eff, peaks, step_ms=ms / steps)
                else:
                    worst = max(stages, key=lambda st: st['eager_ms'])
                    out['roofline'] = {'bound': 'tensor', 'kernel': f"bottleneck stage {worst['layers']} (tcgen05 GEMMs + attention)",
                                       'achieved': worst['tflops'], 'peak': peaks['bf16_tflops_sustained'], 'unit': 'TFLOP/s',
                                       'frac': worst['tflops'] / peaks['bf16_tflops_sustained'], 'traffic': None,
                                       'note': 'stage FLOPs / sum of its event-bracketed kernel times (upper bound on time); the '
                                               'per-kernel roofline is in the N=1 line',
                                       'pipeline_frac_of_stage_bound': (ms / steps) / worst['eager_ms']}
            if rank == 0 and world > 1:
                ctx.cmd_broadcast(0)
            elif world > 1:
                stop.wait(60)
    if rank == 0 and out is not None:
        if not args.no_cpu_baseline and world == 1:
            out['cpu_baseline'] = cpu_baseline_child(args)
        print(json.dumps(out))


def run_quick(args, spec, ubatch, seq):
    """`--quick`: a bare resident-input loop of direct shard calls on one GPU (for ncu runs)."""
    from pipeedge_b200 import ops
    torch.cuda.set_device(0)
    dev = torch.device('cuda', 0)
    shard = make_shard(spec, synth_weights(spec, seed=0), 1, spec.layers)
    shard.use_cuda_graph = not args.eager
    xs = [synth_input(spec, ubatch, seed=100 + i, seq_len=seq or 128).to(dev) for i in range(4)]
    stream = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(stream):
        for i in range(max(3, args.warmup)):
            shard(xs[i % 4])
        stream.synchronize()
        l0 = ops.launch_count()
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record(stream)
        for i in range(args.steps):
            logits = shard(xs[i % 4])
        end.record(stream)
        torch.cuda.synchronize()
    ms = start.elapsed_time(end)
    if args.dump_outputs:
        dump_output(args.dump_outputs, 'logits', logits)
    print(json.dumps({'quick': True, 'value': args.steps * ubatch / (ms * 1e-3), 'ms_per_step': ms / args.steps,
                      'gpu_launches': int(ops.launch_count() - l0)}))


def main():
    faulthandler.enable()   # a native crash in any thread prints every thread's Python stack to stderr
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None, help='timed micro-batches (default 300; 24 with --impl reference)')
    ap.add_argument('--warmup', type=int, default=20)
    ap.add_argument('--impl', choices=['ours', 'reference'], default='ours')
    ap.add_argument('--workload', choices=sorted(WORKLOADS), default='vit-base')
    ap.add_argument('--ubatch', type=int, default=0)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--quick', action='store_true', help='only a resident-input loop of direct shard calls (for ncu runs)')
    ap.add_argument('--eager', action='store_true', help='with --quick: no CUDA graph (every kernel visible to ncu)')
    ap.add_argument('--dump-outputs', metavar='DIR', help="write the timed path's last outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 24 if args.impl == 'reference' else 300   # a bounded CPU sample by default
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    model, ubatch, seq, qbit, metric, unit = WORKLOADS[args.workload]
    ubatch = args.ubatch or ubatch
    spec = MODEL_SPECS[model]
    if args.impl == 'reference':
        run_reference_arm(args, spec, ubatch, seq, qbit, metric, unit, args.workload)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - pipeedge_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    if args.quick:
        run_quick(args, spec, ubatch, seq)
        return
    run_gpu(args, spec, ubatch, seq, qbit, metric, unit, args.workload)
    sys.stdout.flush()
    sys.stderr.flush()


if __name__ == '__main__':
    main()
