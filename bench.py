#!/usr/bin/env python
"""Headline benchmark: tokens/sec of LLaMA-7B int4 g128 batch-1 decode on B200 (BASELINE.json metric),
plus the roofline of the dominant kernel and the CPU baseline, as ONE JSON line on rank 0.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 7b|13b-int3|65b|prefill]   # our arm
    python bench.py --impl reference [--steps K] [--warmup W]                                  # the reference's arithmetic on the host cores
    ... --dump-outputs DIR   # also write what the timed path computed in its last step as DIR/<name>.npy

The inputs are seeded, so two builds run with the same arguments can be compared output for output.  Compare the decode outputs with a
tolerance: the persistent kernel combines split-K partial sums with unordered fp32 atomics, so even one build differs from run to run by
fp16 rounding noise (DESIGN.md, run-to-run spread; on a B200 at 1000 W, 32 layers: logits within 0.023 of an rms of 1.29, same greedy token).

A "step" is one decoded token: one replay of the captured CUDA graph of gptq_llama_decode_step (ONE persistent kernel) over a
random-init LLaMA-7B-shaped GPTQ model (32 distinct layers, 3.6 GB of packed weights per step, i.e. far larger than the 126 MB
L2, so every step streams from HBM) at context position seq-1 = 2047.
N > 1 (torchrun): the path does not shard at this size ("replicas only", DESIGN.md): every rank decodes its own sequence on its
own GPU, no data-path collective; value = total tokens/s, scaling = weak.
--config selects the other BASELINE.json configurations (13b-int3 = config 4, 65b = the config-5 model on one GPU, prefill = config 3);
the default is config 2, the one the metric is quoted on.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, 'gptq-for-llama_b200')):
    if p not in sys.path:
        sys.path.insert(0, p)


def _host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


if '--impl' in sys.argv and 'reference' in sys.argv:
    # the CPU arm sets its thread count itself (torchrun exports OMP_NUM_THREADS=1, which must not leak into it), before torch / libgomp
    # are loaded.  32 threads: the restatement is bound by its bit-unpacking loop per 32-column block and two OpenMP runtimes are alive in
    # the process (torch's and the oracle's); with all 128 hardware threads of the B200 hosts spinning in both, a token took 3.5 - 13.8 s from
    # run to run, with 8 threads of the build container 4.6 s.  Passive waiting keeps idle workers off the cores.
    os.environ['OMP_NUM_THREADS'] = os.environ.get('BENCH_CPU_THREADS', str(min(32, _host_threads())))
    os.environ['OMP_WAIT_POLICY'] = 'passive' 

import torch  # noqa: E402

METRIC = 'tokens/sec LLaMA-7B int4 g128 batch=1; matvec HBM GB/s vs 8 TB/s roofline'
SEQ = 2048
# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of llama_decode_mega_kernel on the 32-layer model at context 2047
# (ncu --set full, profiles/r2_mega_summary.txt, profiles/r2_mega_final.ncu-rep)
NCU_TRAFFIC_BYTES = {'7b': 4737481728}  # 4.7074 GB read + 30.1 MB written (algorithmic: 4.7084 GB)
CONFIGS = {  # name -> (size, bits, act_order, BASELINE.json config)
    '7b': ('7b', 4, False, 'LLaMA-7B int4 g128 batch=1 decode'),
    '13b-int3': ('13b', 3, True, 'LLaMA-13B int3 g128 act-order batch=1 decode'),
    '65b': ('65b', 4, False, 'LLaMA-65B int4 g128 batch=1 decode on ONE GPU'),
    '65b-tp': ('65b', 4, False, 'LLaMA-65B int4 g128 batch=1 decode, tensor-parallel over the N GPUs (BASELINE config 5)'),
}
GROUP = 128
DUMP_LIMIT_BYTES = 64 << 20
PREFILL_DUMP_ROWS = 256  # seeded sample of the M = 65536 prefill rows that --dump-outputs writes


def dump_outputs(out_dir, arrays):
    """Write each tensor as <out_dir>/<name>.npy: integers as float64 (exact), everything else as float32."""
    import numpy as np
    conv = {k: v.detach().cpu().numpy().astype(np.float32 if v.is_floating_point() else np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in conv.values())
    assert total <= DUMP_LIMIT_BYTES, f'outputs to dump are {total} bytes, more than {DUMP_LIMIT_BYTES}'
    os.makedirs(out_dir, exist_ok=True)
    for k, a in conv.items():
        np.save(os.path.join(out_dir, k + '.npy'), a)


def alg_bytes_qlinear(K, N, bits, M=1, gs=GROUP):
    """SURVEY.md 8(d): qweight + scales + qzeros + g_idx + x + out."""
    G = (K + gs - 1) // gs
    return K * N * bits // 8 + G * N * 2 + G * N * bits // 8 + 4 * K + 2 * M * K + 2 * M * N


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        d = json.load(open(path))
        return d.get('hbm_gbs', 6650.0), d.get('bf16_tflops', 1590.0), d.get('bf16_tflops_sustained', 1400.0), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 1590.0, 1400.0, 'fallback (B200_PROFILING.md)'


# ----------------------------------------------------------------------------------------------------
# CPU arm: the oracle's C/OpenMP restatement of the reference kernels (the reference has no CPU forward), timed on
# WHOLE decoded tokens of the same workload: 32 x (RMSNorm, qkv, RoPE-free attention over a 2047-token cache, o_proj, RMSNorm,
# fused gate/up + SwiGLU, down) + final norm + fp16 lm_head.  One layer's tensors are reused for the 32 layers (they fit the
# host's last-level cache the second time round, which favours the CPU).
# ----------------------------------------------------------------------------------------------------
class CpuToken:
    def __init__(self):
        from oracle import gptq_oracle as O
        from oracle import cref
        self.O = O
        self.Q = cref if cref.available() else O  # C/OpenMP restatement (all host threads) when built, else the numpy/torch one
        self.kind = 'C/OpenMP (oracle/qlinear_ref.c)' if cref.available() else 'numpy/torch (oracle/gptq_oracle.py)'
        self.H, self.I, self.NH, self.V, self.L = 4096, 11008, 32, 32000, 32
        H, I = self.H, self.I
        shapes = {'qkv': (H, 3 * H), 'o': (H, H), 'gate': (H, I), 'up': (H, I), 'down': (I, H)}
        self.W = {k: O.random_packed(K, N, 4, GROUP, seed=i)[:4] for i, (k, (K, N)) in enumerate(shapes.items())}
        g = torch.Generator().manual_seed(0)
        self.x = torch.randn(1, H, generator=g).half()
        self.nw = torch.ones(H).half()
        self.kc = (torch.randn(self.NH, SEQ, H // self.NH, generator=g) * 0.5).half()
        self.vc = (torch.randn(self.NH, SEQ, H // self.NH, generator=g) * 0.5).half()
        self.lm_head = (torch.randn(self.V, H, generator=g) * 0.02).half()

    def token(self):
        O, Q, W, H, NH = self.O, self.Q, self.W, self.H, self.NH
        x = self.x
        for _ in range(self.L):
            qkv = Q.qlinear_fwd(O.rmsnorm_fwd(x, self.nw, 1e-6), *W['qkv'], 4).view(3, NH, H // NH)
            s = torch.einsum('hd,htd->ht', qkv[0].float(), self.kc.float()) * (H // NH)**-0.5
            att = torch.einsum('ht,htd->hd', torch.softmax(s, -1), self.vc.float()).half().reshape(1, H)
            x = x + Q.qlinear_fwd(att, *W['o'], 4)
            mid = Q.fused_mlp_fwd(O.rmsnorm_fwd(x, self.nw, 1e-6), W['gate'], W['up'], 4)
            x = (x + Q.qlinear_fwd(mid, *W['down'], 4)) * 0.5  # keep the synthetic residual bounded
        return O.rmsnorm_fwd(x, self.nw, 1e-6).float() @ self.lm_head.float().t()

    def time_tokens(self, steps, warmup):
        for _ in range(warmup):
            self.token()
        ts = []
        for _ in range(steps):
            t0 = time.perf_counter()
            self.logits = self.token()
            ts.append(time.perf_counter() - t0)
        return ts


def cpu_baseline(steps=2, warmup=1):
    c = CpuToken()
    ts = c.time_tokens(steps, warmup)
    t = statistics.median(ts)
    threads = int(os.environ.get('OMP_NUM_THREADS', _host_threads()))
    torch.set_num_threads(min(threads, torch.get_num_threads()) if 'OMP_NUM_THREADS' in os.environ else torch.get_num_threads())
    return {
        'value': 1.0 / t, 'unit': 'tokens/s', 'cores': threads, 'kind': 'port',
        'sample': f'oracle {c.kind} restatement of matmul_248 / fusedmatmul_248 on {threads} host threads: {steps} WHOLE decoded tokens (32 layers x 5 quantized linears at '
                  f'M=1 + attention over 2047 cached tokens + fp16 lm_head), median {t:.2f} s/token; one layer\'s tensors reused for all 32 layers',
    }, ts, c.logits


def cpu_baseline_subprocess(steps=3, warmup=1):
    """The cpu_baseline leg of our arm = the reference arm itself on a short sample, in its own process (its thread settings must be in
    place before torch / libgomp load, and must not disturb the GPU arm)."""
    try:
        out = subprocess.run([sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--steps', str(steps), '--warmup', str(warmup)], capture_output=True,
                             text=True, timeout=240, env={k: v for k, v in os.environ.items() if k not in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK', 'OMP_NUM_THREADS')})
        line = [ln for ln in out.stdout.splitlines() if ln.startswith('{')][-1]
        return json.loads(line)['cpu_baseline']
    except Exception as e:  # the GPU line must not depend on the host leg
        return {'value': None, 'unit': 'tokens/s', 'cores': None, 'kind': 'port', 'sample': f'cpu leg failed: {e!r}'}


def run_reference(args):
    """`--impl reference`: the reference's own arithmetic on the host cores, rank 0 only."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    torch.set_num_threads(int(os.environ['OMP_NUM_THREADS']))
    steps = args.steps  # a few seconds per token
    warm = min(max(0, args.warmup), 1)
    base, ts, logits = cpu_baseline(steps, warm)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {'logits': logits})
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': base['value'], 'unit': 'tokens/s', 'n_gpus': args.gpus, 'steps': steps, 'warmup': warm,
        'ms_per_step': statistics.mean(ts) * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f16', 'data': 'synthetic',
        'config': {'workload': f'LLaMA-7B int4 g128 batch=1 decode, context {SEQ - 1} (seq={SEQ}), 32 layers, random-init packed weights',
                   'note': f'CPU arm: {steps} whole tokens; same workload as the GPU arm'},
        'cpu_baseline': base,
        'e2e': {'value': base['value'], 'unit': 'tokens/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.FIELDS}', '--format=csv,noheader,nounits', '-lms', '100', '-i', str(index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            pass

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, pw, reasons = [], [], [], set()
        for ln in out.strip().splitlines():
            f = [t.strip() for t in ln.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
                pw.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'power_w_max': max(pw) if pw else None, 'samples': len(sm),
                'reasons': sorted(reasons)}


def timed(fn, steps, dist_on):
    """EXACTLY `steps` calls of fn bracketed by barrier + synchronize; device time from CUDA events."""
    import torch.distributed as dist
    if dist_on:
        dist.barrier()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    if dist_on:
        dist.barrier()
    return a.elapsed_time(b) / 1e3


def run_decode(args):
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    dist_on = world > 1
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if dist_on:
        dist.init_process_group('nccl', device_id=dev)
    from gptq_b200 import engine, ops

    size, bits, act, title = CONFIGS[args.config]
    steps, warm = args.steps, max(3, args.warmup)
    tp = args.config.endswith('-tp') and world > 1  # ONE sequence sharded over the ranks (strong scaling) instead of one replica per rank
    if tp:
        dec = engine.synthetic_llama_tp(size, rank, world, bits=bits, groupsize=GROUP, device=str(dev), seed=0, max_seq=SEQ)
    else:
        dec = engine.synthetic_llama(size, bits=bits, groupsize=GROUP, act_order=act, device=str(dev), seed=rank, max_seq=SEQ)
    # synthetic context: the cache holds seq-1 = 2047 tokens of random K/V; the step decodes token 2048
    gen = torch.Generator(device=dev).manual_seed(1000 + rank)
    dec.k_cache.normal_(0, 0.5, generator=gen)
    dec.v_cache.normal_(0, 0.5, generator=gen)
    pos = SEQ - 1
    dec.positions.fill_(pos)
    dec.tokens.fill_(1)

    # ---- device-resident arm: inputs already in HBM ------------------------------------------------
    for _ in range(warm):
        dec.step()
    torch.cuda.synchronize()
    assert bool(torch.isfinite(dec.logits).all()), 'non-finite logits'
    sampler = ClockSampler(local) if rank == 0 else None
    t_dev = timed(dec.step, steps, dist_on)
    # what the caller of the last timed step receives: logits, the greedy next token, and the K/V the step wrote at `pos` of every layer
    # (taken now: the end-to-end arm below feeds the tokens it picks back in)
    outputs = {'logits': dec.logits.float().cpu(), 'next_tokens': dec.next_tokens.cpu(), 'k_cache_at_pos': dec.k_cache[:, :, :, pos].float().cpu(),
               'v_cache_at_pos': dec.v_cache[:, :, :, pos].float().cpu()} if args.dump_outputs else None

    # ---- end-to-end arm: host token in -> H2D -> step -> D2H logits, every step -----------------------
    tok_host = torch.ones(1, dtype=torch.int32).pin_memory()
    pos_host = torch.full((1, ), pos, dtype=torch.int32).pin_memory()
    logits_host = torch.empty(1, dec.vocab, dtype=torch.float16).pin_memory()

    def e2e_step():
        dec.tokens.copy_(tok_host, non_blocking=True)
        dec.positions.copy_(pos_host, non_blocking=True)
        dec.step()
        logits_host.copy_(dec.logits, non_blocking=True)
        torch.cuda.current_stream().synchronize()  # the caller needs the logits before it can pick the next token
        tok_host[0] = int(logits_host[0, :8].float().argmax())  # touch the result on the host

    for _ in range(warm):
        e2e_step()
    t_e2e = timed(e2e_step, steps, dist_on)
    clocks = sampler.stop() if sampler else None

    # ---- the drop-in op in isolation: standalone fused gate/up matvec (gptq_fused_mlp_fwd) over the layers' distinct weights ------
    mlp = None
    if bits == 4 and not act and not tp:
        x = torch.randn(1, dec.hidden, device=dev).half()
        gates = [(ly['gate'], ly['up']) for ly in dec.layers]

        def mlp_all():
            for g, u in gates:
                ops.fused_mlp(x, (g.qweight, g.scales, g.qzeros, g.g_idx), (u.qweight, u.scales, u.qzeros, u.g_idx), bits, GROUP)

        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            mlp_all()
            side.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side):
                mlp_all()
        torch.cuda.synchronize()
        for _ in range(3):
            graph.replay()
        reps = 10
        t_k = timed(graph.replay, reps, False) / (reps * len(gates))
        kbytes = 2 * alg_bytes_qlinear(dec.hidden, dec.intermediate, bits) - 2 * dec.hidden  # two weights, x read once
    peak, _, _, peak_src = measured_peaks()

    # max over ranks, whole-job aggregate
    tt = torch.tensor([t_dev, t_e2e], device=dev, dtype=torch.float64)
    if dist_on:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_dev, t_e2e = tt.tolist()
    if rank == 0:
        base = cpu_baseline_subprocess() if (world == 1 and args.config == '7b') else None
        H, I, V, L = dec.hidden, engine.LLAMA_SHAPES[size][1], dec.vocab, len(dec.layers)
        jobs = 1 if tp else world  # sequences decoded concurrently
        # algorithmic bytes per token (SURVEY.md 8(d)): quant linears of the CHECKPOINT (not of derived buffers) + fp16 lm_head + KV cache read at this context
        per_layer = alg_bytes_qlinear(H, 3 * H, bits) + alg_bytes_qlinear(H, H, bits) + 2 * alg_bytes_qlinear(H, I, bits) + alg_bytes_qlinear(I, H, bits)
        kv = 2 * L * SEQ * H * 2
        step_bytes = L * per_layer + V * H * 2 + kv
        t_step = t_dev / steps
        line = {
            'metric': METRIC if args.config == '7b' else f'tokens/sec {title}', 'value': jobs * steps / t_dev, 'unit': 'tokens/s', 'n_gpus': world, 'steps': steps,
            'warmup': warm, 'ms_per_step': t_step * 1e3, 'higher_is_better': True, 'scaling': 'strong' if tp else 'weak', 'vs_baseline': None, 'dtype': 'f16', 'data': 'synthetic',
            'config': {
                'workload': f'{title}, context {pos} (seq={SEQ}), {L} layers, random-init packed weights',
                'parallelism': (f'tp{world}: heads / MLP columns sharded, o_proj and down_proj partial sums RED-added into every rank over NVLink inside the kernel' if tp else
                                'replicas only (one independent sequence per GPU, no data-path collective)' if world > 1 else 'single GPU'),
                'l2': f'each step streams {L * per_layer / 1e9:.1f} GB of weights + {kv / 1e9:.2f} GB of KV cache (inputs >> 126 MB L2); no explicit flush needed',
                'arithmetic': 'raw int4 nibbles x fp16 activations on the tensor pipe (mma.sync, exact products, fp32 accumulate), fp16 scale and zero applied once per '
                              'quantisation group on the fp32 accumulator, fp16 store; within 1e-3 of the reference kernel (tests/)',
            },
            'e2e': {'value': jobs * steps / t_e2e, 'unit': 'tokens/s', 'h2d_bytes_per_step': 8, 'd2h_bytes_per_step': dec.vocab * 2,
                    'note': 'host token+position (pinned) -> H2D -> CUDA-graph decode step -> D2H fp16 logits, synchronised every step'},
            'gpu_launches': dec.launches_per_step() * steps,
            'roofline': None,
            'clocks': clocks,
        }
        assert dec.launches_per_step() == 1, 'the persistent kernel must be the measured path'
        # the whole token is ONE persistent kernel: its launch duration is the step time measured above with CUDA events
        line['roofline'] = {'bound': 'hbm', 'kernel': 'llama_decode_mega_kernel (persistent decode step: all quantized matvecs + attention + lm_head of a token)',
                            'achieved': step_bytes / t_step / 1e9 / (world if tp else 1), 'peak': peak, 'unit': 'GB/s',
                            'frac': step_bytes / t_step / 1e9 / peak / (world if tp else 1), 'peak_source': peak_src + (' per GPU' if tp else ''),
                            'bytes_per_launch': step_bytes, 'us_per_launch': t_step * 1e6, 'frac_of_8TBs': step_bytes / t_step / 8e12,
                            'traffic': NCU_TRAFFIC_BYTES.get(args.config), 'traffic_source': 'dram__bytes_read.sum + dram__bytes_write.sum, ncu --set full, profiles/'}
        if mlp is None and bits == 4 and not act and not tp:
            ach = kbytes / t_k / 1e9
            line['roofline']['standalone_fused_mlp'] = {'kernel': 'qmatvec_int4_kernel<dual> (standalone gptq_fused_mlp_fwd, timed alone over the layers\' distinct weights)',
                                                        'achieved': ach, 'frac': ach / peak, 'bytes_per_launch': kbytes, 'us_per_launch': t_k * 1e6}
        ref_path = os.path.join(ROOT, 'profiles', 'r2_reference_triton_decode.json')
        if args.config == '7b' and os.path.exists(ref_path):
            try:
                rt = json.loads(open(ref_path).readline())
                line['reference_triton'] = {'tokens_per_s': rt['tokens_per_s'], 'ms_per_token': rt['ms_per_token'],
                                            'source': 'profiles/r2_reference_triton_decode.json: the unmodified reference modules (Triton kernels) on a B200 of this pool, '
                                                      'measured separately by tools/refshim/ref_decode_bench.py; not re-measured in this run'}
            except (ValueError, KeyError):
                pass
        if base is not None:
            line['cpu_baseline'] = base
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if dist_on:
        dist.destroy_process_group()


def run_prefill(args):
    """BASELINE.json config 3: LLaMA-7B int4 g128 prefill, batch 32 x seq 2048 (M = 65536): a step = the quantized linears of one decoder
    layer on the tcgen05 GEMM path (qkv, o, fused gate/up + SwiGLU, down); tokens/s counts the 32 layers' linears only."""
    from gptq_b200 import engine, ops
    dev = torch.device('cuda', int(os.environ.get('LOCAL_RANK', '0')))
    torch.cuda.set_device(dev)
    M, H, I = 65536, 4096, 11008
    gen = torch.Generator(device=dev).manual_seed(0)
    L = {k: engine.random_qlayer(K, N, 4, GROUP, dev, gen) for k, (K, N) in {'qkv': (H, 3 * H), 'o': (H, H), 'gate': (H, I), 'up': (H, I), 'down': (I, H)}.items()}
    t4 = lambda w: (w.qweight, w.scales, w.qzeros, w.g_idx)
    x = torch.randn(M, H, device=dev, generator=gen).half()

    out = {}

    def layer():
        out['qkv'] = ops.matmul248(x, *t4(L['qkv']), 4, None, groupsize=GROUP)
        out['o'] = ops.matmul248(x, *t4(L['o']), 4, None, groupsize=GROUP)
        out['mlp'] = ops.fused_mlp(x, t4(L['gate']), t4(L['up']), 4, GROUP)
        out['down'] = ops.matmul248(out['mlp'], *t4(L['down']), 4, None, groupsize=GROUP)

    steps, warm = args.steps, max(3, min(args.warmup, 5))
    for _ in range(warm):
        layer()
    sampler = ClockSampler(dev.index)
    t = timed(layer, steps, False) / steps
    clocks = sampler.stop()
    if args.dump_outputs:  # the four outputs of the last step on a seeded sample of PREFILL_DUMP_ROWS of the M rows
        rows = torch.randperm(M, generator=torch.Generator().manual_seed(0))[:PREFILL_DUMP_ROWS].sort().values.to(dev)
        dump_outputs(args.dump_outputs, {'rows': rows, **{k: v.index_select(0, rows).float() for k, v in out.items()}})
    flops = 2 * M * (H * 3 * H + H * H + 2 * H * I + I * H)
    _, burst, sustained, src = measured_peaks()
    print(json.dumps({
        'metric': 'prefill tokens/sec LLaMA-7B int4 g128 batch=32 seq=2048 (quantized linears, tcgen05 GEMM path)', 'value': M / (t * 32), 'unit': 'tokens/s', 'n_gpus': 1,
        'steps': steps, 'warmup': warm, 'ms_per_step': t * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f16', 'data': 'synthetic',
        'config': {'workload': 'LLaMA-7B int4 g128 prefill batch 32 x seq 2048 (M=65536): the 4 quantized linears of one decoder layer per step; tokens/s = M / (32 x step)',
                   'l2': 'activations 0.5-1.4 GB per operand (>> 126 MB L2)'},
        'gpu_launches': 4 * steps, 'clocks': clocks,
        'roofline': {'bound': 'tensor', 'kernel': 'qgemm_tcgen05_kernel', 'achieved': flops / t / 1e12, 'peak': sustained, 'unit': 'TFLOP/s', 'frac': flops / t / 1e12 / sustained,
                     'frac_of_burst': flops / t / 1e12 / burst, 'peak_source': src + ' (sustained cuBLAS bf16)', 'traffic': None},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default='7b', choices=sorted(CONFIGS) + ['prefill'])
    ap.add_argument('--dump-outputs', metavar='DIR', help='write what the timed path computed in its last step as DIR/<name>.npy (float32 / float64)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        run_reference(args)
    elif args.config == 'prefill':
        run_prefill(args)
    else:
        run_decode(args)


if __name__ == '__main__':
    main()
