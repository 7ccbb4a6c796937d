#!/usr/bin/env python
"""bench.py — mel-frames/sec of the E2-TTS flow-matching hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|3|4|5] [--dropout P] [--dump-outputs DIR]

Workloads (BASELINE.json `configs`):
  2 (default, the metric's config)  E2TTS(dim 512, depth 8, heads 8, 100 mels) forward + loss.backward(), per-GPU batch 16 x 1024 frames
  3  E2TTS(dim 1024, depth 24, heads 16), per-GPU batch 8 x 2048 frames, forward + backward
  4  DurationPredictor(dim 512, depth 8), batch 32 x 1024 frames, forward + backward
  5  E2TTS(dim 1024, depth 24, heads 16).sample(): 32-step midpoint ODE with CFG/APG, batch 8, prompt 256 -> 2048 frames
bf16 tensor-core compute, text conditioning on every step, synthetic data, random-init weights. One process per GPU (torchrun),
weak scaling; gradients of the N replicas are averaged by ONE flat ncclAllReduce per step (e2_tts_pytorch_b200.GradSync) right after
the CUDA-graph replay of forward + backward.
One JSON line is printed by rank 0 (contract: see DESIGN.md §measurement):
  value     whole-job mel-frames/s with the batch already resident in HBM (device-timed, max over ranks)
  e2e       same metric through the public API with HOST (pinned) inputs: H2D of the inputs every step + D2H of the result
  roofline  tcgen05 GEMM kernel family: algorithmic FLOPs of one step's GEMM launches / their device time (the recorded launches replayed
            back to back as one CUDA graph, one CUDA-event pair around the replay) vs the measured bf16 peak (MEASURED_PEAKS.json)
  cpu_baseline  the oracle port (oracle/e2tts_oracle.py = the reference algorithm in fp32 PyTorch) on the host cores, on
                BASELINE cfg1 exactly (B = 2 x 1024 frames, same d512 / depth-8 model): 2 warm-up + 5 timed steps, median
`--impl reference` times that CPU path alone (the reference itself is pure Python + unvendored deps and cannot travel
to the GPU box; see DESIGN.md).
`--dump-outputs DIR` writes, after the timed steps, what the last step of the timed path (the one `value` reports) returned to its
caller, as float32 .npy files: for training steps `loss`, `grad_norms` (the norm of every parameter's gradient, in
model.parameters() order) and `grads_sample` (a fixed seeded sample of 2^23 entries of all gradients concatenated in that order),
for cfg5 the generated mel frames `mel`. Weights (torch and Python's random module), inputs and random draws are seeded, so the files
of two builds compare entry for entry. Two runs of one build agree to the last bits only: some kernels (loss sums, bias and gain
gradients, hyper-connection backward) accumulate with float atomics, whose order varies from run to run; on a B200 (1000 W) two cfg2
runs gave the same loss and gradients within 2e-7 of each other (largest entry 0.024).
"""
import argparse
import json
import os
import random
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark leaves the tree as it found it (it may be read-only)

import torch  # noqa: E402

METRIC = 'mel-frames/sec E2TTS fwd+bwd (d512 depth8 L1024)'
TEXT = ['Hello', 'Goodbye']
CONFIGS = {
    1: dict(kind='train', dim=512, depth=8, heads=8, batch=2, seq=1024, name='cfg1: E2TTS d512 depth8 h8, B2 x N1024 x 100 mel, CPU fwd+bwd (README snippet)'),
    2: dict(kind='train', dim=512, depth=8, heads=8, batch=16, seq=1024, name='cfg2: E2TTS d512 depth8 h8, B16 x N1024 x 100 mel, fwd+bwd'),
    3: dict(kind='train', dim=1024, depth=24, heads=16, batch=8, seq=2048, name='cfg3: E2TTS d1024 depth24 h16, B8 x N2048 per GPU, fwd+bwd'),
    4: dict(kind='duration', dim=512, depth=8, heads=8, batch=32, seq=1024, name='cfg4: DurationPredictor d512 depth8, B32 x N1024, fwd+bwd'),
    5: dict(kind='sample', dim=1024, depth=24, heads=16, batch=8, seq=2048, prompt=256, ode_steps=32,
            name='cfg5: E2TTS d1024 depth24 h16 sample(), 32-step midpoint ODE + CFG/APG, B8, prompt 256 -> 2048 frames'),
}


def forward_flops(cfg, B, text=True, time_cond=True):
    """Algorithmic FLOPs of one transformer forward (SURVEY §8d formulas)."""
    d, L, h, N = cfg['dim'], cfg['depth'], cfg['heads'], cfg['seq']
    dt, I, S, Np = d // 2, h * 64, 4, N + 32
    T = B * Np
    f = 0.0
    for i in range(L):
        f += 6 * T * d * I + 2 * T * I * d + 4 * T * Np * I + 24 * T * d * d + 2 * T * 31 * d + 2 * T * d * h * (1 if i == 0 else 2)
        if i >= L // 2:
            f += 4 * S * T * d * d
        f += 2 * 3 * T * (4 * S * d * (S + 1) + 4 * S * d) * 0.5
        if text:
            f += 6 * T * dt * I + 2 * T * I * dt + 4 * T * Np * I + 24 * T * dt * dt + 2 * T * 31 * dt + 2 * T * dt * h * (1 if i == 0 else 2)
            f += 2 * S * T * (d + dt) * d + (2 * S * T * (d + dt) * dt if i != L - 1 else 0)
            f += 2 * 3 * T * (4 * S * dt * (S + 1) + 4 * S * dt) * 0.5
    f += (4 if time_cond else 2) * B * N * 100 * d + 2 * B * N * d * (100 if time_cond else 0)
    return f


def step_flops(cfg, B):
    """Algorithmic FLOPs of the timed unit of work of `cfg` on one GPU."""
    if cfg['kind'] == 'sample':   # 62 NFE x (text pass + null pass), SURVEY §8d
        nfe = 2 * (cfg['ode_steps'] - 1)
        return nfe * (forward_flops(cfg, B, text=True) + forward_flops(cfg, B, text=False))
    return 3 * forward_flops(cfg, B, text=True, time_cond=cfg['kind'] == 'train')


# ----------------------------------------------------------------------------------------------------------------------
def cpu_step_fn(cfg, threads):
    """The reference algorithm on the host: fp32 oracle port, forward + backward on cfg1 (README snippet: B = 2, N = 1024)."""
    import e2_tts_pytorch_b200 as pkg
    from oracle import e2tts_oracle as O
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    batch, N = cfg['batch'], cfg['seq']
    model = pkg.E2TTS(transformer=dict(dim=cfg['dim'], depth=cfg['depth'], heads=cfg['heads'], dropout=0.), use_vocos=False)
    sd = {k: v.detach().clone().requires_grad_(v.is_floating_point()) for k, v in model.state_dict().items()}
    ocfg = O.TransformerCfg(dim=cfg['dim'], depth=cfg['depth'], heads=cfg['heads'])
    mel = torch.randn(batch, N, 100)
    text = O.list_str_to_tensor([TEXT[i % 2] for i in range(batch)])
    span = torch.zeros(batch, N, dtype=torch.bool)
    span[:, N // 10: N - N // 10] = True

    def step():
        out = O.e2tts_forward(sd, ocfg, mel, text, x0=torch.randn_like(mel), times=torch.rand(batch), span_mask=span)
        out['loss'].backward()
        for v in sd.values():
            v.grad = None
        return float(out['loss'])

    return step


def run_cpu(steps, warmup, budget_s=150.0, threads=None):
    """BASELINE cfg1 exactly (SURVEY §8d): `warmup` + `steps` steps, median of the timed ones. A slow host stops early at the budget;
    the number of steps actually timed is reported."""
    cfg = CONFIGS[1]
    threads = threads or min(os.cpu_count() or 1, 32)   # more threads than this only oversubscribes the small per-layer GEMMs
    step = cpu_step_fn(cfg, threads)
    times = []
    t_begin = time.time()
    for i in range(warmup + steps):
        t0 = time.time()
        step()
        dt = time.time() - t0
        if i >= warmup:
            times.append(dt)
        if time.time() - t_begin > budget_s:
            if not times:
                times.append(dt)
            break
    times.sort()
    med = times[len(times) // 2]
    return dict(value=cfg['batch'] * cfg['seq'] / med, unit='mel-frames/s', cores=threads, kind='port', timed_steps=len(times),
                sample=f'BASELINE cfg1: {cfg["batch"]} sequences x {cfg["seq"]} frames per step (same d512/depth-8 model and seq_len as cfg2), fp32, '
                       f'{warmup} warm-up + median of {len(times)} timed step(s), {threads} host threads, spread {times[0] * 1e3:.0f}-{times[-1] * 1e3:.0f} ms',
                ms_per_step=med * 1e3)


def run_cpu_bounded(steps, warmup, timeout_s):
    """Run the CPU leg in a child process with a hard wall-clock bound, so that a slow host can never cost the GPU line.
    timeout_s=None: no bound, every one of `steps` is timed."""
    budget = float('inf') if timeout_s is None else max(20.0, timeout_s - 40.0)
    cmd = [sys.executable, os.path.abspath(__file__), '--cpu-worker', '--steps', str(steps), '--warmup', str(warmup),
           '--cpu-budget', str(budget)]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout_s)
        for ln in reversed(out.stdout.strip().splitlines()):
            if ln.startswith('{'):
                return json.loads(ln)
        note = 'cpu worker produced no result: ' + out.stderr.strip()[-200:]
    except subprocess.TimeoutExpired:
        note = f'the fp32 CPU steps of the oracle port did not finish within the {timeout_s:.0f} s bound on this host'
    return dict(value=None, unit='mel-frames/s', cores=min(os.cpu_count() or 1, 32), kind='port', sample=note)


# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, idx):
        self.idx, self.samples, self.stop = idx, [], False
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
            'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
        while not self.stop:
            try:
                out = subprocess.run(['nvidia-smi', f'--id={self.idx}', f'--query-gpu={q}', '--format=csv,noheader,nounits'],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(',')])
            except Exception:
                pass
            time.sleep(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=3)

    def summary(self):
        if not self.samples:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['unavailable'])
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        reasons = set()
        for s in self.samples:
            for name, v in zip(['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'], s[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=int(self.samples[0][1]) if self.samples[0][1].isdigit() else None,
                    reasons=sorted(reasons), samples=len(self.samples))


def gemm_traffic(config):
    """DRAM bytes of the GEMM family per step from the committed ncu capture (profiles/r2_gemm_traffic.json, written by
    tools/gemm_traffic.py from `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum`), or None."""
    try:
        t = json.load(open(os.path.join(ROOT, 'profiles', 'r2_gemm_traffic.json')))
        return t.get(f'cfg{config}')
    except Exception:
        return None


def run_gpu(args):
    import torch.distributed as dist
    import e2_tts_pytorch_b200 as pkg
    from e2_tts_pytorch_b200 import lib, ops
    cfg = CONFIGS[args.config]
    kind = cfg['kind']
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    torch.manual_seed(0)
    random.seed(0)      # the hyper-connections pick their initial stream with python's randrange (SURVEY A.5)
    tkw = dict(dim=cfg['dim'], depth=cfg['depth'], heads=cfg['heads'], dropout=args.dropout)
    B, N = cfg['batch'], cfg['seq']
    if kind == 'duration':
        model = pkg.DurationPredictor(transformer=tkw).to(dev)
    else:
        model = pkg.E2TTS(transformer=tkw, use_vocos=False).to(dev)
        model.cond_drop_prob = 0.0  # text conditioning on every step: the expensive branch, identical graph on every rank (SURVEY §8d)
    model.train()
    pkg.broadcast_module(model)      # identical replicas, as DDP's constructor guarantees (part of the init is rank dependent)
    sync = pkg.GradSync(list(model.parameters())) if (world > 1 and kind != 'sample') else None   # eager N > 1 step: flat all-reduce too
    torch.manual_seed(rank)
    n_in = cfg['prompt'] if kind == 'sample' else N
    host_mel = torch.randn(B, n_in, 100).pin_memory()
    dev_mel = host_mel.to(dev)
    text = [TEXT[i % 2] for i in range(B)]
    text_dev = pkg.list_str_to_tensor(text).to(dev)
    d2h_bytes = 4
    last = {}     # --dump-outputs: what a recorded eager step returned (the loss detached: see GraphedTrainStep on eager outputs)

    if kind == 'sample':
        model.eval()
        d2h_bytes = B * N * 100 * 4

        def step(mel, readback, record=False):
            out = model.sample(mel, text=text_dev, duration=N, steps=cfg['ode_steps'], cfg_strength=1.0, return_raw_output=True)
            if record:
                last['out'] = out
            return out.cpu() if readback else None
    else:
        def step(mel, readback, record=False):
            loss = model(mel, text=text_dev) if kind == 'duration' else model(mel, text=text_dev).loss
            loss.backward()
            if sync is not None:
                sync()
            if record:
                last['out'], last['grads'] = loss.detach(), [p.grad for p in model.parameters()]
            for p in model.parameters():
                p.grad = None
            return loss.item() if readback else None

    def outputs(out, grads=None):
        """Host copies of one step's results for --dump-outputs (module docstring)."""
        if grads is None:
            return {'mel': out.float().cpu().numpy()}
        params = list(model.parameters())
        flat = torch.cat([(g if g is not None else torch.zeros_like(p)).detach().flatten().float() for p, g in zip(params, grads)])
        idx = torch.randint(flat.numel(), (min(flat.numel(), 1 << 23),), generator=torch.Generator().manual_seed(0))
        return {'loss': out.detach().float().reshape(1).cpu().numpy(),
                'grad_norms': torch.stack([g.float().norm() if g is not None else torch.zeros((), device=dev) for g in grads]).cpu().numpy(),
                'grads_sample': flat[idx.to(dev)].cpu().numpy()}

    def timed(fn, steps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.barrier()
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) / steps

    steps = args.steps
    warm = max(args.warmup, 3) if kind != 'sample' else 1   # one cfg5 step = 124 transformer forwards
    for _ in range(warm):
        step(dev_mel, False)
    # -- time of the tcgen05 GEMM family inside one real step (roofline numerator / denominator): every ops.gemm call of ONE step is
    #    recorded with its live operands, then the same calls are captured into one CUDA graph and replayed — the kernels run back to
    #    back exactly as launched in the step, and the whole list is bracketed by ONE event pair. (Bracketing each launch of an eager
    #    step with its own event pair also brackets the host's launch latency whenever the GPU waits for the host: h + max(kernel, h'),
    #    which inflated the round-1/2 figures by up to 70 % on slow hosts.)
    prof = dict(flops=0.0, calls=[])
    orig_gemm = ops.gemm

    def gemm_recorded(A, Bm, M, Nn, K, **kw):
        out = orig_gemm(A, Bm, M, Nn, K, **kw)
        kw2 = dict(kw)
        kw2['out'] = out          # the replay overwrites this step's outputs in place (nothing reads them afterwards)
        prof['calls'].append((A, Bm, M, Nn, K, kw2))
        prof['flops'] += 2.0 * M * Nn * K
        return out

    def replay_gemms():
        calls = prof['calls']
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for c in calls[:8]:      # warm the descriptor cache / lazy init off the capture
                orig_gemm(c[0], c[1], c[2], c[3], c[4], **c[5])
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for c in calls:
                orig_gemm(c[0], c[1], c[2], c[3], c[4], **c[5])
        times = []
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        del g
        times.sort()
        return times[len(times) // 2]

    step_mode, graph_note, eager_ms = 'eager', None, None
    with ClockSampler(local) as clk:
        n0 = lib.launch_count()
        done = [0]

        def dev_step():     # --dump-outputs: keep the results of the last timed step only, so that no earlier step's stay allocated
            done[0] += 1
            step(dev_mel, False, record=args.dump_outputs is not None and done[0] == steps)

        ms_dev = timed(dev_step, steps)
        launches = (lib.launch_count() - n0) // steps
        dumped = outputs(last['out'], last.get('grads')) if args.dump_outputs else None
        last.clear()
        ms_e2e = timed(lambda: step(host_mel.to(dev, non_blocking=True), True), steps)
        ops.gemm = gemm_recorded
        nprof = 1
        if kind == 'sample':    # profile ONE function evaluation (text pass + null pass) instead of all 62
            with torch.no_grad():
                x = torch.randn(B, N, 100, device=dev)
                model.cfg_transformer_with_pred_head(x, torch.zeros_like(x), times=torch.tensor(0.5, device=dev), text=text_dev,
                                                     mask=torch.ones(B, N, dtype=torch.bool, device=dev), cfg_strength=1.0)
        else:
            step(dev_mel, False)
        torch.cuda.synchronize()
        ops.gemm = orig_gemm
        gemm_ms = replay_gemms()
        n_gemm = len(prof['calls'])
        prof['calls'] = None      # release the step's operands before the graphed step allocates its own pool
        torch.cuda.empty_cache()
        # -- the same train step through pkg.GraphedTrainStep (forward + backward captured in one CUDA graph, then — N > 1 — ONE flat
        #    all-reduce): identical kernels and work, no per-launch host cost. Falls back to the eager numbers if capture fails.
        if kind in ('train', 'duration') and not args.no_graph:
            try:
                eager_loss = step(dev_mel, True)
                torch.cuda.empty_cache()      # the eager pool and the graph's private pool each hold a full set of activations
                graphed = pkg.GraphedTrainStep(model, dev_mel, text=text_dev)
                g_loss = float(graphed().item())
                if not (g_loss == g_loss and 0.5 * eager_loss <= g_loss <= 2.0 * eager_loss):
                    raise RuntimeError(f'graphed loss {g_loss} vs eager {eager_loss}')
                for _ in range(3):
                    graphed()
                ms_g = timed(lambda: graphed(), steps)
                dumped_g = outputs(graphed.out.loss, [p.grad for p in model.parameters()]) if args.dump_outputs else None
                ms_g_e2e = timed(lambda: graphed(host_mel).item(), steps)
                ok = torch.tensor([1.0 if ms_g < ms_dev else 0.0], device=dev)
                if world > 1:
                    dist.all_reduce(ok, op=dist.ReduceOp.MIN)   # (both times are max-over-ranks already; keep the ranks in lockstep)
                if float(ok) > 0:
                    eager_ms, step_mode = ms_dev, 'cuda_graph'
                    ms_dev, ms_e2e, launches, dumped = ms_g, ms_g_e2e, graphed.launches_per_step, dumped_g
                else:
                    graph_note = f'captured but not faster ({ms_g:.2f} ms)'
            except Exception as e:  # noqa: BLE001 - any capture problem: keep the eager measurement
                graph_note = f'unavailable: {type(e).__name__}: {str(e)[:160]}'
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak_tf = peaks.get('bf16_tflops_sustained', 1400.0)
    achieved_tf = prof['flops'] / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    frames = world * B * N
    fl = step_flops(cfg, B)
    what = {'train': 'E2TTS forward + loss.backward()', 'duration': 'DurationPredictor forward + loss.backward()',
            'sample': 'E2TTS.sample(): 31 midpoint steps = 62 function evaluations x (text pass + null pass) + CFG/APG'}[kind]
    line = {
        'metric': METRIC if args.config == 2 else f'mel-frames/sec, {cfg["name"]}', 'value': frames / (ms_dev * 1e-3), 'unit': 'mel-frames/s', 'n_gpus': world,
        'steps': steps, 'warmup': warm, 'ms_per_step': ms_dev, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16',
        'data': 'synthetic',
        'config': {'workload': cfg['name'], 'per_gpu_batch': B, 'seq_len': N, 'global_batch': world * B, 'parallelism': f'dp{world}',
                   'dropout': args.dropout if kind != 'sample' else 0.0, 'text_cond': 'on every step', 'weights': 'random init',
                   'optimizer_step': 'not part of the metric',
                   'l2': 'per-step working set (GBs of activations) >> 126 MB L2, no flush needed',
                   'grad_exchange': ('one flat fp32 ncclAllReduce per step after backward (e2_tts_pytorch_b200.GradSync)' if world > 1 and kind != 'sample' else 'none'),
                   'step': (what + ' replayed through e2_tts_pytorch_b200.GraphedTrainStep (one CUDA graph, same kernels)'
                            if step_mode == 'cuda_graph' else what + ', eager launches'),
                   'streams': ('text sub-blocks of layer i+1 overlap the audio sub-blocks of layer i on a second CUDA stream (fork/join inside the step); '
                               'the roofline pass replays the step\'s GEMM launches back to back as one CUDA graph') if pkg.modules.TWO_STREAM else 'one stream',
                   **({'eager_ms_per_step': eager_ms} if eager_ms is not None else {}), **({'cuda_graph': graph_note} if graph_note else {})},
        'e2e': {'value': frames / (ms_e2e * 1e-3), 'unit': 'mel-frames/s', 'ms_per_step': ms_e2e, 'h2d_bytes_per_step': host_mel.numel() * 4,
                'd2h_bytes_per_step': d2h_bytes},
        'gpu_launches': int(launches),
        'clocks': clk.summary(),
        'roofline': {'kernel': 'gemm_tcgen05_kernel (all GEMMs of the step: fwd, dX, dW)' if kind != 'sample' else 'gemm_tcgen05_kernel (all GEMMs of one function evaluation)',
                     'bound': 'tensor', 'achieved': achieved_tf, 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': achieved_tf / peak_tf if peak_tf else None,
                     'traffic': gemm_traffic(args.config),
                     'launches_per_step': n_gemm // max(nprof, 1), 'ms_per_step': gemm_ms / max(nprof, 1),
                     'peak_source': 'MEASURED_PEAKS.json bf16_tflops_sustained' if peaks else 'fallback 1.4 PF/s sustained',
                     'step_flops': fl, 'step_tensor_frac': fl / (ms_dev * 1e-3) / 1e12 / peak_tf},
    }
    if world == 1 and not args.no_cpu:
        line['cpu_baseline'] = run_cpu_bounded(steps=5, warmup=2, timeout_s=170.0)
    if dumped is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + '.npy'), arr)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', type=int, default=2, choices=[2, 3, 4, 5])
    ap.add_argument('--dropout', type=float, default=0.1)
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-graph', action='store_true', help='time the eager step only (skip the CUDA-graph replay of the same step)')
    ap.add_argument('--cpu-worker', action='store_true', help=argparse.SUPPRESS)
    ap.add_argument('--cpu-budget', type=float, default=150.0, help=argparse.SUPPRESS)
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the outputs of the last timed step to DIR/<name>.npy (module docstring)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.cpu_worker:
        print(json.dumps(run_cpu(steps=args.steps, warmup=args.warmup, budget_s=args.cpu_budget)), flush=True)
        return
    if args.impl == 'reference':
        if int(os.environ.get('RANK', '0')) != 0:
            return
        cfg = CONFIGS[args.config]
        r = run_cpu_bounded(steps=args.steps, warmup=min(max(args.warmup, 1), 2), timeout_s=None)
        print(json.dumps({
            'impl': 'reference', 'metric': METRIC, 'value': r['value'], 'unit': 'mel-frames/s', 'n_gpus': args.gpus, 'steps': r.get('timed_steps', 0),
            'warmup': min(max(args.warmup, 1), 2), 'ms_per_step': r.get('ms_per_step'), 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': cfg['name'], 'requested_steps': args.steps, 'requested_warmup': args.warmup,
                       'note': 'reference algorithm on the host CPU cores (oracle port), timed on BASELINE cfg1 = 2 of the 16 sequences of cfg2 per step '
                               '(same model, same seq_len)'},
            'cpu_baseline': {k: r.get(k) for k in ('value', 'unit', 'cores', 'kind', 'sample')},
            'e2e': {'value': r['value'], 'unit': 'mel-frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}))
        return
    run_gpu(args)


if __name__ == '__main__':
    main()
