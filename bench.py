#!/usr/bin/env python
"""Benchmark of the text->mel hot path (BASELINE.json configs[1]: LJSpeech ForwardTransformer 6+6 layers, d=256,
inference, batch 64 per GPU, 128 phonemes -> 1000 mel frames, durations/pitch forced).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision bf16x3|bf16] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  `value` = mel frames/s with inputs resident in HBM, CUDA-event timed, max over
ranks; `e2e` = the same metric through ForwardTransformer.predict() with host inputs (pinned H2D) and the mel copied
back to the host every step; `roofline` = decoder conv GEMM launches (the dominant kernel) timed with CUDA events in
the same run; `cpu_baseline` = the CPU oracle (torch fp32, all host cores) on a bounded sample of the same workload.
`--impl reference` times only that CPU path (the reference is TF2 and cannot be installed offline; the oracle is its
literal restatement).  `--dump-outputs DIR` writes what the last timed step returned (rank 0) as DIR/<name>.npy; inputs
and weights are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

WORKLOAD = 'C2: LJ256 ForwardTransformer inference, B=64/GPU, 128 phonemes -> 1000 mel frames (forced durations+pitch)'
CFG_NAME = 'LJ256'
B, TP, TM = 64, 128, 1000
METRIC, UNIT = 'mel_frames_per_sec_fwd', 'frames/s'
DUMP_LIMIT = 64 << 20


def _traffic(key):
    """DRAM bytes per launch of the roofline kernel from the committed ncu --set full capture (profiles/traffic.json,
    written by profiles/summarize.py); None when no capture is committed."""
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'profiles', 'traffic.json')) as f:
            return json.load(f).get(key)
    except Exception:
        return None


def _peaks():
    f = ROOT / 'MEASURED_PEAKS.json'
    if f.exists():
        d = json.loads(f.read_text())
        return float(d.get('bf16_tflops_sustained', d.get('bf16_tflops', 1590.0))), float(d.get('hbm_gbs', 6650.0)), 'measured (MEASURED_PEAKS.json, sustained bf16)'
    return 1590.0, 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index
        q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
            'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={index}', f'--query-gpu={q}', '--format=csv,noheader,nounits', '-lms', '20'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            parts = [x.strip() for x in r.split(',')]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def _pick_threads() -> int:
    """Host threads for the CPU arm: the count that actually runs fastest.  A container may see far more cores than its
    CPU quota allows (the pool's boxes report 128 but 128 torch threads ran ~150x slower than 8), so time a small GEMM
    at a few thread counts and keep the best; the JSON line states what was used."""
    cores = os.cpu_count() or 1
    try:
        cores = min(cores, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q, per = open('/sys/fs/cgroup/cpu.max').read().split()
        if q != 'max':
            cores = max(1, min(cores, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    cands = sorted({c for c in (4, 8, 16, 32, 64, cores) if c <= cores} | {cores})
    a = torch.randn(1024, 1024)
    b = torch.randn(1024, 1024)
    best, best_t = cands[0], float('inf')
    for c in cands:
        torch.set_num_threads(c)
        (a @ b)
        t0 = time.perf_counter()
        for _ in range(6):
            (a @ b)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def _inputs(seed):
    from oracle import forward_oracle as fo
    return fo.make_inputs('full', B, TP, TM, seed=seed)


def _tf_reference_available() -> bool:
    """SURVEY 8c: prefer the real TF2 reference when it can be imported on this box (it cannot in this image: there is
    no tensorflow wheel); tests/golden/make_golden_tf.py is the script that uses it when it exists."""
    try:
        import importlib.util
        return importlib.util.find_spec('tensorflow') is not None and (ROOT / 'baseline' / '_ref').exists()
    except Exception:
        return False


def dump_outputs(dirname, out):
    """The arrays of one step's result dict as DIR/<name>.npy (nested dicts as <name>.<key>.npy; None entries, such as
    attention maps that were not requested, carry no array): floating-point arrays in float32, integer and boolean ones in
    float64 (exact)."""
    import numpy as np
    arrays = {}
    for k, v in out.items():
        for sub, t in (v.items() if isinstance(v, dict) else [(None, v)]):
            if t is None:
                continue
            a = t.detach().cpu()
            arrays[k if sub is None else f'{k}.{sub}'] = (a.float() if a.is_floating_point() else a.double()).numpy()
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f'--dump-outputs: {total / 2**20:.0f} MB of outputs exceed the {DUMP_LIMIT >> 20} MB limit')
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + '.npy'), a)


def _config_dict(world):
    return {'workload': WORKLOAD, 'model': CFG_NAME, 'global_batch': B * world, 'seq_len': TM}


def cpu_forward_rate(budget_s, min_passes=1, max_passes=8):
    """The CPU path on the WHOLE 64-row batch of the workload (same rows, same shapes as the GPU step): one untimed pass
    (builds the positional-encoding cache), then whole-batch passes until `budget_s` is used.  Returns (frames/s, passes,
    seconds, cores, last output)."""
    from oracle import forward_oracle as fo
    cores = _pick_threads()
    cfg = fo.CONFIGS[CFG_NAME]
    p = fo.init_params(cfg, seed=7)
    tok, dur, pit = _inputs(200)
    cache = {}
    with torch.no_grad():
        fo.forward_transformer_call(p, cfg, tok[:1], dur[:1, :, None], pit[:1, :, None], _cache=cache)
        t0 = time.perf_counter()
        n = 0
        ref = None
        while n < min_passes or (time.perf_counter() - t0 < budget_s and n < max_passes):
            ref = fo.forward_transformer_call(p, cfg, tok, dur[:, :, None], pit[:, :, None], _cache=cache)
            n += 1
        dt = time.perf_counter() - t0
    return B * TM * n / dt, n, dt, cores, ref


def cpu_reference_line(args, rank, world):
    """--impl reference: the CPU path (oracle restatement of the TF2 graph) on the host cores.  Every step is the whole
    64-row batch of the GPU arm's step (same config), and exactly --steps of them are timed; warm-up passes beyond the
    first are capped at 15 % of a 240 s budget."""
    from oracle import forward_oracle as fo
    if rank != 0:
        return None
    cores = _pick_threads()
    cfg = fo.CONFIGS[CFG_NAME]
    p = fo.init_params(cfg, seed=7)
    tok, dur, pit = _inputs(200)
    cache = {}

    def run():
        with torch.no_grad():
            return fo.forward_transformer_call(p, cfg, tok, dur[:, :, None], pit[:, :, None], _cache=cache)

    with torch.no_grad():
        fo.forward_transformer_call(p, cfg, tok[:1], dur[:1, :, None], pit[:1, :, None], _cache=cache)
    t0 = time.perf_counter()
    run()                                   # first whole step: also the estimate for the budget
    t1 = time.perf_counter() - t0
    budget = 240.0
    warm = max(0, min(args.warmup - 1, int(0.15 * budget / t1)))
    steps = args.steps
    for _ in range(warm):
        run()
    t0 = time.perf_counter()
    for _ in range(steps):
        run()
    dt = time.perf_counter() - t0
    val = B * TM * steps / dt
    sample = (f'{steps} whole steps of {B} rows x {TM} frames (a whole step takes {t1:.1f} s on this host), '
              f'torch-CPU fp32 oracle, {cores} threads')
    return {'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': steps,
            'warmup': warm + 1, 'ms_per_step': dt / steps * 1e3, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': _config_dict(1),
            'cpu_baseline': {'value': val, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample},
            'e2e': {'value': val, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'tf_reference_available': _tf_reference_available(),
            'note': 'TF2 reference cannot be installed offline (no tensorflow wheel); oracle/ is its CPU restatement'}


def hbm_bench(args, rank, world, dev, cfg):
    """The two HBM-bound rows of the scope table, each timed alone with CUDA events and an L2 flush between iterations:
    'stft'  : BASELINE configs[3], 256 clips x 220500 samples -> (256, 862, 80) log-mel, algorithmic bytes = audio in + mel out;
    'expand': the length regulator of C2 (durations -> int -> index map -> gather), algorithmic bytes = x in + expanded out."""
    import numpy as np
    import torch.distributed as dist
    from oracle import audio_oracle as ao
    from oracle import forward_oracle as fo
    from transformertts_b200 import lib
    from transformertts_b200.data.audio import Audio
    _, peak_hbm, _ = _peaks()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2
    steps = args.steps
    times = []
    if args.mode == 'stft':
        n_clips, n_samples = 256, 220500
        audio = Audio(sampling_rate=22050, n_fft=1024, mel_channels=80, hop_length=256, win_length=1024, f_min=0, f_max=8000,
                      normalizer='MelGAN', device=str(dev))
        clips = ao.make_clips(4, n_samples, seed=400 + rank)
        wav = torch.from_numpy(np.tile(clips, (n_clips // 4, 1))).to(dev)
        wav += 0.01 * torch.randn_like(wav)
        fn = lambda: audio.mel_spectrogram_device(wav)
        out = fn()
        alg_bytes = wav.numel() * 4 + out.numel() * 4
        units, unit_name, metric = n_clips, 'clips/s', 'stft_mel_clips_per_sec'
        workload = 'C4: STFT->log-mel, 256 clips x 10 s @ 22.05 kHz, n_fft 1024 hop 256, 80 mels'
        ref = ao.mel_spectrogram(wav[0].cpu().numpy())
        err = float(np.abs(out[0].cpu().numpy() - ref).max())
        t0 = time.perf_counter()
        for i in range(4):
            ao.mel_spectrogram(wav[i].cpu().numpy())
        cpu = {'value': 4 / (time.perf_counter() - t0), 'unit': unit_name, 'cores': 1, 'kind': 'port',
               'sample': '4 clips, numpy restatement of librosa.stft + mel filterbank (single thread)', 'max_abs_err_gpu_vs_cpu': err}
    else:
        tok, dur, pit = fo.make_inputs('full', B, TP, TM, seed=200 + rank)
        d = cfg['encoder_model_dimension']
        x = torch.randn(B, TP, d, device=dev)
        dur_f = dur.to(dev).float()
        dur_i = torch.empty((B, TP), dtype=torch.int32, device=dev)
        lens = torch.empty((B,), dtype=torch.int32, device=dev)
        idx = torch.empty((B, TM), dtype=torch.int32, device=dev)
        out = torch.empty((B, TM, d), dtype=torch.float32, device=dev)

        def fn():
            lib.durations_to_int(dur_f, 1.0, None, None, dur_i, lens)
            lib.expand_indices(dur_i, TM, idx)
            lib.length_regulate_fwd(x, idx, out)
            return out
        fn()
        alg_bytes = x.numel() * 4 + dur_f.numel() * 4 + out.numel() * 4
        units, unit_name, metric = B * TM, 'frames/s', 'length_regulator_frames_per_sec'
        workload = 'C2-LR: length regulator alone, B=64, 128 phonemes -> 1000 frames, d=256 fp32'
        want = fo.expand(x.cpu(), dur[..., None].float())
        cpu = {'value': None, 'unit': unit_name, 'cores': 0, 'kind': 'port', 'sample': 'parity only',
               'bit_exact_vs_oracle': bool(torch.equal(out.cpu(), want))}
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    for _ in range(steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    t = torch.tensor([sum(times) / len(times)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    if rank == 0:
        gbs = alg_bytes / (ms * 1e-3) / 1e9
        print(json.dumps({'metric': metric, 'value': units * world / (ms * 1e-3), 'unit': unit_name, 'n_gpus': world, 'steps': steps, 'warmup': 3,
                          'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
                          'config': {'workload': workload, 'l2': '256 MB buffer rewritten between timed iterations (L2 flush)'},
                          'roofline': {'bound': 'hbm', 'achieved': gbs, 'peak': peak_hbm, 'unit': 'GB/s', 'frac': gbs / peak_hbm, 'traffic': None,
                                       'algorithmic_bytes_per_launch': alg_bytes},
                          'cpu_baseline': cpu}), flush=True)


def train_bench(args, rank, world, dev, cfg, params, steps=None):
    """BASELINE configs[2]: LJ256 training step (fwd + bwd + Adam, dropout 0.1, bf16 tensor-core products), batch 32 per
    GPU, 128 phonemes -> 1000 frames, gradients all-reduced with NCCL (sum, scaled 1/N inside the Adam kernel).
    Returns the record (rank 0) or None; the caller prints it (alone for --mode train, as the `train` key of the default
    line otherwise)."""
    import torch.distributed as dist
    from oracle import forward_oracle as fo
    from transformertts_b200 import lib
    from transformertts_b200.model.models import ForwardTransformer
    from transformertts_b200.model.training import Adam
    Bt = 32
    steps = steps or args.steps
    warm = max(args.warmup, 3)
    model = ForwardTransformer(**cfg, device=str(dev), train_dropout=True, train_graphs=not args.no_graphs)
    model.set_weights(params)
    model._compile(Adam(1e-4))
    eng = model._get_engine()
    eng.rank = rank
    tok, dur, pit = fo.make_inputs('full', Bt, TP, TM, seed=300 + rank)
    mel = fo.make_mel_targets(dur, cfg['mel_channels'], seed=400 + rank)
    tok_d, dur_d, pit_d, mel_d = tok.to(dev), dur.to(dev), pit.to(dev), mel.to(dev)

    def timed(dp):
        """K device-resident steps, CUDA events, max over ranks -> ms per step."""
        for _ in range(warm):
            model.train_step(tok_d, mel_d, dur_d, pit_d, data_parallel=dp)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        lib.reset_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            model.train_step(tok_d, mel_d, dur_d, pit_d, data_parallel=dp)
        e1.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        n_launch = lib.launch_count()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / steps, n_launch

    sampler = ClockSampler(dev.index or 0) if rank == 0 else None
    ms_step, launches = timed(world > 1)
    clocks = sampler.stop() if sampler else None
    # the same step WITHOUT the gradient all-reduce: the difference is the communication time the overlap did not hide
    ms_local = timed(False)[0] if world > 1 else ms_step
    # end to end through train_step() with HOST batches: the next batch's pinned H2D copies run on a side stream under the
    # current step, the loss comes back to pinned host memory every step (read one step late, so no per-step host sync)
    host = [t_.pin_memory() for t_ in (tok, mel, dur, pit)]
    h2d_bytes = int(sum(t_.numel() * t_.element_size() for t_ in host))
    side = torch.cuda.Stream(device=dev)
    loss_h = [torch.zeros(1).pin_memory() for _ in range(2)]

    def stage():
        with torch.cuda.stream(side):
            b = [t_.to(dev, non_blocking=True) for t_ in host]
            ev = torch.cuda.Event()
            ev.record(side)
        return b, ev

    def e2e_loop(n):
        nxt = stage()
        last = None
        for i in range(n):
            (tk, ml, du, pi), ev = nxt
            torch.cuda.current_stream().wait_event(ev)
            for t_ in (tk, ml, du, pi):
                t_.record_stream(torch.cuda.current_stream())
            if i + 1 < n:
                nxt = stage()
            o = model.train_step(tk, ml, du, pi, data_parallel=world > 1)
            loss_h[i & 1].copy_(o['loss'].reshape(1), non_blocking=True)
            last = i & 1
        torch.cuda.synchronize()
        return float(loss_h[last])

    e2e_loop(warm)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    loss_val = e2e_loop(steps)
    if world > 1:
        dist.barrier()
    dt = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    peak_tf, _, peak_src = _peaks()
    flops = 3.0 * fo.forward_flops(cfg, [TP] * Bt, [TM] * Bt)
    if rank != 0:
        return None
    sps = 1e3 / ms_step
    return {'metric': 'train_steps_per_sec', 'value': sps, 'unit': 'steps/s', 'n_gpus': world, 'steps': steps,
            'warmup': warm, 'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
            'config': {'workload': 'C3: LJ256 training step (fwd+bwd+Adam, dropout 0.1, MAE losses [1,1,3]), 32 rows/GPU, 128 phonemes -> 1000 frames',
                       'model': CFG_NAME, 'global_batch': Bt * world, 'seq_len': TM,
                       'parallelism': f'dp{world} (NCCL all-reduce of the flat fp32 gradient in 2 buckets, decoder bucket overlapped with the encoder backward)',
                       'launch': 'eager' if args.no_graphs else 'CUDA graphs (forward + decoder backward | encoder backward), Adam and the NCCL all-reduces launched eagerly',
                       'l2': 'per-step working set exceeds the 126 MB L2'},
            'frames_per_sec': sps * Bt * TM * world,
            'ms_per_step_without_allreduce': ms_local, 'nccl_exposed_ms': max(0.0, ms_step - ms_local) if world > 1 else 0.0,
            'allreduce_bytes_per_step': int(eng.flat_g.numel() * 4) if world > 1 else 0,
            'e2e': {'value': steps / float(dt.item()), 'unit': 'steps/s', 'h2d_bytes_per_step': h2d_bytes, 'd2h_bytes_per_step': 4},
            'gpu_launches': int(launches), 'clocks': clocks, 'loss': loss_val,
            'roofline': {'bound': 'tensor', 'achieved': flops / (ms_step * 1e-3) / 1e12, 'peak': peak_tf, 'unit': 'TFLOP/s',
                         'frac': flops / (ms_step * 1e-3) / 1e12 / peak_tf, 'traffic': None, 'peak_source': peak_src,
                         'kernel': 'whole step (3x forward algorithmic FLOPs per GPU)'},
            'cpu_baseline': None}


def aligner_flops(cfg, B, Tp, T, r=1):
    """Algorithmic FLOPs of one teacher-forced Aligner forward (2 per multiply-add; the look-ahead mask halves the
    decoder self-attention products)."""
    de, dd, mel = cfg['encoder_model_dimension'], cfg['decoder_model_dimension'], cfg['mel_channels']
    fe, fd = cfg['encoder_feed_forward_dimension'], cfg['decoder_feed_forward_dimension']
    enc = len(cfg['encoder_num_heads']) * (2 * de * 3 * de + 2 * 2 * de * de + 4 * de * fe + 4 * Tp * de)
    dec_layers = len(cfg['decoder_num_heads'])
    dec = dec_layers * (2 * dd * 3 * dd + 4 * dd * dd + 2 * T * dd + 2 * dd * dd + 4 * dd * dd + 4 * Tp * dd + 4 * dd * fd)
    kv = dec_layers * 2 * de * 2 * dd
    pre = 2 * (mel * cfg['decoder_prenet_dimension'] + cfg['decoder_prenet_dimension'] * dd)
    post = 2 * dd * r * mel + r * 2 * mel * (mel + 3)
    return float(B) * (Tp * (enc + kv) + T * (dec + pre + post))


def aligner_bench(args, rank, world, dev):
    """BASELINE configs[4] (C5): Aligner teacher-forced step, batch 16, 800 mel frames, r = 1, aligner_settings as shipped.
    Built so far: forward + validation losses (mel MAE, scaled stop CE, diagonal attention loss); no backward."""
    import torch.distributed as dist
    from oracle import aligner_oracle as alo
    from transformertts_b200 import lib
    from transformertts_b200.model.aligner import Aligner
    B, Tp, T = 16, 130, 800
    cfg = alo.ALIGNER_CONFIGS['A5']
    params = alo.init_aligner_params(cfg, seed=7)
    model = Aligner.from_config(dict(cfg, device=str(dev), cuda_graphs=not args.no_graphs), max_r=cfg['max_r'])
    model.set_weights(params)
    model.set_constants(reduction_factor=1, force_decoder_diagonal=True)
    tok, mel, stop = alo.make_aligner_inputs(cfg, B, Tp, T + 1, seed=500 + rank, ragged=False)
    tok_d, mel_d, stop_d = tok.to(dev), mel.to(dev), stop.to(dev)

    def step():
        return model._val_step(tok_d, mel_d, stop_d)

    for _ in range(max(args.warmup, 3)):
        out = step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(dev.index or 0) if rank == 0 else None
    lib.reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = step()
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches = lib.launch_count()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    clocks = sampler.stop() if sampler else None
    tok_h, mel_h, stop_h = tok.pin_memory(), mel.pin_memory(), stop.pin_memory()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        o = model._val_step(tok_h.to(dev, non_blocking=True), mel_h.to(dev, non_blocking=True), stop_h.to(dev, non_blocking=True))
        loss_val = float(o['loss'])
    torch.cuda.synchronize()
    dt = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    # ---- the training step (models.py:212-216): forward with dropout 0.1 in single-pass bf16 + backward + Adam
    from transformertts_b200.model.training import Adam
    tmodel = Aligner.from_config(dict(cfg, device=str(dev), train_dropout=True, train_graphs=not args.no_graphs), max_r=cfg['max_r'])
    tmodel.set_weights(params)
    tmodel._compile(cfg['stop_loss_scaling'], Adam(1e-4))
    tmodel.set_constants(reduction_factor=1, force_decoder_diagonal=True)
    tmodel._get_engine().rank = rank
    for _ in range(max(args.warmup, 3)):
        to = tmodel.train_step(tok_d, mel_d, stop_d)
    torch.cuda.synchronize()
    lib.reset_launch_count()
    t0e, t1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0e.record()
    for _ in range(args.steps):
        to = tmodel.train_step(tok_d, mel_d, stop_d)
    t1e.record()
    torch.cuda.synchronize()
    train_launches = lib.launch_count()
    tt = torch.tensor([t0e.elapsed_time(t1e)], device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    train_ms = float(tt.item()) / args.steps
    train_loss = float(to['loss'])
    peak_tf, _, peak_src = _peaks()
    flops = aligner_flops(cfg, B, Tp, T)
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        nthr = _pick_threads()
        torch.set_num_threads(nthr)
        rows = 2
        with torch.no_grad():
            alo.gta_forward(params, cfg, tok[:rows], mel[:rows], stop[:rows], r=1, force_decoder_diagonal=True)
            c0 = time.perf_counter()
            reps = 0
            while time.perf_counter() - c0 < 10.0:
                alo.gta_forward(params, cfg, tok[:rows], mel[:rows], stop[:rows], r=1, force_decoder_diagonal=True)
                reps += 1
            cdt = time.perf_counter() - c0
        cpu = {'value': reps * rows / B / cdt, 'unit': 'steps/s', 'cores': nthr, 'kind': 'port',
               'sample': f'{reps} oracle passes over {rows} of the 16 rows in {cdt:.1f} s (torch CPU fp32), scaled to 16-row steps'}
    if rank == 0:
        sps = args.steps / (ms * 1e-3)
        line = {'metric': 'aligner_teacher_forced_steps_per_sec', 'value': sps * world, 'unit': 'steps/s', 'n_gpus': world,
                'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': ms / args.steps, 'higher_is_better': True,
                'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16x3 GEMMs + fp16 attention, fp32 accumulate', 'data': 'synthetic',
                'config': {'workload': 'C5: Aligner teacher-forced forward + validation losses (mel MAE, scaled stop CE, diagonal loss), '
                                       '16 rows/GPU, 130 tokens, 800 decoder frames, r=1, aligner_settings as shipped; train_step = the full training step',
                           'model': 'A5', 'global_batch': B * world, 'seq_len': T, 'parallelism': f'independent replicas x{world}',
                           'l2': 'working set (~0.6 GB of activations + attention maps) exceeds the 126 MB L2'},
                'frames_per_sec': sps * B * T * world,
                'e2e': {'value': args.steps / float(dt.item()) * world, 'unit': 'steps/s',
                        'h2d_bytes_per_step': int(tok.numel() * 4 + mel.numel() * 4 + stop.numel() * 4), 'd2h_bytes_per_step': 4},
                'gpu_launches': int(launches), 'clocks': clocks, 'loss': loss_val,
                'train_step': {'value': 1e3 / train_ms * world, 'unit': 'steps/s', 'ms_per_step': train_ms, 'loss': train_loss,
                               'gpu_launches_per_step': int(train_launches) // args.steps,
                               'what': 'fwd (dropout 0.1, single-pass bf16) + bwd + Adam, same batch, no gradient all-reduce in this mode'},
                'roofline': {'bound': 'tensor', 'achieved': flops / (ms / args.steps * 1e-3) / 1e12, 'peak': peak_tf, 'unit': 'TFLOP/s',
                             'frac': flops / (ms / args.steps * 1e-3) / 1e12 / peak_tf, 'traffic': None, 'peak_source': peak_src,
                             'kernel': 'whole forward step (algorithmic FLOPs); ~90 small launches per step, latency-bound at this size'},
                'cpu_baseline': cpu}
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--precision', default='bf16x3', choices=['bf16x3', 'bf16'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-graphs', action='store_true', help='inference: eager launches instead of CUDA-graph replay')
    ap.add_argument('--no-train', action='store_true', help='default mode: skip the C3 training-step record')
    ap.add_argument('--mode', default='infer', choices=['infer', 'train', 'stft', 'expand', 'aligner'],
                    help="'train': BASELINE configs[2] (fwd+bwd+Adam, bf16, batch 32/GPU, NCCL data parallel); 'stft': configs[3] "
                         "(STFT->mel, 256 clips x 10 s); 'expand': the length regulator alone (C2-LR)")
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='default mode: write the outputs of the last timed step (rank 0) as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'ours' or args.mode != 'infer'):
        ap.error('--dump-outputs applies to the default inference workload (--impl ours --mode infer)')
    args.warmup = max(args.warmup, 3) if args.impl == 'ours' else args.warmup

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))

    if args.impl == 'reference':
        line = cpu_reference_line(args, rank, world)
        if line is not None:
            print(json.dumps(line), flush=True)
        return

    import torch.distributed as dist
    from oracle import forward_oracle as fo
    from transformertts_b200 import lib
    from transformertts_b200.model.models import ForwardTransformer

    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    lib.load()

    cfg = fo.CONFIGS[CFG_NAME]
    params = fo.init_params(cfg, seed=7)  # random-init weights of the named architecture
    if args.mode in ('stft', 'expand'):
        hbm_bench(args, rank, world, dev, cfg)
        if world > 1:
            dist.destroy_process_group()
        return
    if args.mode == 'aligner':
        aligner_bench(args, rank, world, dev)
        if world > 1:
            dist.destroy_process_group()
        return
    if args.mode == 'train':
        rec = train_bench(args, rank, world, dev, cfg, params)
        if rec is not None:
            print(json.dumps(rec), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return
    model = ForwardTransformer(**cfg, device=str(dev), precision=args.precision, cuda_graphs=not args.no_graphs)
    model.set_weights(params)
    tok, dur, pit = _inputs(200 + rank)  # per-rank shard of the synthetic batch (weak scaling: 64 rows per GPU)
    tok_d, dur_d, pit_d = tok.to(dev), dur.to(dev).float(), pit.to(dev)

    def step_resident():
        return model.call(tok_d, target_durations=dur_d, target_pitch=pit_d)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident throughput ----------------
    for _ in range(args.warmup):
        step_resident()
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    lib.reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = step_resident()
    e1.record()
    barrier()
    launches = lib.launch_count()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    frames_total = world * B * TM * args.steps
    value = frames_total / (ms * 1e-3)

    # ---------------- roofline of the dominant kernel (decoder conv GEMMs), CUDA events, same process ----------------
    model._prof = {}
    for _ in range(3):
        step_resident()
    torch.cuda.synchronize()
    prof, model._prof = model._prof, None
    peak_tf, peak_hbm, peak_src = _peaks()
    tags = {k: v for k, v in prof.items() if k.startswith('decoder.conv')}
    dur_ms = [a.elapsed_time(b) for v in tags.values() for a, b, _ in v]
    flops = [f for v in tags.values() for _, _, f in v]
    gemm_tf = sum(flops) / (sum(dur_ms) * 1e-3) / 1e12 if dur_ms else None
    conv_share = sum(dur_ms) / 3 / (ms / args.steps) if dur_ms else None
    roofline = {'bound': 'tensor', 'kernel': 'gemm_tc_kernel (decoder Conv1D k=3 GEMMs: 256->1024 and 1024->256, M=64000)',
                'achieved': gemm_tf, 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': gemm_tf / peak_tf if gemm_tf else None,
                'traffic': _traffic('conv_gemm_mean_bytes_per_launch'), 'traffic_source': _traffic('source'),
                'peak_source': peak_src, 'launches_timed': len(dur_ms),
                'avg_launch_ms': sum(dur_ms) / len(dur_ms) if dur_ms else None,
                'algorithmic_gflop_per_launch': sum(flops) / len(flops) / 1e9 if flops else None,
                'share_of_step': conv_share}
    step_flops = fo.forward_flops(cfg, [TP] * B, [TM] * B)
    model_tf = step_flops * world / (ms / args.steps * 1e-3) / 1e12

    # ---------------- end to end through predict(): pinned host inputs, mel copied back every step ----------------
    tok_h = tok.numpy()
    dur_h = dur.float().pin_memory()
    pit_h = pit.pin_memory()
    mel_h = [torch.empty((B, TM, cfg['mel_channels']), dtype=torch.float32).pin_memory() for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    e2e_i = [0]

    def step_e2e():
        # host token ids + pinned durations/pitch go in, the step's mel comes back to pinned host memory; the device->host
        # copy runs on its own stream so that it overlaps the next step's kernels (double-buffered host destination)
        o = model.predict(tok_h, encode=False, phoneme_durations=dur_h.to(dev, non_blocking=True),
                          phoneme_pitch=pit_h.to(dev, non_blocking=True))
        ev = torch.cuda.Event()
        ev.record()
        copy_stream.wait_event(ev)
        mel = o['mel']
        mel.record_stream(copy_stream)
        with torch.cuda.stream(copy_stream):
            mel_h[e2e_i[0] & 1].copy_(mel, non_blocking=True)
        e2e_i[0] += 1

    for _ in range(args.warmup):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    barrier()
    dt = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    e2e_val = frames_total / float(dt.item())
    clocks = sampler.stop() if sampler else None  # sampled across both timed regions (device-resident and end-to-end)
    h2d = tok_h.nbytes + dur_h.numel() * 4 + pit_h.numel() * 4 + 2 * tok_h.size * 4  # tokens + durations + pitch + max/min masks
    d2h = mel_h[0].numel() * 4 + B * 4

    # ---------------- fast single-pass bf16 mode (reported, not the headline: it misses the 1e-3 parity gate) ----------------
    fast = None
    if args.precision == 'bf16x3' and rank == 0 and world == 1:
        m2 = ForwardTransformer(**cfg, device=str(dev), precision='bf16', cuda_graphs=not args.no_graphs)
        m2.set_weights(params)
        for _ in range(3):
            o2 = m2.call(tok_d, target_durations=dur_d, target_pitch=pit_d)
        torch.cuda.synchronize()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(args.steps):
            o2 = m2.call(tok_d, target_durations=dur_d, target_pitch=pit_d)
        f1.record()
        torch.cuda.synchronize()
        fast = {'precision': 'bf16', 'value': B * TM * args.steps / (f0.elapsed_time(f1) * 1e-3), 'unit': UNIT,
                'mel_max_abs_diff_vs_bf16x3': float((o2['mel'] - out['mel']).abs().max())}
        del m2

    # ---------------- CPU baseline (oracle port): whole 64-row steps, same method as --impl reference ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        rate, n_pass, secs, cores, ref = cpu_forward_rate(budget_s=20.0, min_passes=1, max_passes=3)
        cpu = {'value': rate, 'unit': UNIT, 'cores': cores, 'kind': 'port',
               'sample': f'{n_pass} whole steps of {B} rows x {TM} frames in {secs:.1f} s, torch-CPU fp32 oracle (same as --impl reference)',
               'mel_max_abs_err_gpu_vs_cpu': float((out['mel'].cpu() - ref['mel']).abs().max())}

    # ---------------- BASELINE configs[2]: the training step (fwd+bwd+Adam, NCCL data parallel when N > 1) ----------------
    train_rec = None
    if not args.no_train:
        del model
        torch.cuda.empty_cache()
        train_rec = train_bench(args, rank, world, dev, cfg, params)

    if rank == 0:
        line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
                'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'bf16x3 (3-pass bf16 tensor-core products, fp32 accumulate)' if args.precision == 'bf16x3' else 'bf16',
                'data': 'synthetic',
                'config': {**_config_dict(world),
                           'parallelism': f'batch-sharded replicas x{world}, no collective (inference)',
                           'launch': 'eager' if args.no_graphs else 'CUDA graphs (encoder half + decoder half, replayed; outputs copied out of the static buffers)',
                           'l2': 'no explicit flush: per-step working set (~1.5 GB of activations) exceeds the 126 MB L2'},
                'e2e': {'value': e2e_val, 'unit': UNIT, 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h)},
                'gpu_launches': int(launches), 'clocks': clocks, 'roofline': roofline,
                'model_tflops': model_tf, 'algorithmic_gflop_per_step_per_gpu': step_flops / 1e9,
                'cpu_baseline': cpu, 'fast_mode': fast, 'train': train_rec,
                'tf_reference_available': _tf_reference_available()}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
