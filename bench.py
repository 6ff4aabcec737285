#!/usr/bin/env python
"""Benchmark of the hot path: batched incremental generation with the Transformer-XL of BASELINE.json.

Workload (BASELINE.json configs[1], "C2"): musicautobot-default Transformer-XL (d_model 512, 16 layers, 8 heads x 64,
d_inner 2048, mem_len 512, vocab 324, random init), 256 independent streams per GPU, memory filled by a 512-token
prefill of synthetic tokens, then one-token steps (S = 513) with top-k/top-p sampling on the device, bf16.
A "step" = one generated token for every stream.  `value` = generated tokens/s over all GPUs (weak scaling:
256 streams per GPU, no collective on the data path).

  python bench.py [--gpus N] [--steps K] [--warmup W]            this repo's CUDA path
  python bench.py --impl reference [--steps K] [--warmup W]      the reference's algorithm on the host CPU cores
                                                                  (the oracle restatement: the reference itself needs
                                                                  fastai==1.0.61/music21, not installable offline)

`--dump-outputs DIR` (CUDA path) also writes, after the timed steps, what the last timed step of each leg returned to its
caller, as DIR/<name>.npy: `tokens` (C1: the generated stream; C2 / C5: every stream's token of the last step), `train_losses`
(C3: loss, ce, ar, tar, grad_norm after the last step), `bert_logits` (C4: the last-position logits of the last forward).  Inputs
are seeded, so two builds run with the same arguments can be compared output for output.  `tokens` and `bert_logits` repeat bit
for bit from run to run; `train_losses` do not, because the training kernels accumulate some gradients with atomic adds in no
fixed order (two runs on a B200 at its 1000 W power limit differed by up to 4e-5 relative in the losses and 9e-4 in grad_norm).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC, UNIT = 'generated_tokens_per_sec', 'tokens/s'
B_PER_GPU, PREFILL, V = 256, 512, 324
CFG = dict(d_model=512, n_layers=16, n_heads=8, d_head=64, d_inner=2048, mem_len=512)
WORKLOAD = ('C2: Transformer-XL d_model 512, 16 layers, 8 heads x 64, d_inner 2048, mem_len 512, vocab 324; '
            '256 streams/GPU, one-token steps over a full 512-slot memory (S=513), top_k 30 / top_p 0.65 sampling')
# BASELINE.json configs[4] (not the headline; `--workload c5`): the scaled model, streams sharded over the GPUs
CFG_C5 = dict(d_model=1024, n_layers=24, n_heads=16, d_head=64, d_inner=4096, mem_len=1024)
WORKLOAD_C5 = ('C5: Transformer-XL d_model 1024, 24 layers, 16 heads x 64, d_inner 4096, mem_len 1024, vocab 324; '
               '256 streams/GPU (K/V rings 25.8 GB), one-token steps over a full 1024-slot memory, top_k 30 / top_p 0.65 sampling')


def measured_peaks():
    try:
        p = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        return float(p['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md)'


def dump_outputs(path, outputs):
    """Writes `outputs` (name -> array) as path/<name>.npy, float64 arrays as float64 and everything else as float32.  The files stay
    under 64 MB in all: an array above 16 MB (there are at most three) keeps a fixed, seeded sample of its rows."""
    os.makedirs(path, exist_ok=True)
    for name, a in outputs.items():
        a = np.asarray(a)
        a = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
        if a.nbytes > 16 << 20:
            keep = (16 << 20) // (a.nbytes // len(a))
            a = a[np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))]
        np.save(os.path.join(path, name + '.npy'), a)


def attention_bytes_per_launch(B, H=8, Dh=64, M=512, e=2):
    "Algorithmic bytes of ONE fused decode-attention launch (one layer): K and V rings read once, new K/V written, "
    "rel-pos key cache once, q/k/v of the new token read, output written (DESIGN.md section 5)."
    kv_read = B * H * M * 2 * Dh * e
    kv_write = B * H * 2 * Dh * e
    rcache = H * (M + 1) * Dh * e
    qkv_in = B * 3 * H * Dh * 4
    out = B * H * Dh * e
    return kv_read + kv_write + rcache + qkv_in + out


def step_bytes(B, L=16, d=512, H=8, Dh=64, di=2048, M=512, e=2):
    "Algorithmic HBM bytes of one whole decode step (SURVEY.md 8d): K/V read+write, weights once, rel-pos cache."
    HD = H * Dh
    kv = B * L * M * 2 * HD * e + B * L * 2 * HD * e
    w = (L * (d * 3 * HD + HD * d + d * di + di * d) + V * d) * e
    r = L * (M + 1) * HD * e
    return kv + w + r


class ClockSampler:
    "nvidia-smi clocks + throttle reasons sampled DURING the timed region."
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '100',
                                          '-i', str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(',')]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 <= t <= t1 + 0.2] or [r for _, r in self.rows]
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for n, val in zip(names, r[2:6]):
                if val.lower().startswith('active'):
                    reasons.add(n)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


# --------------------------------------------------------------------------------------------- CPU reference arm
class CpuReference:
    """The reference algorithm on the host: eager PyTorch fp32, hidden-state memory re-projected to K/V every step, materialised
    _line_shift (oracle/txl.py).  Memory is pre-filled with random hidden states (its contents do not change the cost)."""
    def __init__(self):
        from oracle import txl
        torch.manual_seed(0)
        self.threads = os.cpu_count() or 1
        torch.set_num_threads(self.threads)
        self.model = txl.get_language_model(V, txl.baseline_config()).eval()

    def run(self, batch, steps, warmup, budget_s):
        "-> (tokens/s, steps timed, seconds)"
        enc = self.model[0]
        enc.reset(); enc.init = True
        enc.hidden = [torch.randn(batch, CFG['mem_len'], CFG['d_model']) for _ in range(CFG['n_layers'] + 1)]
        x = torch.randint(0, V, (batch, 1), generator=torch.Generator().manual_seed(1234))
        t_begin = time.time()
        with torch.no_grad():
            for _ in range(warmup):
                x = self.model(x)[0][:, -1].argmax(-1, keepdim=True)
            done, t0 = 0, time.time()
            for _ in range(steps):
                x = self.model(x)[0][:, -1].argmax(-1, keepdim=True)
                done += 1
                if time.time() - t_begin > budget_s:
                    break
            dt = time.time() - t0
        return batch * done / dt, done, dt

    def best_batch(self, candidates=(8, 32, 64)):
        "The CPU's own best case: the batch (of the candidates) with the highest tokens/s over three steps."
        rates = {}
        for b in candidates:
            rates[b] = self.run(b, 3, 1, budget_s=60.0)[0]
        return max(rates, key=rates.get), rates


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    if args.workload == 'c1':
        return print(json.dumps(c1_line(args, cpu_only=True)), flush=True)
    ref = CpuReference()
    batch, rates = ref.best_batch()
    warm = min(args.warmup, 2)
    value, done, dt = ref.run(batch, args.steps, warm, budget_s=150.0)
    sample = (f'{batch} streams x {done} one-token steps over a full 512-slot memory, greedy, fp32 eager PyTorch oracle '
              f'(reference algorithm: hidden-state mems re-projected every step), {ref.threads} threads; batch chosen as the '
              f'fastest of a sweep: ' + ', '.join(f'{b}: {r:.0f} tok/s' for b, r in rates.items()))
    line = {'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': done,
            'warmup': warm, 'ms_per_step': 1e3 * dt / max(done, 1), 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'cpu_batch': batch, 'cpu_batch_sweep_tok_s': rates},
            'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': ref.threads, 'kind': 'port', 'sample': sample},
            'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------- C1: the reference's own CPU-runnable case
def c1_line(args, cpu_only=False, outputs=None):
    """BASELINE.json configs[0]: random-init Transformer-XL (C2's model), seed = the whole encoded fur_elise.mid, 512 greedy tokens,
    fp32.  CPU: the oracle's reference loop (deep_music_genre.py:1853-1972), wall time split into prefill and decode.  GPU: the same
    call through MusicLearner.predict in fp32 mode; the two token streams must be identical."""
    from oracle import codec as ocodec, sampling as osamp, txl
    mid = os.path.join(ROOT, 'tests', 'golden', 'fur_elise.mid')
    ov = ocodec.MusicVocab.create()
    seed = ocodec.seed_from_midi(mid, ov, strip_eos=True)
    pos = ocodec.position_enc(seed.copy(), ov)
    n_words = 512
    torch.manual_seed(0)
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    om = txl.get_language_model(V, txl.baseline_config()).eval()
    with torch.no_grad():
        om[1].decoder.bias[308:] = -50.          # mt*/dummy* ids: never filtered by the reference, never produced by a trained model
    marks = []
    t0 = time.time()
    ref = osamp.predict(om, ov, seed, pos, n_words=n_words, temperatures=(1., 1., 1.), min_bars=10 ** 6, top_k=1, top_p=0.0,
                        on_step=lambda i, lg: marks.append(time.time()))
    t_cpu = time.time() - t0
    prefill_cpu = marks[0] - t0
    cpu = {'value': len(ref) / (t_cpu - prefill_cpu), 'unit': UNIT, 'cores': threads, 'kind': 'port',
           'sample': f'the whole case: seed {len(seed)} tokens prefilled in {prefill_cpu:.1f} s, {len(ref)} greedy tokens in '
                     f'{t_cpu - prefill_cpu:.1f} s, total wall {t_cpu:.1f} s (fp32 eager-PyTorch oracle, reference loop)',
           'wall_s': t_cpu, 'prefill_s': prefill_cpu}
    base = {'metric': METRIC, 'unit': UNIT, 'n_gpus': 1, 'steps': len(ref), 'warmup': 0, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'fur_elise.mid seed (tests/golden), random-init weights',
            'config': {'workload': 'C1: Transformer-XL d_model 512, 16 layers, 8 heads x 64, mem_len 512, vocab 324, random init; '
                                   f'generate {n_words} greedy tokens from the encoded fur_elise.mid ({len(seed)} tokens), batch 1, fp32'},
            'cpu_baseline': cpu}
    if cpu_only:
        return dict(base, impl='reference', value=cpu['value'], ms_per_step=1e3 * (t_cpu - prefill_cpu) / max(len(ref), 1),
                    e2e={'value': cpu['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}, gpu_launches=0)
    from deepmusicgeneration_b200 import _lib
    from deepmusicgeneration_b200.codec import MusicDataBunch, MusicItem
    from deepmusicgeneration_b200.learner import MusicLearner
    from deepmusicgeneration_b200.model import get_language_model
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device - the CUDA path has no CPU fallback')
    lib = _lib.load()
    data = MusicDataBunch.empty('')
    item = MusicItem.from_file(mid, data.vocab)
    item = MusicItem(item.data[:-1], data.vocab) if item.data[-1] == data.vocab.stoi['xxeos'] else item
    assert list(item.data) == list(seed), 'MIDI -> token encoding differs from the oracle'
    pm = get_language_model(V, txl.baseline_config(), dtype='f32', device=0, max_batch=1, max_seq=len(seed), keep_hidden=False, init=False)
    pm.load_state_dict(om.state_dict())
    learn = MusicLearner(data, pm)
    learn.predict(item, n_words=8, temperatures=(1., 1., 1.), min_bars=10 ** 6, top_k=1, top_p=0.0)        # warm-up
    torch.cuda.synchronize()
    l0 = lib.dmg_launch_count()
    t0 = time.time()
    pred, _ = learn.predict(item, n_words=n_words, temperatures=(1., 1., 1.), min_bars=10 ** 6, top_k=1, top_p=0.0)
    torch.cuda.synchronize()
    t_gpu = time.time() - t0
    if outputs is not None:
        outputs['tokens'] = np.asarray(pred.data)
    same = list(pred.data) == list(ref)
    return dict(base, value=len(pred.data) / t_gpu, ms_per_step=1e3 * t_gpu / max(len(pred.data), 1),
                config=dict(base['config'], token_stream_identical_to_oracle=same, gpu_wall_s=t_gpu,
                            note='value = generated tokens / wall seconds of the whole predict() call (seed encoding excluded, '
                                 'prefill of the seed included), host buffers in, tokens out'),
                e2e={'value': len(pred.data) / t_gpu, 'unit': UNIT, 'h2d_bytes_per_step': 16 * len(seed) // max(len(pred.data), 1),
                     'd2h_bytes_per_step': 4},
                gpu_launches=int(lib.dmg_launch_count() - l0))


# --------------------------------------------------------------------------------------------- CUDA arm
def run_b200(args):
    "C2 headline + (default run) the C3 training step and the C4 encoder forward as sub-records of the one JSON line."
    outputs = {} if args.dump_outputs else None
    line = measure_c2(args, outputs)
    if args.workload == 'c2' and not args.no_extra_legs:
        import argparse
        import bench_bert
        import bench_train
        sub = argparse.Namespace(**vars(args))
        sub.steps, sub.warmup = args.train_steps, 4
        train = bench_train.measure(sub, sample_clocks=False, outputs=outputs)
        sub.steps, sub.warmup = args.bert_steps, 3
        bert = bench_bert.measure(sub, sample_clocks=False, outputs=outputs)
        if line is not None:
            line['train'], line['bert'] = train, bert
            line['gpu_launches_all_legs'] = line['gpu_launches'] + train['gpu_launches'] + bert['gpu_launches']
    if line is not None:
        print(json.dumps(line), flush=True)
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)


def measure_c2(args, outputs=None):
    from deepmusicgeneration_b200 import _lib, sharding
    from deepmusicgeneration_b200.app_utils import baseline_config
    from deepmusicgeneration_b200.codec import MusicDataBunch
    from deepmusicgeneration_b200.learner import MusicLearner, sampler_params, vocab_layout
    from deepmusicgeneration_b200.model import _ptr, get_language_model

    rank, local_rank, world = sharding.init_distributed()
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device - the CUDA path has no CPU fallback (use --impl reference for the CPU arm)')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    B, K, W = args.batch, args.steps, max(args.warmup, 3)
    lib = _lib.load()

    c5 = args.workload == 'c5'
    shape = CFG_C5 if c5 else CFG
    workload = WORKLOAD_C5 if c5 else WORKLOAD
    PREFILL = shape['mem_len']                     # fills the memory ring exactly
    cfg = dict(baseline_config(), **shape, ctx_len=PREFILL)
    model = get_language_model(V, cfg, dtype='bf16', device=local_rank, max_batch=B, max_seq=PREFILL, max_rows=B * 64,
                               keep_hidden=False, seed=0)
    data = MusicDataBunch.empty('')
    learn = MusicLearner(data, model)
    e = model._e

    # synthetic LakhMIDI-shaped seeds: (note, duration, instrument) triplets; every stream ends on an instrument token
    g = torch.Generator().manual_seed(1234 + rank)
    trip = torch.stack([torch.randint(12, 140, (B, PREFILL // 3 + 1), generator=g),
                        torch.randint(140, 301, (B, PREFILL // 3 + 1), generator=g),
                        torch.randint(301, 308, (B, PREFILL // 3 + 1), generator=g)], dim=2).reshape(B, -1)
    seeds = trip[:, -PREFILL:].contiguous()
    assert seeds.shape == (B, PREFILL) and int(seeds[0, -1]) >= 301
    seeds_pinned = seeds.pin_memory()

    model.reset()
    learn._prefill(seeds_pinned.to(dev, non_blocking=True), None)
    vl = vocab_layout(data.vocab)
    params = sampler_params(data.vocab, 10 ** 9, (1.0, 1.0, 1.0), 10 ** 6, 30, 0.65, None, flags=_lib.SAMPLE_MASK_UNUSED, seed=7)
    prev = np.ascontiguousarray(seeds[:, -1].numpy().astype(np.int32))
    lp = np.zeros(B, dtype=np.int64)
    _lib.check(lib.dmg_sampler_init(e.h, C.byref(vl), C.byref(params), prev.ctypes.data_as(C.c_void_p),
                                    lp.ctypes.data_as(C.c_void_p), B), 'dmg_sampler_init')
    toks = torch.empty(max(K, W), B, dtype=torch.int32, device=dev)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def generate(n):
        _lib.check(lib.dmg_generate(e.h, n, _ptr(toks), stream), 'dmg_generate')

    generate(W)                                   # warm-up (also captures the CUDA graph of the one-token forward)
    torch.cuda.synchronize()

    # ---- timed region: K steps, device-resident (inputs already in HBM)
    sharding.barrier(); torch.cuda.synchronize()
    clocks = ClockSampler(local_rank) if rank == 0 else None
    launches0 = lib.dmg_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    ev0.record()
    generate(K)
    ev1.record()
    torch.cuda.synchronize()
    t1 = time.time()
    sharding.barrier()
    ms = ev0.elapsed_time(ev1)
    launches = int(lib.dmg_launch_count() - launches0)
    clock_info = clocks.stop(t0, t1) if clocks else None
    ms_max = sharding.max_over_ranks(ms, device=dev)
    value = B * world * K / (ms_max / 1e3)
    good = int((toks[:K] >= 0).all().item())
    if outputs is not None:
        outputs['tokens'] = toks[K - 1].cpu().numpy()

    # ---- end to end through the C ABI with HOST buffers: H2D of the step's input ids, D2H of the sampled tokens
    Ke = min(K, 512)
    ids_host = torch.empty(B, dtype=torch.int64).pin_memory()
    tok_host = torch.empty(B, dtype=torch.int32).pin_memory()
    ids_host.copy_(toks[K - 1].to(torch.int64).clamp_min(1).cpu())
    for _ in range(3):
        _lib.check(lib.dmg_generate_step_host(e.h, C.c_void_p(ids_host.data_ptr()), C.c_void_p(tok_host.data_ptr()), stream), 'step_host')
        ids_host.copy_(tok_host.to(torch.int64).clamp_min(1))
    sharding.barrier(); torch.cuda.synchronize()
    ev0.record()
    for _ in range(Ke):
        _lib.check(lib.dmg_generate_step_host(e.h, C.c_void_p(ids_host.data_ptr()), C.c_void_p(tok_host.data_ptr()), stream), 'step_host')
        ids_host.copy_(tok_host.to(torch.int64).clamp_min(1))        # the host's view of x = new_tensor([idx])
    ev1.record()
    torch.cuda.synchronize()
    e2e_ms = sharding.max_over_ranks(ev0.elapsed_time(ev1), device=dev)
    e2e_value = B * world * Ke / (e2e_ms / 1e3)

    # ---- roofline of the dominant kernel, timed alone with CUDA events on its stream.  The pipelined step (B > 32 streams) spends
    # its time in decode_dual_kernel: the attention of one half of the streams (HBM-bound: that half's K/V rings once) next to the
    # fused layer step of the other half (one layer's weights once); 2 L - 1 such launches per step.  Launches over consecutive
    # layers touch different rings and weights (4.4 GB per sweep) -> every launch reads cold data (L2 = 126 MB).
    L = cfg['n_layers']
    peak, peak_src = measured_peaks()
    geo = dict(H=shape['n_heads'], Dh=shape['d_head'], M=shape['mem_len'])
    sbytes = step_bytes(B, L=shape['n_layers'], d=shape['d_model'], di=shape['d_inner'], **geo)
    reps = 8
    dual_on = lib.dmg_decode_dual_launch(e.h, 0, stream) == 0
    traffic = None
    if dual_on:
        for l in range(L - 1):
            _lib.check(lib.dmg_decode_dual_launch(e.h, l, stream), 'decode_dual_launch')
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(reps):
            for l in range(L - 1):
                lib.dmg_decode_dual_launch(e.h, l, stream)
        ev1.record()
        torch.cuda.synchronize()
        k_ms = ev0.elapsed_time(ev1) / (reps * (L - 1))
        half = B - ((B + 31) // 32 + 1) // 2 * 32                                  # streams of the attention role (second half)
        d_, di_, HD_ = shape['d_model'], shape['d_inner'], shape['n_heads'] * shape['d_head']
        wbytes = (HD_ * d_ + 2 * d_ * di_ + d_ * 3 * HD_) * 2                      # out-proj, FFN up / down, next q|k|v (bf16)
        abytes = attention_bytes_per_launch(half, **geo) + wbytes
        per_step = 2 * L - 1
        kname = 'decode_dual_kernel (decode_layer.cu): attn_decode3 body over half the streams + fused layer step of the other half'
        tpath = os.path.join(ROOT, 'profiles', 'decode_dual_traffic.json')
    else:
        for l in range(L):
            _lib.check(lib.dmg_attn_decode_layer(e.h, l, stream), 'attn_decode_layer')
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(reps):
            for l in range(L):
                lib.dmg_attn_decode_layer(e.h, l, stream)
        ev1.record()
        torch.cuda.synchronize()
        k_ms = ev0.elapsed_time(ev1) / (reps * L)
        abytes = attention_bytes_per_launch(B, **geo)
        per_step = L
        third = shape['mem_len'] % 128 == 0 and shape['mem_len'] <= 512 and shape['d_head'] == 64
        kname = ('attn_decode3_kernel (attention_decode3.cuh)' if third else
                 'attn_decode2_kernel<G> (attention_decode2.cuh; mem_len outside the third kernel\'s range)')
        tpath = os.path.join(ROOT, 'profiles', 'attn_decode_traffic.json')
    achieved = abytes / (k_ms / 1e3) / 1e9
    if os.path.exists(tpath) and not c5:                     # the ncu captures were taken at the C2 geometry
        try: traffic = json.load(open(tpath)).get('dram_bytes_per_launch')
        except Exception: traffic = None
    roofline = {'bound': 'hbm', 'kernel': kname, 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                'frac': achieved / peak, 'traffic': traffic, 'peak_source': peak_src,
                'algorithmic_bytes_per_launch': abytes, 'kernel_ms': k_ms, 'launches_per_step': per_step,
                'kernel_share_of_step': k_ms * per_step / (ms / K),
                'step_algorithmic_bytes': sbytes, 'step_frac': sbytes / (ms / K / 1e3) / 1e9 / peak}

    uses_tc = bool(lib.dmg_uses_tcgen05(e.h))
    del learn, model, e, toks
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    cpu = None
    if world == 1 and not args.no_cpu_baseline and not c5:
        ref = CpuReference()
        cb, rates = ref.best_batch((8, 32))
        v, done, dt = ref.run(cb, 100000, 1, budget_s=15.0)                    # a bounded sample: about 15 s of host work
        cpu = {'value': v, 'unit': UNIT, 'cores': ref.threads, 'kind': 'port',
               'sample': f'{cb} streams x {done} one-token steps over a full 512-slot memory, fp32 eager-PyTorch oracle '
                         f'(reference algorithm), {dt:.1f} s; batch = the faster of ' + ', '.join(f'{b}: {r:.0f} tok/s' for b, r in rates.items())}
    line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': K, 'warmup': W,
            'ms_per_step': ms_max / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16',
            'data': 'synthetic',
            'config': {'workload': workload, 'batch_per_gpu': B, 'global_batch': B * world, 'prefill': PREFILL,
                       'parallelism': f'streams sharded over {world} GPU(s), no collective',
                       'l2': f'inputs larger than L2: every step streams {sbytes / 1e9:.1f} GB of K/V through a 126 MB L2',
                       'tcgen05_gemm': uses_tc, 'all_streams_alive': bool(good)},
            'roofline': roofline, 'cpu_baseline': cpu,
            'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': B * 8, 'd2h_bytes_per_step': B * 4, 'steps': Ke},
            'gpu_launches': launches, 'clocks': clock_info}
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None)
    ap.add_argument('--warmup', type=int, default=None)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='c2', choices=['c1', 'c2', 'c3', 'c4', 'c5'],
                    help='c2 (default, the headline; its line also carries the c3 and c4 legs as `train` / `bert`): batched incremental '
                         'generation; c1: 512 greedy tokens from fur_elise.mid, CPU oracle wall + CUDA fp32; c3: data-parallel training '
                         'step alone; c4: remix (masked-BERT) encoder forward alone; c5: the scaled generation model')
    ap.add_argument('--no-extra-legs', action='store_true', help='c2 only: skip the `train` (C3) and `bert` (C4) sub-records')
    ap.add_argument('--train-steps', type=int, default=12, help='timed steps of the C3 leg inside the default run')
    ap.add_argument('--bert-steps', type=int, default=5, help='timed forwards of the C4 leg inside the default run')
    ap.add_argument('--batch', type=int, default=B_PER_GPU, help='c2: streams per GPU')
    ap.add_argument('--train-batch', type=int, default=32, help='c3: sequences per GPU and step')
    ap.add_argument('--bert-batch', type=int, default=512, help='c4: sequences per GPU and forward')
    ap.add_argument('--bert-chunk', type=int, default=32, help='c4: sequences per activation chunk of the encoder forward (max_rows / 1024)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last timed step returned (rank 0) as DIR/<name>.npy')
    args = ap.parse_args()
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the CUDA path (--impl b200)')
    if args.workload == 'c1':
        if args.impl == 'reference':
            return run_reference(args)
        if int(os.environ.get('RANK', '0')) == 0:
            outputs = {} if args.dump_outputs else None
            print(json.dumps(c1_line(args, outputs=outputs)), flush=True)
            if outputs is not None:
                dump_outputs(args.dump_outputs, outputs)
        return
    if args.workload == 'c3':
        import bench_train
        args.steps = args.steps if args.steps is not None else 30
        args.warmup = args.warmup if args.warmup is not None else 5
        return bench_train.run_reference(args) if args.impl == 'reference' else bench_train.run_b200(args)
    if args.workload == 'c4':
        import bench_bert
        args.steps = args.steps if args.steps is not None else 10
        args.warmup = args.warmup if args.warmup is not None else 3
        return bench_bert.run_reference(args) if args.impl == 'reference' else bench_bert.run_b200(args)
    args.steps = args.steps if args.steps is not None else 2048
    args.warmup = args.warmup if args.warmup is not None else 32
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
