#!/usr/bin/env python
"""Headline benchmark: audio-seconds processed per wall-second (real-time factor) of the SOME inference
hot path (waveform -> log-mel -> two-head conformer -> decoded notes), BASELINE.json configs[1]:
configs/two_head_model.yaml, 64 x 30 s synthetic 44.1 kHz mono clips per GPU, bf16 operands / fp32 accumulate.

    python bench.py --gpus N --steps K --warmup W            # this repo (libsome_b200.so kernels)
    python bench.py --impl reference ...                     # the reference algorithm on the host CPU cores
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/<name>.npy

A "step" = one pass of the hot path over one batch (64 clips x 30 s = 1920 audio-seconds per GPU; weak
scaling: each rank owns its own 64 clips, the only exchange is one all-gather of the packed notes).
  value   : device-timed (CUDA events, max over ranks), audio already resident in HBM when the region starts
  e2e     : the same metric through the plugin's public infer() with HOST numpy buffers: pinned H2D of the
            audio and D2H of the notes (+ the NCCL all-gather at N > 1) inside the timed region
  configs : short legs on the other BASELINE.json configs (C3 quantised head, C4 midi_conformer 32 x 10 s per GPU,
            C5 one 5-minute recording through the slicer: latency), same measurement, fewer steps
  roofline / cpu_baseline / clocks / gpu_launches / parity_check / e2e_breakdown / strong_scaling: DESIGN.md §6.
"""
import argparse
import contextlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

from some_b200 import synth  # noqa: E402

METRIC = 'audio-seconds/sec (real-time factor) two_head conformer'
YAML = {'two_head': 'two_head_model', 'quant_two_head': 'quant_two_head_model', 'midi_conformer': 'midi_conformer'}


def workload_name(config, clips, seconds):
    return (f'configs/{YAML[config]}.yaml, batch={clips}x{seconds:g} s synthetic 44.1 kHz mono clips per GPU, bf16 operands')


def load_peaks():
    try:
        with open(os.path.join(REPO, 'MEASURED_PEAKS.json')) as f:
            p = json.load(f)
        return {'hbm_gbs': p['hbm_gbs'], 'tf_burst': p['bf16_tflops'], 'tf_sustained': p['bf16_tflops_sustained'],
                'source': 'measured (MEASURED_PEAKS.json)'}
    except Exception:
        return {'hbm_gbs': 6650.0, 'tf_burst': 1590.0, 'tf_sustained': 1400.0, 'source': 'fallback (B200_PROFILING.md)'}


def make_clips(first_index, count, seconds):
    """Deterministic synthetic clips.  Generating 64 x 30 s sung-note signals costs ~1 s each; to keep the
    default run within minutes a pool of 8 distinct clips is generated and rotated with distinct gains and
    circular shifts (still 64 different waveforms of the named length)."""
    n = int(round(seconds * synth.SR))
    pool = [synth.synth_waveform(1000 + j, num_samples=n) for j in range(min(8, count))]
    clips = []
    for i in range(count):
        gi = first_index + i
        base = pool[gi % len(pool)]
        clips.append(np.ascontiguousarray(np.roll(base, 4099 * (gi // len(pool))) * np.float32(1.0 - 0.01 * (gi % 7))))
    return clips


DUMP_BYTES = 64 * 10 ** 6 - 2 ** 16            # --dump-outputs: 64 MB in all, with room for the .npy headers


def dump_outputs(out_dir, arrays, seed=0):
    """Writes each array as out_dir/<name>.npy, DUMP_BYTES in all.  The arrays are written smallest first and each may use an
    equal share of the bytes left; a larger one is cut to a fixed, seeded sample of its rows, and <name>_rows.npy holds the
    indices of the rows kept.  Same shapes -> same sample, so two builds can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_BYTES
    items = sorted(arrays.items(), key=lambda kv: kv[1].nbytes)
    for i, (name, a) in enumerate(items):
        share = left // (len(items) - i)
        if a.nbytes > share:
            keep = share // (a.nbytes // len(a) + 8)                # + the float64 row index
            rows = np.sort(np.random.default_rng(seed).choice(len(a), keep, replace=False))
            np.save(os.path.join(out_dir, f'{name}_rows.npy'), rows.astype(np.float64))
            a = a[rows]
            left -= rows.size * 8
        np.save(os.path.join(out_dir, f'{name}.npy'), a)
        left -= a.nbytes


def device_step_outputs(eng, ws, m, cu, note_count):
    """What one device step hands its caller, on the host: the head outputs of every frame and the decoded notes in the
    layout of the note buffers (clip j's notes in rows cu[j] .. cu[j] + note_count[j] - 1, zero beyond), with durations in
    seconds as Engine.infer returns them.  The shapes depend on the inputs only."""
    count = note_count.cpu().numpy().astype(np.int64)
    frames = np.diff(cu)
    used = np.arange(m) - np.repeat(cu[:-1], frames) < np.repeat(count, frames)
    return {'probs': ws.probs[:m].cpu().numpy(), 'bounds': ws.bounds[:m].cpu().numpy(),
            'note_count': count.astype(np.float64),
            'note_midi': np.where(used, ws.note_midi[:m].cpu().numpy(), 0).astype(np.float32),
            'note_dur': np.where(used, ws.note_dur[:m].cpu().numpy() * eng.timestep, 0).astype(np.float64),
            'note_rest': np.where(used, ws.note_rest[:m].cpu().numpy(), 0).astype(np.float32)}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.gpu_index, self.proc, self.path = gpu_index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix='.csv')
            os.close(fd)
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '50', '-i', str(self.gpu_index)],
                                         stdout=open(self.path, 'w'), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, reasons = [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(',')]
                if len(f) < 9:
                    continue
                sm.append(float(f[1]))
                out['sm_max_mhz'] = float(f[2])
                for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out['sm_mhz'] = float(np.median(sm))
            out['samples'] = len(sm)
        out['reasons'] = sorted(reasons)
        return out


# ----------------------------------------------------------------------------------------- reference arm
def time_cpu_reference(config_name, clips, threads=None):
    """Times the reference ALGORITHM on the host cores: the oracle port (oracle/decode.infer = the serial batch-1 loop of
    inference/base_infer.py:46-53 in fp32 torch, with the vectorised decode forms that match the speed of the reference's
    torch ops and the mel basis built once).  /root/reference itself is not on the GPU box; the port is pinned to it by
    tests/golden (also at 30 s / 10 s clips)."""
    from oracle import decode as odecode
    if threads:
        torch.set_num_threads(threads)
    config = synth.named_config(config_name)
    sd = synth.fabricate_state_dict(config, seed=1234)
    t0 = time.perf_counter()
    odecode.infer(sd, config, clips, quantized=config_name.startswith('quant'), fast=True)
    dt = time.perf_counter() - t0
    return sum(len(c) for c in clips) / synth.SR / dt, dt


def pick_cpu_threads(config_name, clip):
    """The reference's small fp32 GEMMs do not scale to every core of a big host (64 threads were slower than 8 in
    the first measurements), and torchrun pins OMP_NUM_THREADS=1.  Be fair to the CPU arm: try a few thread counts
    on one clip and keep the fastest; the sweep is reported."""
    avail = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    cands = sorted({c for c in (8, 16, 32, avail) if c <= avail} | {avail})
    best, best_v, sweep = avail, -1.0, {}
    for c in cands:
        time_cpu_reference(config_name, [clip], threads=c)                # warm-up at this thread count
        v, _ = time_cpu_reference(config_name, [clip], threads=c)
        sweep[str(c)] = round(v, 1)
        if v > best_v:
            best, best_v = c, v
    torch.set_num_threads(best)
    return best, sweep


def run_reference(args, rank, world):
    if rank != 0:
        return
    n_clips = args.ref_clips
    clips = make_clips(0, n_clips, args.seconds)
    cores, sweep = pick_cpu_threads(args.config, clips[0])
    for _ in range(args.warmup):
        time_cpu_reference(args.config, clips[:1])
    times = []
    for _ in range(args.steps):
        _, dt = time_cpu_reference(args.config, clips)
        times.append(dt)
    total = n_clips * args.seconds * args.steps / sum(times)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': total, 'unit': 'audio-s/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1000.0 * sum(times) / len(times),
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': workload_name(args.config, args.clips, args.seconds),
                   'sample': f'{n_clips} x {args.seconds:.0f} s clips per step (serial batch-1 loop)'},
        'cpu_baseline': {'value': total, 'unit': 'audio-s/s', 'cores': cores, 'kind': 'port',
                         'threads_sweep_audio_s_per_s': sweep,
                         'sample': f'{n_clips} x {args.seconds:.0f} s clips x {args.steps} steps, torch fp32 + vectorised decode, '
                                   f'{cores} threads'},
        'e2e': {'value': total, 'unit': 'audio-s/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------- this repo
def build_plugin(config_name, local_rank):
    from some_b200 import plugin
    config = synth.named_config(config_name)
    with tempfile.TemporaryDirectory() as d, contextlib.redirect_stdout(sys.stderr):   # stdout = the ONE JSON line
        ckpt = synth.write_checkpoint(d, config, seed=1234)
        cls = plugin.QuantizedMIDIExtractionInference if config_name.startswith('quant') else plugin.MIDIExtractionInference
        return cls(config=config, model_path=ckpt, device=f'cuda:{local_rank}')


def _pinned(clips):
    from some_b200.engine import pinned_array
    out = []
    for c in clips:
        a = pinned_array(len(c))
        a[:] = c
        out.append(a)
    return out


def measure_batch(ins, config_name, clips_per_gpu, seconds, steps, warmup, rank, world, dev, full, sampler=None,
                  dump_dir=None):
    """Device-resident value, end-to-end value and per-kernel roofline of one (config, batch) on this rank; `full` adds the
    pageable-input variant, the e2e breakdown, the strong-scaling figure and the parity check of the headline line.
    `dump_dir`: write the outputs of the last timed device step there (dump_outputs)."""
    import torch.distributed as dist
    from some_b200 import dist as sdist
    eng = ins.model
    quant = config_name.startswith('quant')
    clips = make_clips(rank * clips_per_gpu, clips_per_gpu, seconds)
    audio_seconds_rank = sum(len(c) for c in clips) / synth.SR

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---------------- device-resident arm ("value")
    host, tables, cu = eng.pack(clips)
    b, m, max_frames = len(clips), int(cu[-1]), int(np.diff(cu).max())
    wave = host.to(dev)
    tables_d, cu_d = tables.to(dev), torch.from_numpy(cu).to(dev)
    ws = eng.workspace(m)
    note_count = torch.empty(b, dtype=torch.int32, device=dev)

    def device_step():
        eng.run_mel(wave, tables_d[:b], tables_d[b:], cu_d, b, max_frames, None, ws.units)
        eng.run_trunk(ws, m, b, cu_d, max_frames, 'softmax' if quant else 'sigmoid')
        eng.run_decode(ws, m, b, cu_d, note_count, quant)

    for _ in range(max(warmup, 3)):
        device_step()
    barrier()
    if sampler is not None:
        sampler.start()
    launches0 = eng.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(steps):
        device_step()                       # product path: native launch sequencer (some_forward)
    ev1.record()
    barrier()
    dev_ms = ev0.elapsed_time(ev1)
    launches = eng.launches - launches0
    if dump_dir is not None:
        dump_outputs(dump_dir, device_step_outputs(eng, ws, m, cu, note_count))
    # second pass of the same K steps with CUDA events around every launch (recorded by the sequencer itself) for the roofline
    eng.start_profile(cu)
    barrier()
    for _ in range(steps):
        device_step()
    prof = eng.stop_profile()
    barrier()
    clocks = sampler.stop() if sampler is not None else None

    # ---------------- end-to-end arm ("e2e"): host numpy in, host numpy out, through the plugin
    # The step's inputs sit in PINNED host memory (numpy views of page-locked buffers, as a production loader would hand
    # them over): the engine copies host -> device straight from them.  (Pageable numpy arrays go through a pinned staging
    # memcpy first; that variant is reported as e2e.pageable_value.)
    pinned_clips = _pinned(clips)
    all_clips = None
    if world > 1:
        # every rank needs the LENGTHS of all clips (they are identical here); only its own shard's samples are touched
        all_clips = [pinned_clips[i % clips_per_gpu] for i in range(world * clips_per_gpu)]

    def e2e_step(src=None):
        if world > 1:
            res = sdist.infer_sharded(ins, all_clips)       # shard -> infer -> ONE NCCL all-gather of the packed notes
            if rank == 0:
                res.materialise()                           # rank 0 consumes every clip's notes (the others: their own)
            return res
        return ins.infer(pinned_clips if src is None else src)

    for _ in range(max(1, min(warmup, 2))):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        res = e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    out = {'audio_seconds_rank': audio_seconds_rank, 'dev_ms': dev_ms, 'e2e_ms': e2e_s * 1000.0, 'launches': launches,
           'prof': prof, 'clocks': clocks, 'frames': m, 'clips': b,
           'h2d': int(host.numel() * 4 + tables.numel() * 8 + cu.nbytes), 'd2h': int(m * 9 + b * 4) * world,
           'audio_mb': host.numel() * 4 / 1e6}
    if not full:
        return out

    if world == 1:                                  # same call with ordinary (pageable) numpy inputs
        e2e_step(clips)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        for _ in range(min(steps, 3)):
            e2e_step(clips)
        out['pageable_s'] = (time.perf_counter() - t1) / min(steps, 3)

    # ---------------- where the end-to-end step goes (each phase timed on its own, median of 3; they overlap in the step)
    def med(fn, n=3):
        ts = []
        for _ in range(n):
            torch.cuda.synchronize(dev)
            t = time.perf_counter()
            fn()
            torch.cuda.synchronize(dev)
            ts.append((time.perf_counter() - t) * 1e3)
        return float(np.median(ts))

    starts, lens, _, total = eng.tables([len(c) for c in clips])
    stage_d = torch.empty(max(total, 4), dtype=torch.float32, device=dev)

    def h2d_all():
        for s, c in zip(starts, pinned_clips):
            stage_d[s:s + len(c)].copy_(torch.from_numpy(c), non_blocking=True)
    slab_d = torch.empty(9 * m + 4 * b + 64, dtype=torch.uint8, device=dev)
    slab_h = torch.empty(slab_d.numel(), dtype=torch.uint8).pin_memory()
    _, _, nbytes = eng.slab_layout(lens)
    if world > 1:
        r_ = sdist.infer_sharded(ins, all_clips)
        t_u = time.perf_counter()
        r_.materialise()
        unpack_ms = (time.perf_counter() - t_u) * 1e3
    else:
        slab, cu_x, layout_x, _ = eng.enqueue(pinned_clips, quant)
        slab_h[:slab.numel()].copy_(slab)
        torch.cuda.synchronize(dev)
        hostbuf = slab_h[:slab.numel()].numpy()
        t_u = time.perf_counter()
        eng.unpack_slab(hostbuf, cu_x, layout_x)
        unpack_ms = (time.perf_counter() - t_u) * 1e3
    bd = {'h2d_audio_ms': med(h2d_all), 'kernels_ms': dev_ms / steps,
          'd2h_notes_ms': med(lambda: slab_h.copy_(slab_d, non_blocking=True)), 'unpack_host_ms': unpack_ms,
          'note': 'phases timed separately; inside infer() the H2D of pipeline chunk c+1 overlaps the kernels of chunk c'}
    if world > 1:
        g = torch.empty(world * nbytes, dtype=torch.uint8, device=dev)
        bd['all_gather_ms'] = med(lambda: dist.all_gather_into_tensor(g, g[rank * nbytes:(rank + 1) * nbytes]))
        bd['all_gather_bytes_per_rank'] = int(nbytes)
        gh = torch.empty(world * nbytes, dtype=torch.uint8).pin_memory()
        bd['d2h_notes_ms'] = med(lambda: gh.copy_(g, non_blocking=True))
        bd['unpack_host_ms_is'] = 'rank 0 materialising all ranks\' clips'
    out['e2e_breakdown'] = bd

    # ---------------- strong scaling: the SAME 64 x 30 s batch split over the N ranks (clips_per_gpu / N each)
    if world > 1:
        for _ in range(2):
            sdist.infer_sharded(ins, pinned_clips)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            r_ = sdist.infer_sharded(ins, pinned_clips)
            if rank == 0:
                r_.materialise()
        barrier()
        out['strong_ms'] = (time.perf_counter() - t0) * 1e3 / steps

    # ---------------- parity of the timed workload: one clip of the batch against the fp32 CPU oracle (checker only)
    if rank == 0:
        try:
            from oracle import decode as odecode
            from oracle.metrics import note_agreement
            config = synth.named_config(config_name)
            sd = synth.fabricate_state_dict(config, seed=1234)
            got = eng.infer([clips[0]], quantized=quant, return_intermediates=True)[0]
            ref = odecode.infer_clip(sd, config, clips[0], quantized=quant, return_intermediates=True, fast=True)
            first = res[0]                                          # clip 0 as decoded inside the LAST timed e2e step
            fr, bd_ = note_agreement(ref, first)
            out['parity_check'] = {
                'clip': 'clip 0 of the timed batch vs the oracle (fp32 torch CPU restatement, pinned to the reference)',
                'max_abs_probs': float(np.abs(got['probs'] - ref['probs']).max()),
                'max_abs_bounds': float(np.abs(got['bounds'] - ref['bounds']).max()),
                'mean_bounds_error': float((got['bounds'].astype(np.float64) - ref['bounds']).mean()),
                'max_abs_logmel': float(np.abs(got['mel'] - ref['mel'].T).max()),
                'tolerance': 1e-2, 'notes': int(len(first['note_midi'])), 'oracle_notes': int(len(ref['note_midi'])),
                'note_frame_agreement': fr, 'note_exact_boundary_agreement': bd_,
                'batched_equals_single': bool(all(np.array_equal(first[k], got[k]) for k in ('note_midi', 'note_dur', 'note_rest'))),
            }
        except Exception as e:                                     # the checker must never take the measurement down
            out['parity_check'] = {'error': repr(e)}
    return out


def summarise(meas, steps, world, peaks):
    """Max-over-ranks times -> values, per-kernel roofline table."""
    import torch.distributed as dist
    dev = torch.device('cuda', torch.cuda.current_device())
    t = torch.tensor([meas['dev_ms'], meas['e2e_ms'], meas.get('strong_ms', 0.0)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, strong_ms = (float(x) for x in t)
    total_audio = meas['audio_seconds_rank'] * world * steps
    prof = meas['prof']
    peak_tf = peaks['tf_sustained']                        # kernels timed inside a long step
    kernels, step_kernel_ms = {}, sum(v['ms'] for v in prof.values())
    for name, v in prof.items():
        rate = v['work'] / (v['ms'] / 1000.0) if v['ms'] > 0 else 0.0
        tensor = name in ('some_gemm', 'some_attention_varlen')
        kernels[name] = {'launches_per_step': v['launches'] // steps, 'ms_per_step': v['ms'] / steps,
                         'share': v['ms'] / step_kernel_ms if step_kernel_ms else 0.0,
                         ('tflops' if tensor else 'gbs'): rate / (1e12 if tensor else 1e9),
                         'frac': rate / ((peak_tf * 1e12) if tensor else (peaks['hbm_gbs'] * 1e9))}
    gemm = prof.get('some_gemm', {'ms': 0.0, 'work': 0.0, 'launches': 0})
    gemm_shapes = {}
    for key, v in sorted(gemm.get('shapes', {}).items()):
        tf = v['work'] / (v['ms'] / 1000.0) / 1e12 if v['ms'] > 0 else 0.0
        gemm_shapes[key] = {'launches_per_step': v['launches'] // steps, 'ms_per_step': round(v['ms'] / steps, 4),
                            'tflops': round(tf, 1), 'frac': round(tf / peak_tf, 3)}
    achieved_tf = gemm['work'] / (gemm['ms'] / 1000.0) / 1e12 if gemm['ms'] > 0 else 0.0
    return {'dev_ms': dev_ms, 'e2e_ms': e2e_ms, 'strong_ms': strong_ms, 'value': total_audio / (dev_ms / 1000.0),
            'e2e_value': total_audio / (e2e_ms / 1000.0), 'kernels': kernels, 'gemm_shapes': gemm_shapes,
            'gemm_tf': achieved_tf, 'peak_tf': peak_tf}


def measure_c5(ins, rank, world, dev, steps=5):
    """C5: ONE 5-minute recording with silence gaps -> slicer (device RMS + host run walk) -> chunks as one var-len batch
    (sharded over the ranks at N > 1) -> notes of every chunk.  Latency, slicer included."""
    import torch.distributed as dist
    from some_b200 import dist as sdist
    from some_b200 import slicer as psl
    from some_b200.engine import pinned_array
    wave = synth.synth_waveform(9002, seconds=300.0, silence_gaps=True)
    pw = pinned_array(len(wave))
    pw[:] = wave
    s = psl.Slicer(synth.SR, max_sil_kept=1000)                      # infer.py:39
    eng = ins.model

    def once():
        if world > 1:
            offs, notes = sdist.infer_sliced_sharded(ins, pw, s)
            if rank == 0 and hasattr(notes, 'materialise'):
                notes.materialise()
            return offs, notes
        return eng.infer_sliced(pw, s)

    for _ in range(2):
        offs, notes = once()
    ts = []
    for _ in range(steps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        once()
        torch.cuda.synchronize(dev)
        ts.append((time.perf_counter() - t0) * 1e3)
    t = torch.tensor([float(np.median(ts))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    return {'workload': 'configs/two_head_model.yaml, one 300 s recording with 0.5-1.0 s silence gaps, utils/slicer2 semantics '
                        '(threshold -40 dB, min_length 5 s, max_sil_kept 1 s), chunks as one var-len batch',
            'chunks': len(offs), 'latency_ms': ms, 'audio_seconds': 300.0, 'value': 300.0 / (ms / 1e3), 'unit': 'audio-s/s',
            'inputs': 'pinned host waveform -> slicer -> notes of every chunk on the host', 'n_gpus': world}


def run_ours(args, rank, world, local_rank):
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    peaks = load_peaks()
    ins = build_plugin(args.config, local_rank)
    eng = ins.model
    sampler = ClockSampler(local_rank) if rank == 0 else None
    meas = measure_batch(ins, args.config, args.clips, args.seconds, args.steps, args.warmup, rank, world, dev, True, sampler,
                         args.dump_outputs if rank == 0 else None)
    s = summarise(meas, args.steps, world, peaks)

    extra = {}
    if not args.skip_extra_configs:
        legs = [('C3_quant_two_head_64x30s', 'quant_two_head', 64, 30.0), ('C4_midi_conformer_32x10s', 'midi_conformer', 32, 10.0)]
        for key, cfg, n, secs in legs:
            if (cfg, n, secs) == (args.config, args.clips, args.seconds):
                continue
            try:
                ins_x = build_plugin(cfg, local_rank)
                mx = measure_batch(ins_x, cfg, n, secs, 3, 3, rank, world, dev, False)
                sx = summarise(mx, 3, world, peaks)
                extra[key] = {'workload': workload_name(cfg, n, secs), 'value': sx['value'], 'e2e_value': sx['e2e_value'],
                              'unit': 'audio-s/s', 'ms_per_step': sx['dev_ms'] / 3, 'e2e_ms_per_step': sx['e2e_ms'] / 3,
                              'steps': 3, 'frames_per_gpu': mx['frames'], 'gemm_tflops': sx['gemm_tf'],
                              'gemm_frac': sx['gemm_tf'] / sx['peak_tf'] if sx['peak_tf'] else None,
                              'kernels_ms_per_step': {k: round(v['ms_per_step'], 3) for k, v in sx['kernels'].items()}}
                del ins_x
                torch.cuda.empty_cache()
            except Exception as e:
                extra[key] = {'error': repr(e)}
        try:
            ins5 = ins if args.config == 'two_head' else build_plugin('two_head', local_rank)
            extra['C5_5min_sliced'] = measure_c5(ins5, rank, world, dev)
        except Exception as e:
            extra['C5_5min_sliced'] = {'error': repr(e)}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ref_clips = make_clips(0, args.ref_clips, args.seconds)
        cores, sweep = pick_cpu_threads(args.config, ref_clips[0])
        v, dt = time_cpu_reference(args.config, ref_clips)
        cpu = {'value': v, 'unit': 'audio-s/s', 'cores': cores, 'kind': 'port', 'threads_sweep_audio_s_per_s': sweep,
               'sample': f'{args.ref_clips} x {args.seconds:.0f} s clips of the same workload, oracle port '
                         f'(torch fp32, serial batch-1 loop, vectorised decode), {dt:.1f} s of CPU work'}
    if rank != 0:
        return

    traffic, traffic_src = None, None
    for name in ('r02_gemm_traffic.json', 'r01_gemm_traffic.json'):
        try:
            with open(os.path.join(REPO, 'profiles', name)) as f:
                traffic = json.load(f).get('dram_bytes_per_launch')
                traffic_src = (f'profiles/{name} (ncu dram__bytes_read.sum + dram__bytes_write.sum of the same command; '
                               f'not re-measured in this run)')
                break
        except Exception:
            pass
    m = meas['frames']
    line = {
        'metric': METRIC, 'value': s['value'], 'unit': 'audio-s/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': max(args.warmup, 3), 'ms_per_step': s['dev_ms'] / args.steps, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
        'config': {'workload': workload_name(args.config, args.clips, args.seconds), 'clips_per_gpu': args.clips,
                   'clip_seconds': args.seconds, 'frames_per_gpu': m, 'parallelism': f'dp{world}',
                   'l2': f'inputs ({meas["audio_mb"]:.0f} MB audio, {m * 512 * 4 * 2 / 1e9:.1f} GB residual streams) exceed the 126 MB L2',
                   'weights': 'seeded random (no pretrained checkpoint offline)',
                   'ln_fold': bool(eng.ln_fold), 'bias_correction': bool(eng.bias_correction)},
        'e2e': {'value': s['e2e_value'], 'unit': 'audio-s/s', 'h2d_bytes_per_step': meas['h2d'], 'd2h_bytes_per_step': meas['d2h'],
                'ms_per_step': s['e2e_ms'] / args.steps, 'inputs': 'pinned host numpy arrays -> plugin.infer -> host numpy notes',
                'pageable_value': (meas['audio_seconds_rank'] / meas['pageable_s']) if meas.get('pageable_s') else None},
        'e2e_breakdown': meas.get('e2e_breakdown'),
        'gpu_launches': meas['launches'],
        'roofline': {'kernel': 'some_gemm (tcgen05, all shapes of a step)', 'bound': 'tensor', 'achieved': s['gemm_tf'],
                     'peak': s['peak_tf'], 'unit': 'TFLOP/s', 'frac': s['gemm_tf'] / s['peak_tf'] if s['peak_tf'] else None,
                     'traffic': traffic, 'traffic_source': traffic_src, 'peak_source': peaks['source'] + ', sustained bf16',
                     'measured_in': 'second pass of the same K steps with CUDA events around every launch (some_profiler)'},
        'kernels': s['kernels'],
        'gemm_shapes': s['gemm_shapes'],
        'clocks': meas['clocks'],
        'parity_check': meas.get('parity_check'),
    }
    if world > 1 and s['strong_ms'] > 0:
        line['strong_scaling'] = {'workload': f'the same {args.clips} x {args.seconds:g} s batch split over {world} ranks',
                                  'ms_per_step': s['strong_ms'], 'value': args.clips * args.seconds / (s['strong_ms'] / 1e3),
                                  'unit': 'audio-s/s', 'path': 'end to end (infer_sharded: host in, all-gathered notes on the host)'}
    if extra:
        line['configs'] = extra
    if cpu is not None:
        line['cpu_baseline'] = cpu
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--ref-clips', type=int, default=8, help='bounded CPU sample: clips per CPU step')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--skip-extra-configs', action='store_true', help='only the headline workload (developer A/B runs)')
    # extra measurements for the BASELINE.md table (the default = the contract workload, BASELINE.json configs[1])
    ap.add_argument('--config', default='two_head', choices=['two_head', 'quant_two_head', 'midi_conformer'])
    ap.add_argument('--clips', type=int, default=64, help='clips per GPU')
    ap.add_argument('--seconds', type=float, default=30.0, help='clip length')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write the outputs of the last one (rank 0: probs, bounds, notes) as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of this project\'s path (--impl ours)')
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == '__main__':
    main()
