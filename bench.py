#!/usr/bin/env python
"""bench.py -- embeddings/sec of the waveform -> front-end -> backbone -> embedding path on the BASELINE.json configs.

    python bench.py [--config c2|c3|c4|c5] [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Default (what the driver runs): c2 = EcapaTdnn + Fbank-80, 256 x 3 s @ 16 kHz per GPU (BASELINE configs[1]).  The other
BASELINE configurations are selected with --config (SURVEY.md 8d):
    c3  CAM++ + Fbank-80, 256 x 3 s per GPU (global 2048 on 8 GPUs)
    c4  ResNetSE + MelSpectrogram (README.md:303-311 method_args), 128 x 5 s per GPU
    c5  ERes2Net 55 M + Fbank-80, ragged 1-10 s (randint(16000, 160001) samples), 64 per GPU (global 256 on 4 GPUs),
        every shard padded to the GLOBAL longest item (reference single-batch semantics)
One "step" = one pass of the hot path over one global batch (weak scaling: per-GPU work fixed).  All configs shard by
contiguous utterance ranges through the product API ``mvector.distributed`` (``gather_embeddings`` /
``predict_batch_sharded``): one all-gather of the [B/R, 192] embeddings, no other collective.

Timed quantities (CUDA events on the launching stream, max over ranks, barrier + synchronize on both sides):
  value    : whole-job embeddings/s with the (padded) waveforms already resident in HBM:
             MVectorPredictor.embed_device (vp_embed_wave per chunk) + all-gather
  e2e      : the same through the public API on HOST data -- predict_batch_sharded(list of host float32 arrays): native
             threaded gather into pinned memory, H2D, kernels, all-gather, D2H -- all inside the timed region
  roofline : the dominant kernel (largest device-time share among the program's ops, measured live with per-op CUDA
             events by vp_embed_profiled on extra steps after the timed region): algorithmic FLOPs / its launch time vs
             the measured dense bf16 tensor peak of MEASURED_PEAKS.json (burst figure: the kernel is timed alone);
             `whole_step` uses the sustained figure
  cpu_baseline : the UNMODIFIED reference (oracle/_ref, installed by build()) through its own
             MVectorPredictor.predict_batch on the box's host cores, bounded sample, separate process (falls back to the
             oracle port only if oracle/_ref is missing)
  gpu_eager_baseline : the same reference on the same GPU with stock PyTorch eager kernels (cuDNN / cuBLAS), TF32 as
             shipped and off, with its parity error against the reference's CPU fp32 result -- context, not the target
`--impl reference` runs the reference arm alone and prints the same JSON line with "impl": "reference".
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_POOL = 4                     # rotating input batches: >= 160 MB per GPU > 126 MB L2
FBANK80 = dict(sample_frequency=16000, num_mel_bins=80)
MEL64 = dict(sample_rate=16000, n_fft=1024, win_length=1024, hop_length=320, f_min=50.0, f_max=14000.0, n_mels=64)

CONFIGS = {
    'c2': dict(idx=2, model='EcapaTdnn', margs=dict(embd_dim=192, pooling_type='ASP', channels=[512, 512, 512, 512, 1536]),
               feature='Fbank', fargs=FBANK80, fdim=80, per_gpu=256, samples=48000, ragged=False, steps=50,
               metric='embeddings/sec (3s@16kHz) ECAPA-TDNN', ref_sample=64, cpu_sample=32,
               workload='EcapaTdnn+Fbank80, batch 256 x 3 s @ 16 kHz per GPU (BASELINE configs[1])'),
    'c3': dict(idx=3, model='CAMPPlus', margs=dict(embd_dim=192), feature='Fbank', fargs=FBANK80, fdim=80, per_gpu=256,
               samples=48000, ragged=False, steps=30, metric='embeddings/sec (3s@16kHz) CAM++', ref_sample=32, cpu_sample=32,
               workload='CAM++ +Fbank80, batch 256 x 3 s @ 16 kHz per GPU = 2048 over 8 GPUs (BASELINE configs[2])'),
    'c4': dict(idx=4, model='ResNetSE', margs=dict(embd_dim=192, pooling_type='ASP'), feature='MelSpectrogram', fargs=MEL64,
               fdim=64, per_gpu=128, samples=80000, ragged=False, steps=30, metric='embeddings/sec (5s@16kHz) ResNetSE',
               ref_sample=16, cpu_sample=16,
               workload='ResNetSE+MelSpectrogram(n_fft 1024, hop 320, 64 mels; README.md:303-311), batch 128 x 5 s @ 16 kHz '
                        'per GPU (BASELINE configs[3])'),
    'c5': dict(idx=5, model='ERes2Net', margs=dict(embd_dim=192, m_channels=64, mul_channel=2, expansion=4, base_width=24, scale=3),
               feature='Fbank', fargs=FBANK80, fdim=80, per_gpu=64, samples=None, ragged=True, steps=10,
               metric='embeddings/sec (ragged 1-10s@16kHz) ERes2Net-55M', ref_sample=4, cpu_sample=4,
               workload='ERes2Net 55M +Fbank80, ragged batch randint(16000,160001) samples, 64 per GPU = 256 over 4 GPUs, '
                        'padded to the global longest item (BASELINE configs[4])'),
}


def bench_config(cfg, n_gpus, lmax):
    return {'workload': cfg['workload'], 'global_batch': cfg['per_gpu'] * n_gpus, 'samples_per_utt': cfg['samples'] or f'1..10 s, padded to {lmax}',
            'parallelism': f'utterance-sharded x{n_gpus} (mvector.distributed) + one all-gather of the embeddings',
            'l2': f'inputs rotate over {N_POOL} distinct batches (> L2); per-step activation traffic is several GB',
            'weights': 'seeded random init + randomised BN statistics (oracle.models.random_state_dict seed 0)',
            'precision': 'fp32 in/out; tensor-core GEMMs use error-compensated two-term splits (fp32-grade, 1e-4 parity)'}


def batch_lens(cfg, n, seed):
    """Lengths (samples) of a global batch of n utterances (SURVEY.md 8d)."""
    if not cfg['ragged']:
        return [cfg['samples']] * n
    import torch
    g = torch.Generator().manual_seed(seed)
    return torch.randint(16000, 160001, (n,), generator=g).tolist()


def synth_waves(lens, seed):
    """One seeded randn stream, sigma 0.1 (= -20 dBFS, what _load_audio's normaliser emits); same code as
    baseline/ref_driver.py so both arms see identical waveforms."""
    import torch
    g = torch.Generator().manual_seed(seed)
    return [(torch.randn(int(n), generator=g) * 0.1).numpy() for n in lens]


def yml_config(cfg):
    return {'dataset_conf': {'dataset': {'min_duration': 0.3, 'max_duration': 3, 'sample_rate': 16000,
                                         'use_dB_normalization': False, 'target_dB': -20},
                             'eval_conf': {'batch_size': 16, 'max_duration': 20}},
            'preprocess_conf': {'use_hf_model': False, 'feature_method': cfg['feature'], 'method_args': dict(cfg['fargs'])},
            'model_conf': {'model': cfg['model'], 'model_args': dict(cfg['margs'])}}


def save_weights(cfg, td):
    import torch
    from oracle import models as om
    gain = getattr(om, 'CONDITIONED_GAIN', {}).get(cfg['model'])
    kw = dict(gain=gain) if gain is not None else {}
    sd = om.random_state_dict(cfg['model'], cfg['fdim'], seed=0, **kw, **cfg['margs'])
    torch.save({'0.' + k: v for k, v in sd.items()}, os.path.join(td, 'model.pth'))
    return sd


def write_dumps(path, arrays):
    """--dump-outputs: one float32 DIR/<name>.npy per timed path, what a caller received from its last timed step
    (at most 2048 x 192 floats each)."""
    if not path:
        return
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + '.npy'), np.ascontiguousarray(a, dtype=np.float32))


def cpu_model():
    try:
        with open('/proc/cpuinfo') as f:
            return next(l.split(':', 1)[1].strip() for l in f if l.startswith('model name'))
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------------------------
# reference arm: the unmodified reference in a separate process (baseline/ref_driver.py)
# ------------------------------------------------------------------------------------------------------------------
def ref_available():
    from oracle import reference
    return reference.installed()


def run_ref_driver(cfg, model_dir, lens, seed, device='cpu', steps=1, warmup=1, budget_s=0.0, tf32=None, mode='predict_batch',
                   batch_size=32, save_emb=None, timeout=1500):
    spec = {'configs': yml_config(cfg), 'model_path': model_dir, 'lens': [int(x) for x in lens], 'seed': seed, 'device': device,
            'steps': steps, 'warmup': warmup, 'budget_s': budget_s, 'tf32': tf32, 'mode': mode, 'batch_size': batch_size,
            'save_emb': save_emb}
    with tempfile.NamedTemporaryFile('w', suffix='.json', delete=False) as f:
        json.dump(spec, f)
        path = f.name
    env = {k: v for k, v in os.environ.items() if k not in ('OMP_NUM_THREADS', 'MKL_NUM_THREADS', 'RANK', 'WORLD_SIZE', 'LOCAL_RANK',
                                                            'MASTER_ADDR', 'MASTER_PORT', 'PYTHONPATH')}
    if device == 'cpu':
        env['CUDA_VISIBLE_DEVICES'] = ''
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, 'baseline', 'ref_driver.py'), path], capture_output=True, text=True,
                           timeout=timeout, env=env, cwd=os.path.join(ROOT, 'baseline'))
    except subprocess.TimeoutExpired:
        return {'unavailable': 'reference driver timed out'}
    finally:
        os.unlink(path)
    for ln in reversed(r.stdout.strip().splitlines()):
        if ln.startswith('{'):
            return json.loads(ln)
    return {'unavailable': 'reference driver failed: ' + (r.stderr.strip().splitlines() or ['no output'])[-1][:300]}


def port_pass(cfg, sd, waves):
    """Fallback when oracle/_ref is absent: the oracle port of predict.py:244-264 (kind = "port")."""
    import numpy as np
    import torch
    from oracle import frontend as ofe
    from oracle import models as om
    with torch.no_grad():
        x, ratio = ofe.pad_batch(waves)
        feats = ofe.featurize(x, ratio, cfg['feature'], cfg['fargs'])
        out = [om.forward(cfg['model'], sd, feats[i:i + 32], **cfg['margs']) for i in range(0, feats.shape[0], 32)]
    return torch.cat(out).numpy()


def run_reference_arm(args, cfg):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    n = cfg['ref_sample']
    lens = batch_lens(cfg, n, 4321 + cfg['idx'])
    lmax = max(lens)
    sample = (f'{n} utterances per step (bounded sample of the {cfg["per_gpu"]}-utterance per-GPU batch'
              + (f', ragged, padded to {lmax} samples' if cfg['ragged'] else f' x {cfg["samples"] / 16000:.0f} s') + ')')
    with tempfile.TemporaryDirectory() as td:
        sd = save_weights(cfg, td)
        if ref_available():
            out = run_ref_driver(cfg, td, lens, 4321, device='cpu', steps=args.steps, warmup=max(args.warmup, 1))
            kind = 'reference'
            sample += '; unmodified reference MVectorPredictor.predict_batch (oracle/_ref), default batch_size 32, autograd on as shipped'
        else:
            out = {'unavailable': 'oracle/_ref missing'}
        if 'unavailable' in out:
            import torch
            kind = 'port'
            sample += f'; oracle port of predict_batch ({out["unavailable"]})'
            waves = synth_waves(lens, 4321)
            torch.set_num_threads(max((os.cpu_count() or 2) // 2, 1))
            for _ in range(max(args.warmup, 1)):
                port_pass(cfg, sd, waves)
            t0 = time.perf_counter()
            for _ in range(args.steps):
                port_pass(cfg, sd, waves)
            el = time.perf_counter() - t0
            out = {'emb_per_s': n * args.steps / el, 'ms_per_step': 1e3 * el / args.steps, 'threads': torch.get_num_threads(),
                   'cpu_model': cpu_model()}
    v = out['emb_per_s']
    line = {'impl': 'reference', 'metric': cfg['metric'], 'value': v, 'unit': 'emb/s', 'n_gpus': args.gpus, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': out['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': bench_config(cfg, args.gpus, lmax),
            'cpu_baseline': {'value': v, 'unit': 'emb/s', 'cores': out.get('threads'), 'kind': kind, 'sample': sample,
                             'cpu_model': out.get('cpu_model')},
            'e2e': {'value': v, 'unit': 'emb/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi sampled DURING the timed region (B200_PROFILING.md clocks line): started before the warm-up so that it is
    already streaming, every sample carries a timestamp and only those inside [t0, t1] (the timed region) are used."""
    Q = ('timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
        self.p = None
        self.t0 = self.t1 = None
        try:
            self.p = subprocess.Popen(['nvidia-smi', f'--id={gpu_index}', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                       '-lms', '20'], stdout=self.f, stderr=subprocess.DEVNULL)
            time.sleep(1.0)                      # let it start streaming
        except Exception:
            self.p = None

    def mark_start(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        import datetime
        out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': []}
        if self.p is None:
            return out
        time.sleep(0.05)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        rows = []
        for ln in self.f.read().splitlines():
            c = [x.strip() for x in ln.split(',')]
            if len(c) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(c[0], '%Y/%m/%d %H:%M:%S.%f').timestamp()
                rows.append((ts, float(c[1]), float(c[2]), c[5:9]))
            except ValueError:
                continue
        inside = [r for r in rows if self.t0 is not None and self.t0 - 0.02 <= r[0] <= self.t1 + 0.02]
        window = 'timed region'
        if len(inside) < 2:                      # region shorter than the sampling period: widen to warm-up + region
            inside, window = rows, 'warm-up + timed region'
        reasons = set()
        for _, _, _, flags in inside:
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), flags):
                if v.lower().startswith('active'):
                    reasons.add(name)
        if inside:
            sm = sorted(r[1] for r in inside)
            out = {'sm_mhz': statistics.median(sm), 'sm_max_mhz': max(r[2] for r in inside), 'reasons': sorted(reasons),
                   'samples': len(inside), 'window': window}
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


# ------------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------------
def run_gpu_arm(args, cfg):
    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    assert torch.cuda.is_available(), 'bench.py needs a GPU (no CPU fallback on the product path)'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)

    def mark(msg):
        if os.environ.get('VPB_BENCH_TRACE'):
            sys.stderr.write(f'[bench rank {rank} {time.strftime("%H:%M:%S")}] {msg}\n')
            sys.stderr.flush()
    if world > 1:
        import datetime
        dist.init_process_group('nccl', device_id=dev, timeout=datetime.timedelta(seconds=300))
        mark('process group up')
    assert world == args.gpus, f'--gpus {args.gpus} but WORLD_SIZE={world}'

    import __graft_entry__ as ge
    ge.build()
    from loguru import logger
    logger.remove()
    from mvector import _lib as L
    from mvector import distributed as mdist
    from mvector.predict import MVectorPredictor
    bound = mdist.bind_rank_to_local_cpus(local, int(os.environ.get('LOCAL_WORLD_SIZE', world)))
    mark(f'cpu affinity: {len(bound) if bound else "unchanged"}')

    td_obj = tempfile.TemporaryDirectory()
    td = td_obj.name
    sd = save_weights(cfg, td)
    pred = MVectorPredictor(configs=yml_config(cfg), model_path=td, use_gpu=True)
    B = cfg['per_gpu']
    n_glob = B * world
    lo, hi = mdist.shard_range(n_glob, rank, world)
    fz = pred._audio_featurizer
    D = pred.predictor.embd_dim

    # ---- synthetic pools: every rank knows all lengths (-> global Lmax) but only materialises its own shard
    pools = []
    for i in range(N_POOL):
        lens = batch_lens(cfg, n_glob, 1234 + cfg['idx'] + 17 * i)
        lmax = max(lens)
        mine = synth_waves(lens[lo:hi], 1234 + 1000 * cfg['idx'] + 100 * rank + i)
        xd = torch.zeros(hi - lo, lmax, dtype=torch.float32)
        for j, w in enumerate(mine):
            xd[j, :w.shape[0]] = torch.from_numpy(w)
        # predict_batch_sharded input: the whole list; entries outside this rank's shard are length-only placeholders
        # (never read: a rank touches only its shard) -- in-shard entries are independently allocated pageable arrays
        full = [mine[j - lo] if lo <= j < hi else np.empty(lens[j], dtype=np.float32) for j in range(n_glob)]
        keep = None
        if cfg['ragged']:                               # mask lengths round(len / Lmax * T) (featurizer.py:82-84), resident too
            keep = fz.keep_frames(torch.tensor([l / lmax for l in lens[lo:hi]], dtype=torch.float32), fz.num_frames(lmax)).to(dev)
        pools.append(dict(lens=lens, lmax=lmax, dev=xd.to(dev), host_list=full, mine=mine, keep=keep))
    lmax0 = pools[0]['lmax']
    emb_all = torch.empty(n_glob, D, dtype=torch.float32, device=dev)

    def step_resident(i):
        p = pools[i % N_POOL]
        loc = pred.embed_device(p['dev'], keep=p['keep'])
        return mdist.gather_embeddings(loc, n_glob, out=emb_all)

    def step_e2e(i):
        return mdist.predict_batch_sharded(pred, pools[i % N_POOL]['host_list'])

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    dumps = {}

    def timed(step_fn, steps, warmup, sampler=None, dump=None):
        for i in range(warmup):
            step_fn(i)
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if sampler:
            sampler.mark_start()
        e0.record()
        for i in range(steps):
            out = step_fn(warmup + i)
        e1.record()
        sync_all()
        if sampler:
            sampler.mark_end()
        if dump and args.dump_outputs and rank == 0:     # copied now: later steps reuse the output buffers
            dumps[dump] = out.cpu().numpy() if torch.is_tensor(out) else np.array(out)
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    mark('programs built, starting timed region')
    clocks = ClockSampler(local) if rank == 0 else None
    ms_res = timed(step_resident, args.steps, args.warmup, clocks, dump='embeddings')
    clk = clocks.stop() if clocks else None
    mark(f'resident timing done: {ms_res:.2f} ms')
    if args.light:
        if rank == 0:
            write_dumps(args.dump_outputs, dumps)
            print(json.dumps({'light': True, 'config': args.config, 'ms_per_step': ms_res / args.steps, 'note': 'not a bench value'}))
        if world > 1:
            dist.destroy_process_group()
        return
    ms_e2e = timed(step_e2e, args.steps, max(args.warmup, 3), dump='e2e_embeddings')
    mark(f'e2e timing done: {ms_e2e:.2f} ms')

    # consistency of the two paths on this rank: resident and host-staged results of the same batch (same kernels, same
    # data; the host path cuts the backbone into smaller chunks, so the fp16-split activation scales may differ: a few ulp)
    i_chk = 0
    e_res = step_resident(i_chk).clone()
    e_host = torch.from_numpy(step_e2e(i_chk)).to(dev)
    sync_all()
    dis = float(((e_res - e_host).norm(dim=1) / e_res.norm(dim=1)).max())
    assert dis <= 2e-6, f'resident and host-staged paths disagree: rel-L2 {dis}'

    # ---- SURVEY 8(d)'s other end-to-end starting point: the shard already zero padded in ONE pinned host matrix (what a
    # serving stack with its own staging hands over).  H2D of the matrix in backbone-chunk pieces on a copy stream, the
    # product's device entry point (embed_device) behind each piece, all-gather, D2H.  Reported beside `e2e`, never instead.
    pinned, pin_err = None, None
    try:                                                 # set-up (pinned allocations) may fail on one rank only ...
        whole_fe = fz.feat_fun.desc.post == 1 and fz.feat_fun.desc.top_db >= 0      # MFCC: the clamp spans the call
        pins = [p['dev'].cpu().pin_memory() for p in pools]
        stage = [torch.empty_like(p['dev']) for p in pools]
        cstream = torch.cuda.Stream(device=dev)
        loc_pin = torch.empty(B, D, dtype=torch.float32, device=dev)
    except Exception as e:
        pin_err = f'{type(e).__name__}: {e}'[:200]
    ok = torch.tensor([0 if pin_err else 1], device=dev)
    if world > 1:                                        # ... so the ranks agree before anyone enters a collective
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if int(ok.item()) == 1:
        def step_pinned(i):
            k = i % N_POOL
            p, src, dst = pools[k], pins[k], stage[k]
            cuts = [B] if whole_fe else pred._host_chunks(B, fz.num_frames(p['lmax']))
            main = torch.cuda.current_stream(dev)
            cstream.wait_stream(main)
            evs, r = [], 0
            with torch.cuda.stream(cstream):
                for c in cuts:
                    dst[r:r + c].copy_(src[r:r + c], non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record(cstream)
                    evs.append(ev)
                    r += c
            r = 0
            for c, ev in zip(cuts, evs):
                main.wait_event(ev)
                pred.embed_device(dst[r:r + c], lens=p['lens'][lo + r:lo + r + c] if cfg['ragged'] else None, out=loc_pin[r:r + c])
                r += c
            return mdist.gather_embeddings(loc_pin, n_glob, out=emb_all).cpu()

        try:                                             # an extra figure: a (rank-symmetric) failure must not take the line down
            ms_pin = timed(step_pinned, args.steps, max(args.warmup, 3), dump='pinned_embeddings')
            e_pin = step_pinned(i_chk).to(dev)
            sync_all()
            dis_pin = float(((e_res - e_pin).norm(dim=1) / e_res.norm(dim=1)).max())
            pinned = {'value': n_glob * args.steps / (ms_pin * 1e-3), 'unit': 'emb/s', 'ms_per_step': ms_pin / args.steps,
                      'max_rel_l2_vs_resident': dis_pin,
                      'input': 'per rank one zero-padded pinned float32 [B/R, Lmax] matrix (no host gather)',
                      'api': 'cudaMemcpyAsync pieces + MVectorPredictor.embed_device + gather_embeddings + D2H'}
            mark(f'pinned-matrix e2e done: {ms_pin:.2f} ms')
        except Exception as e:
            pinned = {'error': f'{type(e).__name__}: {e}'[:200]}
        del pins, stage
    else:
        pinned = {'error': pin_err or 'set-up failed on another rank'}

    T0 = fz.num_frames(lmax0)
    cb = pred._chunk_size(B, T0)
    prog = pred.predictor.program(cb, T0)
    n_chunks = -(-B // cb)
    fe_launches = 3 if fz.feat_fun.desc.post == 1 else 2
    launches_per_step = n_chunks * (prog.launches + fe_launches)

    # ---- live per-op timing for the roofline (extra steps, not part of `value`) ----
    roof = None
    if rank == 0:
        p0 = pools[0]
        ratio = torch.tensor([l / p0['lmax'] for l in p0['lens'][lo:hi]], dtype=torch.float32)
        f_in = fz(p0['dev'][:cb], ratio[:cb] if cfg['ragged'] else None).contiguous()
        emb = torch.empty(cb, D, dtype=torch.float32, device=dev)
        acc, nprof = None, 3
        for _ in range(nprof):
            ops = prog.run_profiled(f_in, emb)
            if acc is None:
                acc = ops
            else:
                for a, o in zip(acc, ops):
                    a['ms'] += o['ms']
        for a in acc:
            a['ms'] /= nprof
        total = sum(a['ms'] for a in acc)
        if args.dump_ops:
            with open(args.dump_ops, 'w') as f:
                json.dump(acc, f, indent=0)
        conv = [a for a in acc if a['kind'] == L.OP_CONV and a['K'] > 0]
        peaks = {}
        ppath = os.path.join(ROOT, 'MEASURED_PEAKS.json')
        if os.path.exists(ppath):
            with open(ppath) as f:
                peaks = json.load(f)
        peak = peaks.get('bf16_tflops')
        peak_src = 'MEASURED_PEAKS.json bf16_tflops (burst: the kernel is event-timed alone; of measured)'
        peak_sus = peaks.get('bf16_tflops_sustained')
        hbm = peaks.get('hbm_gbs')
        if peak is None:
            peak, peak_src, peak_sus, hbm = 1590.0, 'fallback 1.59 PFLOP/s burst (B200_PROFILING.md; of fallback)', 1400.0, 6650.0
        # algorithmic work of every op from the lowered program (same op order as the profile): FLOPs = 2 M N K of the
        # reference's conv / linear, bytes = every operand read once + the result written once
        geo = pred.predictor.lower(cb, T0).finalize().ops
        assert len(geo) == len(acc)
        for a, o in zip(acc, geo):
            rows_in, rows_out = o.B * o.Tin * o.Fin, o.B * o.Tout * o.Fout
            if a['kind'] in (L.OP_CONV, L.OP_CONV_C1):
                cin2 = o.Cin2 if o.src2_mode == L.SRC2_CONCAT else (o.Cin if o.src2_mode == L.SRC2_ADD else 0)
                a['flops'] = 2.0 * a['M'] * a['N'] * a['K']
                a['bytes'] = 4.0 * (rows_in * (o.Cin + cin2) + rows_out * o.Cout * (2 if o.res >= 0 else 1) + o.Cout * a['K'])
            else:
                a['flops'] = 0.0
                reads = {L.OP_EW: 1 + (1 if o.res >= 0 else 0) + (1 if o.mode == L.EW_AFF else 0), L.OP_COLSTATS: 1,
                         L.OP_ASP_POOL: 2, L.OP_POOL2D: 1}.get(a['kind'], 1)
                writes = rows_in * o.Cin if a['kind'] == L.OP_EW else (rows_out * o.Cin if a['kind'] == L.OP_POOL2D else 0)
                a['bytes'] = 4.0 * (reads * rows_in * o.Cin + writes)
            a['t_tensor_ms'] = a['flops'] / (peak * 1e12) * 1e3
            a['t_hbm_ms'] = a['bytes'] / (hbm * 1e9) * 1e3
        classes = {}
        for a in acc:
            classes.setdefault((a['kind'], a['M'], a['N'], a['K'], a['engine']), []).append(a)
        eng_name = {L.ENGINE_TC: 'conv_tc_kernel (tcgen05, split-TF32)', L.ENGINE_TC16: 'conv_tc_kernel (tcgen05, two-term FP16 split)',
                    L.ENGINE_FFMA: 'conv_ffma / linear_small_m (fp32 FFMA)'}
        kind_name = {L.OP_CONV: None, L.OP_CONV_C1: 'conv_c1 (Cin = 1 stem)', L.OP_COLSTATS: 'colstats', L.OP_ASP_POOL: 'asp_pool',
                     L.OP_EW: 'ew', L.OP_POOL2D: 'pool2d'}

        def describe(key, ops):
            kind, M, N, K, eng = key
            ms = sum(o_['ms'] for o_ in ops) / len(ops)
            tt, th = ops[0]['t_tensor_ms'], ops[0]['t_hbm_ms']
            bound = 'tensor' if tt >= th else 'hbm'
            d = {'kernel': (kind_name.get(kind) or eng_name.get(eng, str(eng))) + f' M={M} N={N}' + (f' K={K}' if K else ''),
                 'launches_per_forward': len(ops), 'ms_per_launch': ms, 'share_of_backbone': sum(o_['ms'] for o_ in ops) / total,
                 'bound': bound, 'frac': max(tt, th) / ms}
            if bound == 'tensor':
                d.update(achieved=ops[0]['flops'] / (ms * 1e-3) / 1e12, peak=peak, unit='TFLOP/s')
            else:
                d.update(achieved=ops[0]['bytes'] / (ms * 1e-3) / 1e9, peak=hbm, unit='GB/s')
            return d

        by_time = sorted(classes.items(), key=lambda kv: -sum(o_['ms'] for o_ in kv[1]))
        # the dominant kernel = the single launch with the largest device time; its class mates share shape and kernel
        top_key = max(classes, key=lambda k: max(o_['ms'] for o_ in classes[k]))
        top = describe(top_key, classes[top_key])
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, 'profiles', 'roofline_traffic.json')
        if os.path.exists(tpath):
            with open(tpath) as f:
                tj = json.load(f)
            traffic = tj.get(f'{top_key[1]}x{top_key[2]}x{top_key[3]}')
            traffic_src = tj.get('source', 'profiles/ (ncu --set full capture of the same kernel and shape; not measured in this run)')
        gemm_ms = sum(a['ms'] for a in conv)
        gemm_flops = sum(a['flops'] for a in conv)
        step_flops = gemm_flops * n_chunks * world
        roof = {'bound': top['bound'], 'achieved': top['achieved'], 'peak': top['peak'], 'unit': top['unit'], 'frac': top['frac'],
                'traffic': traffic, 'traffic_source': traffic_src,
                'peak_source': peak_src if top['bound'] == 'tensor' else 'MEASURED_PEAKS.json hbm_gbs (of measured)',
                'kernel': top['kernel'] + f" x{top['launches_per_forward']} per forward",
                'kernel_ms': top['ms_per_launch'], 'kernel_share_of_backbone': top['share_of_backbone'],
                'classes': [describe(k, v) for k, v in by_time if sum(o_['ms'] for o_ in v) / total >= 0.03],
                'all_conv': {'tflops': gemm_flops / (gemm_ms * 1e-3) / 1e12, 'ms': gemm_ms, 'share_of_backbone': gemm_ms / total},
                'backbone_ms_profiled': total,
                'whole_step': {'tflops': step_flops / (ms_res / args.steps * 1e-3) / 1e12, 'peak': peak_sus * world,
                               'frac': step_flops / (ms_res / args.steps * 1e-3) / 1e12 / (peak_sus * world),
                               'peak_source': 'bf16_tflops_sustained x n_gpus (kernels timed inside a long step)'}}

    if rank == 0:
        n_emb = n_glob * args.steps
        value = n_emb / (ms_res * 1e-3)
        e2e_v = n_emb / (ms_e2e * 1e-3)
        h2d = (hi - lo) * lmax0 * 4 * world          # every rank copies its zero-padded [B/R, Lmax] shard
        line = {'metric': cfg['metric'], 'value': value, 'unit': 'emb/s', 'n_gpus': world,
                'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_res / args.steps,
                'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
                'config': bench_config(cfg, world, lmax0), 'clocks': clk,
                'e2e': {'value': e2e_v, 'unit': 'emb/s', 'h2d_bytes_per_step': h2d,
                        'd2h_bytes_per_step': n_glob * D * 4, 'ms_per_step': ms_e2e / args.steps,
                        'api': 'mvector.distributed.predict_batch_sharded(MVectorPredictor, list of host float32 arrays) '
                               '(== MVectorPredictor.predict_batch at 1 GPU)',
                        'host': {'cpus_bound': len(bound) if bound else None, 'cgroup_cpu_quota': MVectorPredictor._cgroup_cpus(),
                                 'gather_threads_per_rank': MVectorPredictor._gather_threads()},
                        'from_pinned_matrix': pinned},
                'gpu_launches': args.steps * launches_per_step,
                'launches_per_step': launches_per_step,
                'roofline': roof}
        if world == 1 and not args.no_baselines:
            line.update(side_baselines(cfg, td, sd, pred, dev))
        write_dumps(args.dump_outputs, dumps)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    td_obj.cleanup()


def side_baselines(cfg, td, sd, pred, dev):
    """cpu_baseline (reference CPU), gpu_eager_baseline (reference on the same GPU, PyTorch eager) and this repo's parity
    against the reference's CPU fp32 result -- all on the SAME bounded sample, after the timed regions."""
    import numpy as np
    import torch
    out = {}
    n = cfg['cpu_sample']
    lens = batch_lens(cfg, n, 4321 + cfg['idx'])
    seed = 4321
    lmax = max(lens)
    what = f'{n} utterances' + (f', ragged, padded to {lmax} samples' if cfg['ragged'] else f' x {cfg["samples"] / 16000:.0f} s')
    emb_path = os.path.join(td, 'ref_cpu.npy')
    ref = None
    if ref_available():
        r = run_ref_driver(cfg, td, lens, seed, device='cpu', steps=1, warmup=1, budget_s=10.0, save_emb=emb_path)
        if 'unavailable' not in r:
            out['cpu_baseline'] = {'value': r['emb_per_s'], 'unit': 'emb/s', 'cores': r['threads'], 'kind': 'reference',
                                   'cpu_model': r.get('cpu_model'),
                                   'sample': f'{what}, {r["steps"]} passes in {r["elapsed_s"]:.1f} s; unmodified reference '
                                             'MVectorPredictor.predict_batch (oracle/_ref) in a separate process, autograd on as shipped'}
            ref = np.load(emb_path)
    waves = synth_waves(lens, seed)
    if ref is None:                                     # oracle/_ref missing: oracle port, labelled as such
        torch.set_num_threads(max((os.cpu_count() or 2) // 2, 1))
        port_pass(cfg, sd, waves)
        t0, reps = time.perf_counter(), 0
        while time.perf_counter() - t0 < 10.0:
            ref = port_pass(cfg, sd, waves)
            reps += 1
        el = time.perf_counter() - t0
        out['cpu_baseline'] = {'value': n * reps / el, 'unit': 'emb/s', 'cores': torch.get_num_threads(), 'kind': 'port',
                               'cpu_model': cpu_model(), 'sample': f'{what}, {reps} passes in {el:.1f} s; oracle port of predict_batch'}
    mine = pred.predict_batch(waves)
    rel = np.linalg.norm(mine - ref, axis=1) / np.linalg.norm(ref, axis=1)
    out['parity_vs_reference_cpu'] = {'rel_l2_max': float(rel.max()), 'n': n, 'tolerance': 1e-4,
                                      'against': out['cpu_baseline']['kind']}
    assert rel.max() < 1e-4, f'parity check inside bench failed: rel-L2 {rel.max()}'
    if ref_available():
        eager = {}
        full_lens = batch_lens(cfg, cfg['per_gpu'], 1234 + cfg['idx'])
        torch.cuda.synchronize()
        for tag, tf32 in (('tf32_as_shipped', None), ('tf32_off', False)):
            gp = os.path.join(td, f'ref_gpu_{tag}.npy')
            rs = run_ref_driver(cfg, td, lens, seed, device='cuda', steps=1, warmup=1, tf32=tf32, save_emb=gp)
            if 'unavailable' in rs:
                eager[tag] = rs
                continue
            g = np.load(gp)
            err = float((np.linalg.norm(g - ref, axis=1) / np.linalg.norm(ref, axis=1)).max())
            r1 = run_ref_driver(cfg, td, full_lens, 1234, device='cuda', steps=3, warmup=2, tf32=tf32)
            r2 = run_ref_driver(cfg, td, full_lens, 1234, device='cuda', steps=5, warmup=2, tf32=tf32, mode='model_only', batch_size=32)
            r3 = run_ref_driver(cfg, td, full_lens, 1234, device='cuda', steps=5, warmup=2, tf32=tf32, mode='model_only',
                                batch_size=cfg['per_gpu'])
            eager[tag] = {'predict_batch_emb_per_s': r1.get('emb_per_s'), 'model_only_bs32_emb_per_s': r2.get('emb_per_s'),
                          'model_only_full_batch_emb_per_s': r3.get('emb_per_s'), 'rel_l2_vs_reference_cpu': err,
                          'tf32': rs.get('tf32')}
        eager['note'] = ('unmodified reference modules on this GPU with PyTorch eager (cuDNN/cuBLAS): predict_batch keeps the '
                         'Kaldi front-end on the CPU (predict.py:256); model_only = backbone with features resident on the device')
        out['gpu_eager_baseline'] = eager
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--config', default='c2', choices=sorted(CONFIGS))
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--light', action='store_true', help='resident-input timing only (for runs under ncu): no e2e / '
                    'baselines / per-op profile; the JSON line is NOT a bench value')
    ap.add_argument('--no-baselines', action='store_true', help='skip the cpu / gpu-eager reference side runs')
    ap.add_argument('--dump-ops', default=None, help='write the per-op device-time profile (JSON) to this path')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='b200 arm only: after the timed steps, write the embeddings each timed path returned in its last '
                         'step as DIR/<path>.npy (float32); the inputs depend only on the arguments, so two builds '
                         'compare output for output')
    args = ap.parse_args()
    cfg = CONFIGS[args.config]
    if args.steps is None:
        args.steps = cfg['steps'] if args.impl == 'b200' else 5
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs applies to the b200 arm only')
    if args.impl == 'reference':
        run_reference_arm(args, cfg)
    else:
        run_gpu_arm(args, cfg)


if __name__ == '__main__':
    main()
