"""bench.py - frame-pairs/sec of the adversarial train step at 256x448 (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload train|gen_fwd|ensemble] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Headline workload `train` (BASELINE.json configs[1]/[2]): DAVIS2016-shaped adversarial training, 4 frame pairs per GPU, PWC-Net at
384x640 in the loop, generator + inpainter alternating 1 recover : 3 generator steps (common_flags.py:19-21), synthetic frames and
seeded random-init weights of the reference architecture.  One "step" = one alternating train step on one batch.
`value`: steps with the batch already resident in HBM.  `e2e`: the same steps through AdversarialLearner.step() fed from
pinned host memory (H2D inside the timed region) with a D2H read of the losses every step.
Other arms (not the headline; BASELINE.json configs[0] and configs[4]):
  --workload gen_fwd    mask-net forward on one 128x224 frame pair with a precomputed flow (test_generator.py path of the reference)
  --workload ensemble   multi-crop ensemble inference (test_generator_ensemble.py / generate_buffer_DAVIS2016.sh): per frame pair the
                        four central crops -> PWC-Net 384x640 -> generator at the default 192x384; frames sharded over the ranks
`--impl reference` times the CPU restatement of the same graph (oracle/; TF 1.13 cannot be installed here) on the host cores.
`--dump-outputs DIR` writes what the last timed step returned to its caller as DIR/<name>.npy (train: losses, masks, flows, trained
weights; gen_fwd / ensemble: masks), rank 0's share under data parallelism: inputs and weights are seeded, so two builds run with the
same arguments can be compared output for output.
"""
import argparse
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

METRIC = 'frame-pairs/sec adversarial train step 256x448'
H, W, BPG = 256, 448, 4
WORKLOAD_TRAIN = 'DAVIS2016-shaped adversarial train 256x448, batch 4/GPU, PWC-Net 384x640 in loop, 1 rec : 3 gen (configs[1])'
GFLOP_PER_PAIR_STEP = 228.1    # SURVEY.md section 8(d): algorithmic conv FLOPs of one frame pair through one step, 1R:3G cycle average
DUMP_LIMIT = 64 << 20          # bytes of all --dump-outputs arrays together


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json'))), 'measured'
    except Exception:
        return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0}, 'fallback'


class ClockSampler(threading.Thread):
    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        while not self.stop_flag:
            try:
                o = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q, '--format=csv,noheader,nounits'],
                                   capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(',')])
            except Exception:
                pass
            time.sleep(0.02)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if r[1].isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[3:7]) if v.lower().startswith('active')})
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': reasons,
                'samples': len(self.rows)}


# ---------------------------------------------------------------------------------------------------- CPU reference arm
def pick_threads(probe):
    """torch-CPU oversubscribes badly on many-core hosts (128 threads: tens of seconds per step instead of ~1 s): time `probe` once
    per candidate thread count and keep the fastest -- that IS all the host threads this graph can use."""
    ncpu = os.cpu_count() or 1
    best = None
    for th in sorted({min(ncpu, c) for c in (8, 16, 32, 64)}):
        torch.set_num_threads(th)
        t0 = time.time()
        probe()
        dt = time.time() - t0
        if best is None or dt < best[0]:
            best = (dt, th)
    torch.set_num_threads(best[1])
    return best[1]


def cpu_reference(steps, warmup, batch=1, threads=None):
    """The reference graph restated on torch-CPU (oracle/; the genuine TF1.13 path is not installable here), all host
    threads it can use, identical step schedule (PWC-Net fwd @384x640 -> resize -> generator -> 3x recover -> losses -> backward ->
    clip -> TF-Adam), `batch` frame pair(s) per step.  Timed steps follow the 1R:3G schedule from step `warmup + 1` on."""
    from oracle import params as OP, losses as OL
    from unsupervised_detection_b200.data.synthetic import SyntheticReader
    p = OP.make_params(seed=8964)
    opt = OL.TFAdam()
    rd = SyntheticReader(384, 640, seed=8964)
    img1, img2, _, _ = rd.batch(batch, pinned=False)
    cfg = dict(batch_size=batch)
    if threads is None:
        threads = pick_threads(lambda: OL.train_step({k: v.clone() for k, v in p.items()}, OL.TFAdam(), 1, img1[:1], img2[:1], H, W,
                                                     dict(batch_size=1)))
    torch.set_num_threads(threads)
    times, kinds = [], []
    for s in range(1, warmup + steps + 1):
        t0 = time.time()
        r = OL.train_step(p, opt, s, img1, img2, H, W, cfg)
        if s > warmup:
            times.append(time.time() - t0)
            kinds.append(r['kind'][0].upper())
    tot = sum(times)
    return batch * len(times) / tot, threads, tot / len(times) * 1e3, ''.join(kinds)


def reference_steps(args, most):
    """The CPU arm takes seconds per step, so it times at most `most` steps; it says so on stderr when --steps asks for more."""
    if args.steps > most:
        print('bench.py: the reference arm times %d steps, not the %d asked for' % (most, args.steps), file=sys.stderr)
    return min(args.steps, most)


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    if args.workload != 'train':
        return run_reference_other(args)
    # same config as our arm at N = 1 (4 frame pairs per step, same 1R:3G schedule); bounded to <= 12 timed steps = three cycles
    steps, warmup = reference_steps(args, 12), min(max(args.warmup, 1), 1)
    v, threads, ms, kinds = cpu_reference(steps, warmup, batch=BPG)
    line = {'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': 'frame-pairs/s', 'n_gpus': args.gpus, 'steps': steps, 'warmup': warmup,
            'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': WORKLOAD_TRAIN, 'global_batch': BPG, 'parallelism': 'cpu',
                       'note': 'CPU restatement of the reference graph (TF1.13 not installable here), same batch and step schedule as the '
                               'GPU arm at N=1; timed step kinds: ' + kinds},
            'cpu_baseline': {'value': v, 'unit': 'frame-pairs/s', 'cores': threads, 'kind': 'port',
                             'sample': '%d steps x %d frame pairs (schedule from step %d: %s), thread count swept over {8,16,32,64}' %
                                       (steps, BPG, warmup + 1, kinds)},
            'e2e': {'value': v, 'unit': 'frame-pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}, 'gpu_launches': 0}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------- our arm
def conv_roofline(graph, reps=5):
    """Dominant kernel FAMILY = the tcgen05 implicit-GEMM convolutions (cis_conv_igemm forward / data gradient and cis_conv_wgrad):
    algorithmic FLOPs of every conv launch of one 1R:3G cycle / CUDA-event time of those launches replayed back to back on the
    launching stream.  Returns (FLOPs per step, ms per step, launches per step)."""
    CONV = ('cis_conv_igemm', 'cis_conv_wgrad')
    total_fl, total_ms, n = 0.0, 0.0, 0
    for plan, weight in ((graph.fwd, 4), (graph.bwd['R'], 1), (graph.bwd['G'], 3)):
        ops = [(fn, a) for fn, a, name, _, _ in plan.ops if name in CONV]
        fl = sum(f for _, _, name, f, _ in plan.ops if name in CONV)   # algorithmic 2*MACs on real channels
        # replayed through a CUDA graph (like the real step) so host launch cost does not enter the device time
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for fn, a in ops:
                fn(*a, side.cuda_stream)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            cs = torch.cuda.current_stream().cuda_stream
            for fn, a in ops:
                fn(*a, cs)
        gr.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            gr.replay()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        del gr
        total_fl += weight * fl
        total_ms += weight * ms
        n += weight * len(ops)
    return total_fl / 4, total_ms / 4, n / 4.0


def dominant_launch_roofline(graph, reps=20):
    """The single largest conv launch of the step (PWC-Net level-2 context conv dc_conv21, 3x3 565->128 at 96x160 x batch):
    algorithmic FLOPs / CUDA-event duration on the launching stream, L2 flushed (256 MB memset) before every timed launch."""
    st = torch.cuda.current_stream()
    ops = [(fn, a, f) for fn, a, name, f, _ in graph.fwd.ops if name == 'cis_conv_igemm']
    fn, a, fl = max(ops, key=lambda o: o[2])
    d = a[0]._obj
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=graph.dev)
    ms = []
    for i in range(reps + 3):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        fn(*a, st.cuda_stream)
        e1.record(st)
        torch.cuda.synchronize()
        if i >= 3:
            ms.append(e0.elapsed_time(e1))
    ms.sort()
    med = ms[len(ms) // 2]
    chunks = sum(d.src[i].chunks for i in range(d.nsrc))
    desc = 'cis::conv_halo_kernel<%d> 3x3 conv, %d->%d channels, %dx%dx%d pixels (MT=%d)' % (d.BN, chunks * 8, d.out_ch, d.N, d.OH, d.OW, d.MT)
    return fl, med, desc


def train_outputs(L):
    """What the last train step handed its caller, copied to the host: the four loss scalars (summed over the ranks, as
    AdversarialLearner.step reports them), this rank's masks, recovered flows and generator input flow, and the weights of both
    trained networks, each flattened in variable-name order.  Every rank must call it: the loss read is a collective under data
    parallelism.  The copies matter: any later step overwrites the graph's buffers in place."""
    g = L.graph
    g.pipeline_drain()
    torch.cuda.synchronize()
    ls = g.losses(reduce=L._allreduce())
    out = {'losses': torch.tensor([ls[k] for k in ('generator', 'recover', 'red_rate', 'red_rate_compl')], dtype=torch.float64),
           'masks': g.mask.cpu(), 'recovered_flows': g.pred.cpu(), 'flow': g.flow.cpu()}
    params = g.export_params()
    for net in ('MaskNet', 'FlownetS'):
        out['weights_' + net] = torch.cat([params[k].reshape(-1) for k in sorted(params) if k.startswith(net + '/')]).cpu()
    return out


def dump_outputs(out_dir, arrays):
    """arrays: name -> tensor, written as out_dir/<name>.npy in float64 (if it is float64) or float32."""
    arrays = {k: v.detach().to('cpu', torch.float64 if v.dtype == torch.float64 else torch.float32).numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise ValueError('--dump-outputs: %d bytes exceed the %d-byte limit' % (total, DUMP_LIMIT))
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + '.npy'), a)


def run_ours(args):
    import torch.distributed as dist
    from unsupervised_detection_b200.common_flags import Config
    from unsupervised_detection_b200.models.adversarial_learner import AdversarialLearner
    world = int(os.environ.get('WORLD_SIZE', '1'))
    cfg = Config(img_height=H, img_width=W, batch_size=BPG * world, dataset='SYNTHETIC', flow_ckpt='synthetic', summary_freq=10 ** 9)
    L = AdversarialLearner()
    L.config = cfg
    import contextlib
    with contextlib.redirect_stdout(sys.stderr):        # stdout carries exactly one JSON line
        L.build_train_graph()
    rank, dev = L.rank, L.device
    g = L.graph
    pool = [L.reader.batch(BPG) for _ in range(2)]
    K, Wm = args.steps, max(args.warmup, 3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(k):
            fn(i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    # ---- device-resident arm
    L.feed(pool[0][0], pool[0][1])
    cnt = [0]

    def dev_step(_):
        cnt[0] += 1
        g.train_step('R' if (cnt[0] % (cfg.iters_rec + cfg.iters_gen)) < cfg.iters_rec else 'G', allreduce=ar, use_graph=True, pipeline=PIPE)
    ar = L._allreduce()
    from unsupervised_detection_b200.models import adversarial_learner as AL
    PIPE = AL.PIPELINE          # cross-step software pipeline of the frozen flow network (CIS_PIPELINE=0 turns it off)
    for i in range(Wm):
        dev_step(i)
    smp = ClockSampler(L.local_rank)
    smp.start()
    ms_dev = timed(dev_step, K)
    # ---- end-to-end arm through the public API: pinned host batch -> H2D -> step -> D2H losses
    for i in range(Wm):
        L.step(pool[i % 2], fetch_losses=True, next_batch=pool[(i + 1) % 2])
    off = Wm % 2
    ms_e2e = timed(lambda i: L.step(pool[(i + off) % 2], fetch_losses=True, next_batch=pool[(i + off + 1) % 2]), K)
    smp.stop_flag = True
    smp.join(timeout=2)
    outputs = train_outputs(L) if args.dump_outputs else None     # copied before the per-kind timings below train further
    # each step kind on its own (SURVEY 8d asks for the 1R:3G cycle average AND the two kinds separately); single GPU only, after the
    # headline measurements, and never allowed to take them down
    by_kind = None
    if world == 1:
        try:
            by_kind = {}
            for mode in ('R', 'G'):
                for _ in range(3):
                    g.train_step(mode, allreduce=None, use_graph=True, pipeline=PIPE)
                by_kind['recover' if mode == 'R' else 'generator'] = timed(lambda i, m=mode: g.train_step(m, allreduce=None, use_graph=True, pipeline=PIPE), 8) / 8
        except Exception:
            by_kind = None
    gb = BPG * world
    value = gb * K / (ms_dev / 1e3)
    e2e = gb * K / (ms_e2e / 1e3)
    launches = sum(g.launches_per_step('R' if (i % 4) == 3 else 'G') for i in range(K))
    if rank != 0:
        return
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    pk, src = peaks()
    fl, ms_conv, nconv = conv_roofline(g)
    ach = fl / (ms_conv * 1e-3) / 1e12
    dfl, dms, ddesc = dominant_launch_roofline(g)
    dach = dfl / (dms * 1e-3) / 1e12
    traffic = None
    try:   # DRAM bytes of the best launch from the committed ncu --set full capture (profiles/r02_ncu_full_summary.json)
        prof = json.load(open(os.path.join(ROOT, 'profiles', 'r02_ncu_full_summary.json')))['prof_halo128_dominant'][-1]
        traffic = (float(prof['dram__bytes_read.sum'].split()[0]) + float(prof['dram__bytes_write.sum'].split()[0])) * 1e6
    except Exception:
        pass
    try:
        cv, cores, cms = cpu_reference(4, 0)[:3] if not args.no_cpu else (None, 0, 0)
    except Exception as e:  # the CPU leg must never take the GPU number down
        cv, cores, cms = None, 0, 0
    step_ms = ms_dev / K
    step_tflops = GFLOP_PER_PAIR_STEP * BPG / step_ms          # GFLOP / ms = TFLOP/s, per GPU
    line = {'metric': METRIC, 'value': value, 'unit': 'frame-pairs/s', 'n_gpus': world, 'steps': K, 'warmup': Wm, 'ms_per_step': step_ms,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
            'config': {'workload': WORKLOAD_TRAIN,
                       'global_batch': gb, 'parallelism': 'dp%d' % world, 'l2': 'per-step working set (activations) exceeds the 126 MB L2',
                       'cuda_graph': True, 'ms_per_step_by_kind': by_kind,
                       'flow_net_pipelined': bool(PIPE)},
            'e2e': {'value': e2e, 'unit': 'frame-pairs/s', 'h2d_bytes_per_step': 2 * BPG * 384 * 640 * 3 * 4, 'd2h_bytes_per_step': 32,
                    'ms_per_step': ms_e2e / K},
            'gpu_launches': launches,
            'clocks': smp.summary(),
            # the dominant kernel family BY TIME SHARE (every tcgen05 conv launch of the step), against the sustained measured peak
            'roofline': {'bound': 'tensor', 'kernel': 'tcgen05 implicit-GEMM conv family: cis::conv_halo_kernel / conv_igemm_kernel / '
                                                      'conv_wgrad_kernel, every launch of a 1R:3G cycle',
                         'achieved': ach, 'peak': pk['bf16_tflops_sustained'], 'unit': 'TFLOP/s', 'frac': ach / pk['bf16_tflops_sustained'],
                         'peak_source': src + ' bf16_tflops_sustained (family timed inside a long replay)', 'traffic': None,
                         'algorithmic_gflop_per_step': fl / 1e9, 'ms_per_step': ms_conv, 'launches_per_step': nconv,
                         'share_of_summed_kernel_time': 'see profiles/r02_per_op_gpu_times.txt (the step overlaps two streams, so shares of the wall-clock step are not additive)',
                         'whole_step': {'algorithmic_gflop_per_pair_step': GFLOP_PER_PAIR_STEP, 'achieved': step_tflops,
                                        'frac_of_sustained_peak': step_tflops / pk['bf16_tflops_sustained']},
                         'best_launch': {'kernel': ddesc, 'achieved': dach, 'peak': pk['bf16_tflops'], 'frac': dach / pk['bf16_tflops'],
                                         'peak_source': src + ' bf16_tflops (burst: launch timed alone, L2 flushed)',
                                         'algorithmic_gflop_per_launch': dfl / 1e9, 'us_per_launch': dms * 1e3, 'traffic': traffic}},
            'cpu_baseline': {'value': cv, 'unit': 'frame-pairs/s', 'cores': cores, 'kind': 'port',
                             'sample': 'one 1R:3G cycle (4 steps) x 1 frame pair of the same workload, %.0f ms/step, thread count swept' % cms}}
    print(json.dumps(line))
    sys.stdout.flush()


# ---------------------------------------------------------------------------------------------------- other BASELINE configs
GEN_H, GEN_W = 128, 224          # BASELINE.json configs[0]
ENS_H, ENS_W = 192, 384          # configs[4]: buffers are generated at the reference's default resolution (common_flags.py:6-8)


def _timed_events(fn, k, barrier):
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(k):
        fn(i)
    e1.record()
    barrier()
    return e0.elapsed_time(e1)


def _smooth_flow(B, Hh, Ww, gen):
    lo = torch.randn(B, 2, max(Hh // 16, 2), max(Ww // 16, 2), generator=gen)
    return (torch.nn.functional.interpolate(lo, size=(Hh, Ww), mode='bicubic', align_corners=False) * 0.3).permute(0, 2, 3, 1).contiguous()


def run_ours_other(args):
    import contextlib
    import torch.distributed as dist
    world, rank = int(os.environ.get('WORLD_SIZE', '1')), int(os.environ.get('RANK', '0'))
    K, Wm = args.steps, max(args.warmup, 3)
    pk, src = peaks()
    if args.workload == 'gen_fwd':
        # ---- configs[0]: one 128x224 frame pair, precomputed flow, mask-net forward only.  Does not shard: N > 1 = replicas.
        from unsupervised_detection_b200.step_graph import CISGraph
        from unsupervised_detection_b200 import params_init
        local = int(os.environ.get('LOCAL_RANK', '0'))
        torch.cuda.set_device(local)
        if world > 1 and not dist.is_initialized():
            dist.init_process_group('nccl', device_id=torch.device('cuda', local))
        g = CISGraph(GEN_H, GEN_W, 1, device='cuda:%d' % local, with_pwc=False, train=False)
        p = {}
        p.update(params_init.init_generator())
        p.update(params_init.init_recover())
        g.load_params(p)
        gen = torch.Generator().manual_seed(8964 + rank)
        image = (torch.rand(1, GEN_H, GEN_W, 3, generator=gen) - 0.5).pin_memory()
        flow = _smooth_flow(1, GEN_H, GEN_W, gen).pin_memory()
        mask_host = torch.empty(1, GEN_H, GEN_W, 1).pin_memory()

        def barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
        g.image.copy_(image)
        g.flow.copy_(flow)

        def dev_step(_):
            g.forward_masks(use_graph=True)

        def e2e_step(_):
            g.image.copy_(image, non_blocking=True)
            g.flow.copy_(flow, non_blocking=True)
            g.forward_masks(use_graph=True)
            mask_host.copy_(g.mask, non_blocking=True)
            torch.cuda.current_stream().synchronize()       # the caller reads the mask
        for i in range(Wm):
            dev_step(i)
            e2e_step(i)
        smp = ClockSampler(local)
        smp.start()
        ms_dev = _timed_events(dev_step, K, barrier)
        ms_e2e = _timed_events(e2e_step, K, barrier)
        smp.stop_flag = True
        smp.join(timeout=2)
        t = torch.tensor([ms_dev, ms_e2e], device='cuda')
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_dev, ms_e2e = float(t[0]), float(t[1])
        if rank != 0:
            return
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {'masks': mask_host})      # the mask the last timed step read back for its caller
        gflop = 8.437                                        # SURVEY App. B.1 at 128x224
        cv = cores = None
        if not args.no_cpu:
            cv, cores = cpu_gen_fwd(12)
        nl = g._mask_plan.count()
        line = {'metric': 'frame-pairs/sec mask-net forward 128x224 (BASELINE configs[0])', 'value': world * K / (ms_dev / 1e3),
                'unit': 'frame-pairs/s', 'n_gpus': world, 'steps': K, 'warmup': Wm, 'ms_per_step': ms_dev / K, 'higher_is_better': True,
                'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
                'config': {'workload': 'test_generator.py single frame pair 128x224, precomputed flow, mask-net forward only (configs[0])',
                           'global_batch': world, 'parallelism': 'replicas x%d (a single pair does not shard)' % world, 'cuda_graph': True,
                           'l2': 'working set fits L2 (latency-bound single-sample inference)'},
                'e2e': {'value': world * K / (ms_e2e / 1e3), 'unit': 'frame-pairs/s', 'h2d_bytes_per_step': GEN_H * GEN_W * 5 * 4,
                        'd2h_bytes_per_step': GEN_H * GEN_W * 4, 'ms_per_step': ms_e2e / K},
                'gpu_launches': nl * K, 'clocks': smp.summary(),
                'roofline': {'bound': 'tensor', 'kernel': 'tcgen05 conv family, generator forward (17 layers, batch 1)',
                             'achieved': gflop / (ms_dev / K), 'peak': pk['bf16_tflops_sustained'], 'unit': 'TFLOP/s',
                             'frac': gflop / (ms_dev / K) / pk['bf16_tflops_sustained'], 'peak_source': src, 'traffic': None},
                'cpu_baseline': {'value': cv, 'unit': 'frame-pairs/s', 'cores': cores, 'kind': 'port',
                                 'sample': 'median of 12 oracle generator forwards on the same input'}}
        print(json.dumps(line))
        return
    # ---- configs[4]: multi-crop ensemble inference through AdversarialLearner.inference(aug_test); frames sharded over the ranks
    from unsupervised_detection_b200.common_flags import Config
    from unsupervised_detection_b200.models.adversarial_learner import AdversarialLearner
    L = AdversarialLearner()
    with contextlib.redirect_stdout(sys.stderr):
        L.setup_inference(Config(img_height=ENS_H, img_width=ENS_W, batch_size=1, dataset='SYNTHETIC'), aug_test=True)
        L.restore('synthetic')
    g, rank, world = L.graph, L.rank, L.world
    pool = [L.reader.batch(1) for _ in range(2)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for i in range(Wm):
        L.inference(batch=pool[i % 2])
    smp = ClockSampler(L.local_rank)
    smp.start()
    ms_dev = _timed_events(lambda i: g.forward_masks(use_graph=True), K, barrier)       # crops already resident
    ms_e2e = _timed_events(lambda i: L.inference(batch=pool[i % 2]), K, barrier)        # H2D + device crops + forward + D2H masks/images
    smp.stop_flag = True
    smp.join(timeout=2)
    t = torch.tensor([ms_dev, ms_e2e], device=L.device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e = float(t[0]), float(t[1])
    if rank != 0:
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {'masks': g.mask})              # the last timed inference's pred_masks, one row per crop
    ncrop = len(L.test_crops)
    gflop = ncrop * 123.8                                    # SURVEY 8(d): PWC-Net + generator @192x384 per crop
    cv = cores = None
    if not args.no_cpu:
        cv, cores = cpu_ensemble(1)
    line = {'metric': 'frame-pairs/sec multi-crop ensemble inference 192x384 (BASELINE configs[4])', 'value': world * K / (ms_dev / 1e3),
            'unit': 'frame-pairs/s', 'n_gpus': world, 'steps': K, 'warmup': Wm, 'ms_per_step': ms_dev / K, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
            'config': {'workload': 'generate_buffer ensemble inference: 4 central crops per frame pair, PWC-Net 384x640 + generator 192x384 '
                                   '(configs[4])', 'global_batch': world, 'crops_per_frame': ncrop,
                       'parallelism': 'frames sharded over %d rank(s), no data-path collective' % world, 'cuda_graph': True,
                       'l2': 'per-step working set exceeds the 126 MB L2'},
            'e2e': {'value': world * K / (ms_e2e / 1e3), 'unit': 'frame-pairs/s', 'h2d_bytes_per_step': (2 * 3 + 1) * 384 * 640 * 4,
                    'd2h_bytes_per_step': ncrop * ENS_H * ENS_W * (1 + 1 + 3) * 4, 'ms_per_step': ms_e2e / K,
                    'note': 'one frame pair + ground truth uploaded per step; the 4 central crops and their resizes run on the device '
                            '(cis_crop_resize_bilinear_f32); masks, resized ground truth and the network input image are read back'},
            'gpu_launches': g._mask_plan.count() * K, 'clocks': smp.summary(),
            'roofline': {'bound': 'tensor', 'kernel': 'tcgen05 conv family, PWC-Net + generator forward, 4 crops', 'achieved': gflop / (ms_dev / K),
                         'peak': pk['bf16_tflops_sustained'], 'unit': 'TFLOP/s', 'frac': gflop / (ms_dev / K) / pk['bf16_tflops_sustained'],
                         'peak_source': src, 'traffic': None},
            'cpu_baseline': {'value': cv, 'unit': 'frame-pairs/s', 'cores': cores, 'kind': 'port',
                             'sample': '1 frame pair x 4 crops through the oracle (PWC-Net 384x640 + generator 192x384)'}}
    print(json.dumps(line))


def cpu_gen_fwd(reps):
    from oracle import params as OP, losses as OL, nets as ON
    p = OP.make_params(seed=8964, nets=('MaskNet',))
    gen = torch.Generator().manual_seed(8964)
    image = torch.rand(1, GEN_H, GEN_W, 3, generator=gen) - 0.5
    flow = OL.preprocess_flow_batch(_smooth_flow(1, GEN_H, GEN_W, gen))
    with torch.no_grad():
        th = pick_threads(lambda: ON.generator_net(image, flow, p))
        ts = []
        for _ in range(reps):
            t0 = time.time()
            ON.generator_net(image, flow, p)
            ts.append(time.time() - t0)
    ts.sort()
    return 1.0 / ts[len(ts) // 2], th


def cpu_ensemble(frames):
    from oracle import params as OP, losses as OL, nets as ON, pwcnet as OW
    from unsupervised_detection_b200.data.synthetic import SyntheticReader
    from unsupervised_detection_b200.data.crops import central_crops
    p = OP.make_params(seed=8964, nets=('MaskNet', 'pwcnet'))
    rd = SyntheticReader(384, 640, seed=8964)

    def one():
        a, b, gt, _ = rd.batch(1, pinned=False)
        i1, i2, _ = central_crops(a, b, gt, [0.85, 0.9, 0.95, 1.0])
        fo = OW.predict_from_img_pairs(i1, i2, p)
        im, fl = OL.resize_inputs(i1, fo, ENS_H, ENS_W)
        return ON.generator_net(im, OL.preprocess_flow_batch(fl), p)
    with torch.no_grad():
        th = pick_threads(one)
        t0 = time.time()
        for _ in range(frames):
            one()
    return frames / (time.time() - t0), th


def run_reference_other(args):
    if args.workload == 'gen_fwd':
        steps = reference_steps(args, 20)
        v, th = cpu_gen_fwd(steps)
        metric, wl = 'frame-pairs/sec mask-net forward 128x224 (BASELINE configs[0])', 'test_generator.py single frame pair 128x224, precomputed flow, mask-net forward only (configs[0])'
    else:
        steps = reference_steps(args, 3)
        v, th = cpu_ensemble(steps)
        metric, wl = 'frame-pairs/sec multi-crop ensemble inference 192x384 (BASELINE configs[4])', 'generate_buffer ensemble inference: 4 central crops per frame pair, PWC-Net 384x640 + generator 192x384 (configs[4])'
    print(json.dumps({'impl': 'reference', 'metric': metric, 'value': v, 'unit': 'frame-pairs/s', 'n_gpus': args.gpus, 'steps': steps, 'warmup': 1,
                      'ms_per_step': 1e3 / v, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
                      'config': {'workload': wl, 'global_batch': 1, 'parallelism': 'cpu'},
                      'cpu_baseline': {'value': v, 'unit': 'frame-pairs/s', 'cores': th, 'kind': 'port', 'sample': '%d frame pair(s)' % steps},
                      'e2e': {'value': v, 'unit': 'frame-pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}, 'gpu_launches': 0}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=4)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--workload', default='train', choices=['train', 'gen_fwd', 'ensemble'],
                    help='train = the headline metric; gen_fwd = BASELINE configs[0]; ensemble = BASELINE configs[4]')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the outputs of the last timed step as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs needs --impl ours')
    if args.impl == 'reference':
        run_reference(args)
    else:
        (run_ours if args.workload == 'train' else run_ours_other)(args)
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            dist.barrier()
            dist.destroy_process_group()


if __name__ == '__main__':
    main()
