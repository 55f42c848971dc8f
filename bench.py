#!/usr/bin/env python
"""bench.py -- headline benchmark of the CodeFormer hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes what the last timed step returned to its caller as DIR/<name>.npy (float32): out, logits and
lq_feat of CodeFormer.forward on one GPU, the gathered out on N GPUs.  Inputs and weights are seeded, so two builds of the
project run with the same arguments can be compared output for output.

A "step" = one CodeFormer.forward(x, w=0.5, adain=True) over one batch of 32 synthetic 512x512 faces per
GPU (BASELINE.json configs[1]; N GPUs = configs[4], 32 faces/GPU, weak scaling) followed -- for N>1 -- by
the one NCCL all-gather of `out` (SURVEY.md §8e).  Random-init weights of the reference architecture
(no checkpoints offline) and synthetic inputs; both stated in the JSON line.

Printed (rank 0, ONE line): metric/value/unit/... per the driver contract, plus
  e2e          same metric through the public nn.Module API with pinned HOST input -> H2D -> forward -> D2H of out
  roofline     dominant kernel (the 128->128 3x3 conv at 256^2, 13 of the 128 convs) timed alone with CUDA events
  cpu_baseline the oracle port timed on this box's host cores on a bounded sample (N=1 only)
  clocks       nvidia-smi samples taken during the timed region
`--impl reference` times the reference's CPU algorithm (oracle port; torch CPU fp32 = the reference's own math
backend) on the same config with all host threads, each step a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'faces_per_sec_512x512_batch32'
UNIT = 'faces/s'
GFLOP_PER_FACE = 809.77          # SURVEY.md §8(d): CodeFormer.forward, w>0, 4 connects
FALLBACK_PEAKS = {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0}   # B200_PROFILING.md


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return {k: float(d[k]) for k in FALLBACK_PEAKS}, 'measured'
        except Exception:
            pass
    return dict(FALLBACK_PEAKS), 'fallback'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '200', '-i', str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.25)
        self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.lines:
            f = [s.strip() for s in ln.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for nme, v in zip(names, f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(nme)
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': mx, 'reasons': sorted(reasons),
                'samples': len(sm)}


def synthetic_batch(batch, seed):
    import torch
    g = torch.Generator().manual_seed(seed)
    return torch.randn(batch, 3, 512, 512, generator=g).clamp_(-1, 1)     # SURVEY.md §8d config 5 inputs


def config_dict(n_gpus, batch):
    return {'workload': 'CodeFormer.forward(w=0.5, adain=True) on 512x512 aligned faces, batch 32 per GPU '
                        '(BASELINE.json configs[1]; N GPUs -> configs[4] weak scaling, one NCCL all-gather of out)',
            'batch_per_gpu': batch, 'global_batch': batch * n_gpus, 'w': 0.5, 'adain': True,
            'weights': 'random-init (seed 1) of the reference architecture, 94.1 M params fp32',
            'gflop_per_face': GFLOP_PER_FACE,
            'l2': 'timed iterations rotate over 2 input batches (201 MB > 126 MB L2); activations ~10 GB per step',
            'parallelism': f'dp{n_gpus}'}


def pick_cpu_threads():
    """Thread count for the reference CPU path.  torch CPU/oneDNN with one thread per *logical* CPU is pathological on the
    128-vCPU GPU boxes (measured: 65 s/face at 128 threads vs 2.0 s/face at 16, profiles/round1_cpu_threads.txt), so the
    baseline is given its best setting: a one-face probe of 16 and 32 threads (and os.cpu_count() when <= 32)."""
    import torch
    from codeformer_b200 import spec as S
    from oracle import codeformer_oracle as O
    n = os.cpu_count() or 1
    cands = sorted({min(16, n), min(32, n)} | ({n} if n <= 32 else set()))
    sd = S.random_state_dict(S.codeformer_spec(), 1)
    x = synthetic_batch(1, 7)
    best, best_t = cands[0], None
    with torch.no_grad():
        for c in cands:
            torch.set_num_threads(c)
            t = time.perf_counter()
            O.codeformer_forward(sd, x, w=0.5, adain_on=True)
            dt = time.perf_counter() - t
            if best_t is None or dt < best_t:
                best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def time_oracle(batch, passes, seed=0):
    """faces/s of the oracle port (torch CPU fp32 = the reference's own math backend) on the host cores."""
    import torch
    from codeformer_b200 import spec as S
    from oracle import codeformer_oracle as O
    threads = pick_cpu_threads()
    sd = S.random_state_dict(S.codeformer_spec(), 1)
    x = synthetic_batch(batch, seed)
    times = []
    with torch.no_grad():
        for _ in range(passes):
            t = time.perf_counter()
            O.codeformer_forward(sd, x, w=0.5, adain_on=True)
            times.append(time.perf_counter() - t)
    return times, threads


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port) on the host cores."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    batch = 1 if (args.steps + args.warmup) > 6 else 2      # bounded sample per step: whole run stays within minutes
    times, cores = time_oracle(batch, args.warmup + args.steps)
    timed = times[args.warmup:]
    total = sum(timed)
    value = batch * len(timed) / total
    line = {'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': 1e3 * total / len(timed), 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': dict(config_dict(args.gpus, 32), sample_batch=batch,
                           sample_note=f'the CPU arm times {batch} face(s) per step, not 32: a bounded sample of the batch-32 '
                                       'workload (its per-face time is best at small batch, BASELINE.md section 2, so the '
                                       'GPU/CPU ratio is conservative); it runs on ONE host whatever --gpus is'),
            'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                             'sample': f'{batch} face(s) per step (bounded sample of the batch-32 workload), '
                                       f'{len(timed)} timed steps, torch CPU fp32 oneDNN, best of 16/32 threads '
                                       f'of {os.cpu_count()} logical CPUs'},
            'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line), flush=True)


def committed_traffic():
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture (profiles/): never a
    constant in this file.  -> (bytes or None, source)."""
    for name in ('round2_dominant_kernel.json', 'round1_dominant_kernel.json'):
        path = os.path.join(ROOT, 'profiles', name)
        if os.path.exists(path):
            try:
                d = json.load(open(path))
                return float(d['dram_bytes_read']) + float(d['dram_bytes_write']), f'profiles/{name}: {d.get("source", "")}'
            except Exception:
                continue
    return None, 'no committed capture found under profiles/'


def time_conv_kernel(torch, N, H, Cin, Cout, xf, reps=20):
    """CUDA-event time of ONE tcgen05 conv kernel (cfb_debug_time_conv): 3x3, stride 1.  xf=True: the kernel the forward
    launches for a GroupNorm+SiLU consumer (fused operand transform on the fp32 activation, all-in)."""
    import ctypes
    from codeformer_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(3)
    x = torch.randn(N, H, H, Cin, generator=g).cuda()
    w = (torch.randn(Cout, Cin, 3, 3, generator=g) / (9 * Cin) ** 0.5).cuda()
    out = torch.empty(N, H, H, Cout, device='cuda')
    sc = (1 + 0.1 * torch.randn(N, Cin, generator=g)).cuda() if xf else None
    sh = (0.1 * torch.randn(N, Cin, generator=g)).cuda() if xf else None
    wsb = lib.cfb_conv2d_workspace_bytes(N, H, H, Cin, Cout, 3, 0)
    ws = torch.empty(int(wsb), dtype=torch.uint8, device='cuda')
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    ms = ctypes.c_float(0)
    _lib.check(lib.cfb_debug_time_conv(_lib.ptr(x), _lib.ptr(w), _lib.ptr(out), N, H, H, Cin, Cout, 3, 0, reps, _lib.ptr(ws), wsb, st,
                                       _lib.ptr(sc), _lib.ptr(sh), 1 if xf else 0, ctypes.byref(ms)), 'cfb_debug_time_conv')
    return float(ms.value)


def dominant_kernel_roofline(torch, cb, batch, peaks, peak_kind):
    """The dominant kernel = conv_tc_kernel on the most frequent shape (ResBlock conv 128->128 3x3 at 256^2: 13 launches of
    19.33 GFLOP/face, SURVEY Appendix A), in the variant the forward launches there: GroupNorm+SiLU applied to the fp32
    activation inside the kernel (fused operand transform), split weights prepared at load time.  Timed alone with CUDA
    events on the launching stream, B=8 like the committed ncu capture.  Also reported: the same shape on raw operand planes
    and the 64->64 @512^2 layer (the worst conv family of round 1)."""
    N, H, C = 8, 256, 128
    ms = time_conv_kernel(torch, N, H, C, C, True)
    ms_raw = time_conv_kernel(torch, N, H, C, C, False)
    ms64 = time_conv_kernel(torch, N, 512, 64, 64, True)
    flops = 2.0 * N * H * H * C * C * 9
    achieved = flops / (ms * 1e-3) / 1e12
    traffic, tsrc = committed_traffic()
    return {'bound': 'tensor', 'kernel': 'conv_tc_kernel<128,halo,pair,xform>: GroupNorm+SiLU+conv 3x3 128->128 @256^2, B=8 (kernel only, all-in)',
            'achieved': achieved, 'peak': peaks['bf16_tflops'], 'unit': 'TFLOP/s', 'frac': achieved / peaks['bf16_tflops'],
            'peak_kind': f'{peak_kind} bf16 burst (MEASURED_PEAKS.json)', 'ms_per_launch': ms,
            'algorithmic_gflop_per_launch': flops / 1e9,
            'executed_mma_passes': '2 tcgen05.mma.cta_group::2 (M=256) per k-step (N=256 + N=128) = 3x the nominal MACs (split-fp16 '
                                   'operands): the 3-pass ceiling of this frac is 1/3',
            'traffic': traffic, 'traffic_unit': 'bytes/launch',
            'traffic_source': 'dram__bytes_read.sum + dram__bytes_write.sum of ' + tsrc +
                              ' (ncu --set full, same shape and batch); algorithmic = 268 MB fp32 input + 268 MB fp32 output',
            'other_kernels': {
                'conv 3x3 128->128 @256^2 B=8 on raw fp16 operand planes (no transform)': {
                    'ms_per_launch': ms_raw, 'frac': flops / (ms_raw * 1e-3) / 1e12 / peaks['bf16_tflops']},
                'GroupNorm+SiLU+conv 3x3 64->64 @512^2 B=8 (fused transform, all-in; same FLOPs)': {
                    'ms_per_launch': ms64, 'frac': flops / (ms64 * 1e-3) / 1e12 / peaks['bf16_tflops']}}}


DUMP_BUDGET = 64 * 10**6        # bytes of all .npy files of one --dump-outputs
DUMP_RESERVE = 16 * 10**6       # kept for each array not yet written
NPY_HEADER = 128                # np.save header of a 1-D or 3-D float32 array


def dump_outputs(torch, arrays, out_dir, seed=0):
    """Write each tensor of `arrays` (name -> tensor) as out_dir/<name>.npy in float32, within DUMP_BUDGET bytes in all.
    Smallest first, an array is written whole, in its own shape, while that leaves DUMP_RESERVE bytes for each array still
    to come; an array that does not fit is written as a fixed sample of its flattened elements: the sorted positions
    np.random.default_rng(seed).choice(numel, n, replace=False), n filling its share of the budget that is left.
    -> {name: {'shape', 'elements', 'sample_seed'}} (sample_seed None: the whole array)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    items = sorted(arrays.items(), key=lambda kv: kv[1].numel())
    left, info = DUMP_BUDGET, {}
    for k, (name, t) in enumerate(items):
        rest = len(items) - 1 - k
        flat = t.detach().reshape(-1)
        if NPY_HEADER + 4 * flat.numel() <= left - rest * DUMP_RESERVE:
            a, sample_seed = t.detach().float().cpu().numpy(), None
        else:
            n = (left // (rest + 1) - NPY_HEADER) // 4
            at = np.sort(np.random.default_rng(seed).choice(flat.numel(), n, replace=False))
            a, sample_seed = flat[torch.from_numpy(at).to(flat.device)].float().cpu().numpy(), seed
        path = os.path.join(out_dir, name + '.npy')
        np.save(path, a)
        left -= os.path.getsize(path)
        info[name] = {'shape': list(t.shape), 'elements': int(a.size), 'sample_seed': sample_seed}
    return info


def _median_ms(torch, fn, iters, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2]


def extra_configs(torch, cb, S, net, peaks, dev):
    """The other single-GPU configurations of BASELINE.json, measured AFTER the headline so they cannot perturb it:
    configs[0] single-face latency on the GPU, configs[2] VectorQuantizer microbench (HBM roofline on 17.9 MB),
    configs[3] VQAutoEncoder.forward at batch 64."""
    out = {}
    x1 = synthetic_batch(1, 5).to(dev)
    out['latency_b1_ms'] = {'value': _median_ms(torch, lambda: net(x1, w=0.5, adain=True), 30), 'unit': 'ms',
                            'what': 'BASELINE configs[0] on the GPU: one 512x512 face, CodeFormer.forward(w=0.5, adain=True) through '
                                    'the public module API (CUDA-graph replay), median of 30, input resident on the device'}
    g = torch.Generator().manual_seed(0)
    E = torch.randn(1024, 256, generator=g)
    z = torch.randn(32, 256, 16, 16, generator=g).to(dev)
    vq = cb.VectorQuantizer(1024, 256, 0.25)
    vq.embedding.weight.data.copy_(E)
    vq = vq.to(dev)
    ms = _median_ms(torch, lambda: vq(z, return_min_encodings=False), 50)

    def burst():                       # 20 calls back to back: the launches pipeline, the GPU time per call remains
        for _ in range(20):
            vq(z, return_min_encodings=False)
    ms_pipe = _median_ms(torch, burst, 10) / 20
    nbytes = 17.9e6            # SURVEY section 8(d) config 3: z 8.39 + E 1.05 + z_q 8.39 + idx 0.07 MB
    out['vq_micro'] = {'ms': ms, 'ms_pipelined': ms_pipe, 'launches_per_call': 1,
                       'vectors_per_s': 8192 / (ms_pipe * 1e-3), 'algorithmic_bytes': nbytes,
                       'roofline': {'bound': 'hbm', 'achieved': nbytes / (ms_pipe * 1e-3) / 1e9, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
                                    'frac': nbytes / (ms_pipe * 1e-3) / 1e9 / peaks['hbm_gbs'], 'of': 'ms_pipelined'},
                       'what': 'BASELINE configs[2]: VectorQuantizer.forward (one kernel), z [32,256,16,16] vs 1024 codes, NCHW in / NCHW '
                               'out; ms = one call from a cold queue incl. the host side of the module call (median of 50), '
                               'ms_pipelined = per call of 20 back-to-back calls (indices bit-exact vs the reference golden in '
                               'tests/test_gpu_kernels.py)'}
    del vq, z
    vqae = cb.VQAutoEncoder(512, 64, [1, 2, 2, 4, 4, 8], 'nearest', 2, [16], 1024).to(dev).eval()
    vqae.load_state_dict(S.random_state_dict(S.vqae_spec(), 2), strict=True)
    x64 = synthetic_batch(64, 9).to(dev)
    ms = _median_ms(torch, lambda: vqae(x64, return_min_encodings=False), 3, warm=2)
    out['vqae_b64'] = {'faces_per_s': 64 / (ms * 1e-3), 'ms_per_step': ms, 'gflop_per_face': 580.59,
                       'step_algorithmic_tflops': 64 / (ms * 1e-3) * 580.59 / 1e3,
                       'what': 'BASELINE configs[3]: VQAutoEncoder(512,64,[1,2,2,4,4,8]).forward at batch 64, median of 3'}
    del vqae, x64
    torch.cuda.empty_cache()
    # ---- SURVEY section 8 rows f3 / f4: the caller-side networks on the same engine (random-init weights of the reference
    # architectures, synthetic inputs; parity vs the reference goldens is in tests/test_gpu_aux.py)
    from codeformer_b200 import parsing as P
    pn = cb.ParseNet(in_size=512, out_size=512, parsing_ch=19)
    pn.load_state_dict(P.random_parsenet_state_dict(P.parsenet_spec(512, 512, 32, 64, 19, 10, (32, 256)), 41), strict=True)
    pn = pn.eval().to(dev)
    xf = synthetic_batch(8, 13).to(dev)
    ms = _median_ms(torch, lambda: cb.face_parse_mask(pn(xf, return_img=False)[0]), 5, warm=2)
    out['parsenet_b8'] = {'faces_per_s': 8 / (ms * 1e-3), 'ms_per_step': ms,
                          'what': 'row f3: ParseNet(512,512,parsing_ch=19).forward + argmax/MASK_COLORMAP on 8 restored faces '
                                  '(facelib/utils/face_restoration_helper.py:457-468), median of 5'}
    del pn, xf
    rr = cb.RRDBNet(3, 3, scale=2, num_feat=64, num_block=23, num_grow_ch=32)
    rr.load_state_dict(S.random_state_dict(S.rrdbnet_spec(3, 3, 2, 64, 23, 32), 21), strict=True)
    rr = rr.eval().to(dev)
    xt = torch.rand(1, 3, 480, 480, generator=torch.Generator().manual_seed(4)).to(dev)
    ms = _median_ms(torch, lambda: rr(xt), 5, warm=2)
    gflop = 57600 * 35.8e-3          # 240x240 feature pixels x 35.8 MFLOP (69 dense blocks + body/up/hr convs)
    out['rrdbnet_tile'] = {'ms_per_tile': ms, 'input_mpix_per_s': 0.2304 / (ms * 1e-3), 'algorithmic_tflops': gflop / ms,
                           'what': 'row f4: RRDBNet(3,3,scale=2, 23 blocks) on one 480x480 tile = RealESRGANer tile 400 + 2x40 pad '
                                   '(inference_codeformer.py:36-61), output 960x960, median of 5; ~2.06 TFLOP nominal per tile'}
    del rr, xt
    torch.cuda.empty_cache()
    return out


def run_b200(args):
    import torch
    import torch.distributed as dist
    import codeformer_b200 as cb
    from codeformer_b200 import spec as S

    torch.set_grad_enabled(False)
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if args.gpus > 1 and world != args.gpus:
        raise SystemExit(f'--gpus {args.gpus} needs torchrun with {args.gpus} ranks (WORLD_SIZE={world})')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    batch = args.batch
    net = cb.ARCH_REGISTRY.get('CodeFormer')(dim_embd=512, codebook_size=1024, n_head=8, n_layers=9,
                                            connect_list=['32', '64', '128', '256']).to(dev).eval()
    net.load_state_dict(S.random_state_dict(S.codeformer_spec(), 1), strict=True)
    xs_host = [synthetic_batch(batch, 100 + rank * 2 + i).pin_memory() for i in range(2)]
    xs = [x.to(dev) for x in xs_host]
    gathered = torch.empty((world * batch, 3, 512, 512), device=dev) if world > 1 else None
    from codeformer_b200.parallel import StreamedGather, pipelined_forward_gather
    sg = StreamedGather() if world > 1 else None

    def step(i):
        """-> the arrays the caller of the path receives (name -> tensor); on N GPUs the gathered `out`, which the
        asynchronous gather delivers only at the next submit / flush."""
        out, logits, lq_feat = net(xs[i % 2], w=0.5, adain=True)
        if world > 1:
            # the one collective of the path (section 8e), off the critical path: issued asynchronously after the forward, it
            # completes on NCCL's stream while the next step's forward runs (parallel.StreamedGather); the timed region ends
            # with flush(), so every gather is inside it.  --gather-chunks 2 selects the half-batch pipeline instead.
            if args.gather_chunks > 1:
                return {'out': pipelined_forward_gather(net, xs[i % 2], gathered, chunks=args.gather_chunks, w=0.5, adain=True)[0]}
            sg.submit(out)
            return {}
        return {'out': out, 'logits': logits, 'lq_feat': lq_feat}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(max(args.warmup, 3)):
        step(i)
    if sg is not None:
        sg.flush()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        last = None                                          # a step's outputs are released before the next step runs
        last = step(i)
    if sg is not None:
        done = sg.flush()                                    # the last gather completes inside the timed region
        if done is not None:
            last = {'out': done}
    e1.record()
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    launches = net.last_launch_count * args.steps
    clocks = sampler.stop() if sampler else None
    ms_total = float(ms.item())
    value = world * batch * args.steps / (ms_total * 1e-3)
    dumped = dump_outputs(torch, last, args.dump_outputs) if args.dump_outputs and rank == 0 else None
    del last

    # ---- multi-GPU evidence (section 8d config 5): the gathered tensor holds every rank's shard bit for bit, and where the
    # step time goes on each rank (forward alone, gather alone; CUDA events)
    multi = None
    if world > 1:
        local = net(xs[0], w=0.5, adain=True)[0]
        sg.submit(local)
        gathered = sg.flush()
        torch.cuda.synchronize()
        same = torch.tensor([1 if torch.equal(gathered[rank * batch:(rank + 1) * batch], local) else 0], device=dev)
        # every rank also checks the shard of its right neighbour against that rank's own result (sent as a checksum)
        chk = torch.stack([gathered[r * batch:(r + 1) * batch].double().sum() for r in range(world)])
        mine = local.double().sum().reshape(1)
        allsum = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allsum, mine)
        same2 = torch.tensor([1 if all(float(chk[r]) == float(allsum[r]) for r in range(world)) else 0], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        dist.all_reduce(same2, op=dist.ReduceOp.MIN)
        fe0, fe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        fe0.record()
        for i in range(3):
            o_loc = net(xs[i % 2], w=0.5, adain=True)[0]
        fe1.record()
        torch.cuda.synchronize()
        fwd_ms = fe0.elapsed_time(fe1) / 3
        barrier()
        fe0.record()
        for i in range(3):
            dist.all_gather_into_tensor(gathered, o_loc)
        fe1.record()
        torch.cuda.synchronize()
        gat_ms = fe0.elapsed_time(fe1) / 3
        t = torch.tensor([fwd_ms, gat_ms], device=dev)
        tmax, tmin = t.clone(), t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        multi = {'gather_bit_identical': bool(int(same.item()) == 1 and int(same2.item()) == 1),
                 'forward_only_ms_per_rank_min_max': [float(tmin[0]), float(tmax[0])],
                 'blocking_gather_only_ms_min_max': [float(tmin[1]), float(tmax[1])],
                 'gather_bytes_per_rank': batch * 3 * 512 * 512 * 4, 'gather_chunks': args.gather_chunks,
                 'note': 'timed steps issue the all-gather asynchronously: gather i overlaps forward i+1 (flush inside the timed '
                         'region); measured on 2 GPUs: blocking gather 0.33 ms, two 16-face half-forwards cost +3.4 ms over one '
                         '32-face forward, so the half-batch pipeline is not the default; the step is max over ranks, each GPU '
                         'under its own power-capped clock (forward-only spread above)'}

    # ---- e2e: public API with host buffers, H2D + D2H inside the timed region
    out_host = torch.empty((batch, 3, 512, 512), dtype=torch.float32, pin_memory=True)

    def step_e2e(i):
        x = xs_host[i % 2].to(dev, non_blocking=True)
        out = net(x, w=0.5, adain=True)[0]
        if world > 1:
            dist.all_gather_into_tensor(gathered, out)           # e2e: the caller reads THIS step's collated result
        out_host.copy_(out, non_blocking=True)
        torch.cuda.current_stream().synchronize()               # the caller reads the result (tensor2img .cpu())
    e_steps = max(2, min(args.steps, 5))
    step_e2e(0)
    barrier()
    e0.record()
    for i in range(e_steps):
        step_e2e(i)
    e1.record()
    barrier()
    ms2 = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    e2e_value = world * batch * e_steps / (float(ms2.item()) * 1e-3)
    img_bytes = batch * 3 * 512 * 512 * 4

    # ---- e2e through the caller-loop front-end (SURVEY section 8 f1/f2): uint8 BGR faces in, uint8 restored faces out
    e2e_u8 = None
    if world == 1:
        import numpy as np
        faces = np.random.default_rng(0).integers(0, 256, (batch, 512, 512, 3), dtype=np.uint8)
        net.restore_faces(faces, w=0.5, adain=True, max_batch=batch, on_error='raise')
        torch.cuda.synchronize()
        e0.record()
        for i in range(e_steps):
            net.restore_faces(faces, w=0.5, adain=True, max_batch=batch, on_error='raise')
        e1.record()
        torch.cuda.synchronize()
        e2e_u8 = {'value': batch * e_steps / (e0.elapsed_time(e1) * 1e-3), 'unit': UNIT, 'api': 'CodeFormer.restore_faces',
                  'h2d_bytes_per_step': batch * 3 * 512 * 512, 'd2h_bytes_per_step': batch * 3 * 512 * 512, 'steps': e_steps}

    if rank == 0:
        peaks, peak_kind = load_peaks()
        roof = dominant_kernel_roofline(torch, cb, batch, peaks, peak_kind)
        step_tflops = value / world * GFLOP_PER_FACE / 1e3
        roof['step_algorithmic_tflops_per_gpu'] = step_tflops
        roof['step_frac_of_sustained_peak'] = step_tflops / peaks['bf16_tflops_sustained']
        line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
                'warmup': max(args.warmup, 3), 'ms_per_step': ms_total / args.steps, 'higher_is_better': True,
                'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32 (split-fp16 operands on tensor cores, fp32 accumulate)',
                'data': 'synthetic', 'config': config_dict(world, batch),
                'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': img_bytes, 'd2h_bytes_per_step': img_bytes,
                        'steps': e_steps},
                'gpu_launches': int(launches), 'clocks': clocks, 'roofline': roof}
        if e2e_u8:
            line['e2e_u8'] = e2e_u8
        if dumped:
            line['dump_outputs'] = {'dir': args.dump_outputs, 'arrays': dumped}
        if multi:
            line['multi_gpu'] = multi
            line['gather_bit_identical'] = multi['gather_bit_identical']
        if world == 1 and not args.no_extras:
            line.update(extra_configs(torch, cb, S, net, peaks, dev))
        if world == 1 and not args.no_cpu_baseline:
            times, cores = time_oracle(2, 3)
            best = min(times[1:])
            line['cpu_baseline'] = {'value': 2 / best, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                                    'sample': '2 faces per pass (bounded sample of the batch-32 workload), best of 2 after '
                                              f'1 warm-up, torch CPU fp32 oneDNN, best of 16/32 threads of {os.cpu_count()} logical CPUs'}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--batch', type=int, default=32, help='faces per GPU (the metric is quoted at 32)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extras', action='store_true', help='skip BASELINE configs 1/3/4 (latency, VQ microbench, VQAE B=64)')
    ap.add_argument('--gather-chunks', type=int, default=1,
                    help='N>1: 1 = asynchronous gather overlapping the next step (default); >1 = half-batch pipeline inside a step')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the outputs of the last timed step as DIR/<name>.npy (float32, at most 64 MB in all)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the b200 path only')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
