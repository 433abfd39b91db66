"""bench.py -- frames/sec of the Cutie per-frame path on B200 (BASELINE.json metric), with the roofline of the
dominant kernel and the reference's CPU path timed beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2|northstar]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config.workload = "cfg2", BASELINE.json configs[1]): synthetic 480p (854x480 -> 864x480 padded, 30x54 = 1620
tokens/frame) video, 3 objects, 256-frame working memory (max_mem_frames=256, use_long_term=False, mem_every=5,
top_k=30): a steady-state bank of 413 100 tokens, pre-filled with seeded N(0,1) keys/values and 1+N(0,1)^2 shrinkage
(SURVEY.md section 8(d)); random-init weights of the cutie-base architecture (cutie_b200/utils/synth.py).  A *step* is
one InferenceCore.step on one frame through the reference's own call signature (no extension arguments); every 5th step
is a memory frame (mask encoder + append + FIFO eviction).  N>1: one independent video stream per GPU (weak scaling, no
data-path collective -- SURVEY.md section 8(e).1); after the stream benchmark the N ranks also run the key-sharded
memory read of BASELINE.json configs[4] (`sharded_read`, SURVEY.md section 8(e).2).

Numerics of the timed region = numerics of the parity tests: fp32, cuDNN / cuBLAS TF32 OFF (`amp=False`); every
optional launch form is chosen by a committed table (cutie_b200/utils/dispatch.py, model/fuse.py), nothing is timed to
choose an arithmetic.  After the timed region one frame is re-computed by the CPU oracle from the live state
(`parity_check`).

One JSON line on stdout (rank 0); everything else goes to stderr.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# Exactly ONE line may reach stdout (the JSON).  Libraries (NCCL prints its version banner) write to fd 1 directly, so
# fd 1 is pointed at stderr for the whole run and the JSON goes to a saved copy of the real stdout.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line: dict):
    os.write(_REAL_STDOUT, (json.dumps(line) + '\n').encode())


WORKLOADS = {
    # name: (H, W, objects, memory frames, top_k)
    'cfg2': dict(H=480, W=854, K=3, mem_frames=256, top_k=30,
                 desc='synthetic 480p video, 3 objects, 256-frame working memory (414720 tokens), 1xB200'),
    'northstar': dict(H=480, W=854, K=3, mem_frames=6, top_k=30,
                      desc='synthetic 480p video, 3 objects, ~10k-key working memory (9720 tokens)'),
}
METRIC = 'frames/sec @480p 3-obj'


def usable_cpus() -> int:
    """Host threads this process can actually run: the affinity mask, capped by the cgroup CPU quota if there is one
    (os.cpu_count() reports the machine, not the container; oversubscribing a quota-limited container makes the CPU arm
    slower, which would flatter the GPU arm)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    try:
        quota, period = open('/sys/fs/cgroup/cpu.max').read().split()[:2]
        if quota != 'max':
            n = min(n, max(1, -(-int(quota) // int(period))))
    except Exception:
        try:
            q = int(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read())
            p_ = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
            if q > 0:
                n = min(n, max(1, -(-q // p_)))
        except Exception:
            pass
    return max(1, n)


def make_cfg(wl):
    from cutie_b200.config import default_config
    return default_config(mem_every=5, max_mem_frames=wl['mem_frames'], use_long_term=False, top_k=wl['top_k'])


def make_net(cfg):
    from cutie_b200.model.cutie import CUTIE
    from cutie_b200.utils.synth import synthetic_state_dict      # synthetic weights (data generation, no oracle code)
    net = CUTIE(cfg).eval()
    net.load_state_dict(synthetic_state_dict(net.state_dict(), 0))
    return net


def tokens_per_frame(wl) -> int:
    return (wl['H'] // 16) * (-(-wl['W'] // 16))


def synthetic_bank_chunks(wl, chunk_frames=16, seed=1234):
    """Yields (key [1,64,n], shrinkage [1,1,n], values [1,K,256,n]) CPU chunks of the steady-state bank."""
    HW = tokens_per_frame(wl)
    total = (wl['mem_frames'] - 2) * HW          # perm frame + this many temp frames = one short of the FIFO limit
    g = torch.Generator().manual_seed(seed)
    done = 0
    while done < total:
        n = min(chunk_frames * HW, total - done)
        yield (torch.randn(1, 64, n, generator=g), 1 + torch.randn(1, 1, n, generator=g) ** 2,
               torch.randn(1, wl['K'], 256, n, generator=g))
        done += n


def base_config(args, wl, world):
    """The `config` object: identical for both arms (--impl ours / reference) so the driver can compare them."""
    HW = tokens_per_frame(wl)
    return {'workload': f"{args.workload}: {wl['desc']}", 'resolution': [wl['H'], wl['W']], 'objects': wl['K'],
            'tokens_per_frame': HW, 'memory_tokens': (wl['mem_frames'] - 1) * HW, 'top_k': wl['top_k'], 'mem_every': 5,
            'streams': world, 'parallelism': f'{world} independent streams (1 per GPU)',
            'l2': 'no flush: the bank scanned every frame is larger than the 126 MB L2'
                  if args.workload == 'cfg2' else 'bank fits L2 (north-star size); stated, not flushed',
            'weights': 'seeded random init (no checkpoint offline)', 'precision': 'fp32, TF32 off (amp=False)'}


# ---------------------------------------------------------------------------------------------------
# clocks
def _nvml_handle(idx):
    """NVML handle of torch device `idx` (honours CUDA_VISIBLE_DEVICES through the device's UUID), or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(idx).uuid)
        for cand in (f'GPU-{uuid}', uuid):
            try:
                return pynvml, pynvml.nvmlDeviceGetHandleByUUID(cand.encode())
            except Exception:
                pass
        return pynvml, pynvml.nvmlDeviceGetHandleByIndex(idx)
    except Exception:
        return None


def nvsmi_sampler(stop, out, idx):
    """Samples SM clock, power and throttle reasons DURING the timed region: NVML in-process every ~5 ms, `nvidia-smi`
    every 0.2 s if NVML is unavailable.  Rows: [sm_mhz, sm_max_mhz, power_w, hw_slowdown, hw_thermal_slowdown,
    sw_thermal_slowdown, sw_power_cap]."""
    nv = _nvml_handle(idx)
    if nv is not None:
        pynvml, h = nv
        try:
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            bits = (('hw_slowdown', pynvml.nvmlClocksThrottleReasonHwSlowdown),
                    ('hw_thermal_slowdown', pynvml.nvmlClocksThrottleReasonHwThermalSlowdown),
                    ('sw_thermal_slowdown', pynvml.nvmlClocksThrottleReasonSwThermalSlowdown),
                    ('sw_power_cap', pynvml.nvmlClocksThrottleReasonSwPowerCap))
            while not stop.is_set():
                sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                pw = pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0
                r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                out.append([str(sm), str(mx), f'{pw:.2f}'] + ['Active' if r & b else 'Not Active' for _, b in bits])
                stop.wait(0.005)
            return
        except Exception as e:                       # noqa: BLE001 -- fall through to nvidia-smi
            log(f'[clocks] NVML sampling failed ({type(e).__name__}: {e}); using nvidia-smi')
    q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
    while not stop.is_set():
        try:
            r = subprocess.run(['nvidia-smi', f'--id={idx}', f'--query-gpu={q}', '--format=csv,noheader,nounits'],
                               capture_output=True, text=True, timeout=5)
            if r.returncode == 0 and r.stdout.strip():
                out.append([x.strip() for x in r.stdout.strip().split('\n')[0].split(',')])
        except Exception:
            pass
        stop.wait(0.2)


def summarize_clocks(samples):
    if not samples:
        return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
    sm = [float(s[0]) for s in samples if s[0].replace('.', '').isdigit()]
    reasons = set()
    for s in samples:
        for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), s[3:7]):
            if v.lower().startswith('active'):
                reasons.add(name)
    return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': float(samples[0][1]),
            'power_w_max': max(float(s[2]) for s in samples), 'reasons': sorted(reasons), 'samples': len(samples)}


def percentiles(ms):
    s = sorted(ms)
    pick = lambda q: s[min(len(s) - 1, int(q * len(s)))]
    return {'frames': len(s), 'mean': sum(s) / len(s), 'p50': pick(0.50), 'p90': pick(0.90), 'p99': pick(0.99), 'max': s[-1]}


# ---------------------------------------------------------------------------------------------------
def run_ours(args, wl, rank, world, dev):
    import cutie_b200.kernels as K_
    from cutie_b200.inference.inference_core import InferenceCore
    from cutie_b200.utils.synth import synthetic_video
    K_.lib()                                             # fail loudly if the CUDA library is missing
    torch.backends.cudnn.allow_tf32 = False              # the validated configuration: fp32 convolutions (amp=False)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = not args.no_cudnn_benchmark
    cfg = make_cfg(wl)
    net = make_net(cfg).to(dev)
    if not args.no_optimize:
        # BN folding + channels-last trunks + conv/bias/ReLU epilogues in the form the committed rule names
        net.optimize_for_inference()
    use_graphs = not args.no_graphs
    warm = max(args.warmup, 11) if use_graphs else args.warmup       # every CUDA-graph variant exists after 11 steps
    K = args.steps
    n_frames = warm + 4 * K + 16
    frames, mask = synthetic_video(n_frames, wl['H'], wl['W'], wl['K'], seed=rank)
    objs = list(range(1, wl['K'] + 1))
    proc = InferenceCore(net, cfg=cfg, use_cuda_graphs=use_graphs)
    with torch.inference_mode():
        proc.step(frames[0].to(dev), mask.to(dev), objects=objs)          # permanent first frame
        for key, shr, vals in synthetic_bank_chunks(wl):                   # steady-state bank
            proc.memory.work_mem.add(key.to(dev), {o: vals[:, i].to(dev) for i, o in enumerate(objs)},
                                     shr.to(dev), None, as_permanent='no')
    n_tokens = proc.memory.work_mem.size(0)
    log(f'[rank {rank}] bank prefilled: {n_tokens} tokens, {torch.cuda.memory_allocated(dev) / 2**30:.2f} GiB allocated')
    frames_dev = frames.to(dev)
    frames_pin = frames.pin_memory()
    host_out = torch.empty(wl['H'], wl['W'], dtype=torch.uint8).pin_memory()

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize(dev)

    state = {'t': 1}
    res = {}

    def device_arm(steps, lookahead, profile, keep_last=False):
        """`steps` frames with inputs resident in HBM; returns (per-step event marks, host enqueue ms/step).  keep_last:
        a copy of the last step's output (taken after the last mark) goes to res['outputs']."""
        t = state['t']
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        if profile:
            K_.PROFILE = []
        marks[0].record()
        h0 = time.perf_counter()
        for j in range(steps):
            if lookahead:
                prob = proc.step(frames_dev[t], next_image=frames_dev[t + 1] if j + 1 < steps else None)
            else:
                prob = proc.step(frames_dev[t])
            marks[j + 1].record()
            t += 1
        host_ms = (time.perf_counter() - h0) * 1e3 / steps
        state['t'] = t
        if keep_last:
            res['outputs'] = {'prob': prob.clone()}       # a CUDA-graph replay returns a buffer the next step overwrites
        return marks, host_ms

    def e2e_arm(steps, lookahead):
        """Pinned host frame in, uint8 mask on the host out, copies inside the timed region (H2D double-buffered on a
        copy stream so that the upload of a later frame overlaps this frame's compute)."""
        t0 = state['t']
        copy_stream = torch.cuda.Stream(dev)
        cur = torch.cuda.current_stream(dev)
        NB = 3 if lookahead else 2
        ahead = NB - 1
        bufs = [torch.empty_like(frames_dev[0]) for _ in range(NB)]
        ready = [torch.cuda.Event() for _ in range(NB)]
        free = [torch.cuda.Event() for _ in range(NB)]

        def upload(i):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(free[i % NB])
                bufs[i % NB].copy_(frames_pin[t0 + i], non_blocking=True)
                ready[i % NB].record(copy_stream)
        for ev in free:
            ev.record(cur)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for j in range(min(ahead, steps)):
            upload(j)
        h0 = time.perf_counter()
        for i in range(steps):
            if i + ahead < steps:
                upload(i + ahead)
            cur.wait_event(ready[i % NB])
            if lookahead:
                nxt = None
                if i + 1 < steps:
                    cur.wait_event(ready[(i + 1) % NB])
                    nxt = bufs[(i + 1) % NB]
                prob = proc.step(bufs[i % NB], next_image=nxt)
            else:
                prob = proc.step(bufs[i % NB])
            free[i % NB].record(cur)
            host_out.copy_(proc.output_prob_to_mask(prob).to(torch.uint8), non_blocking=True)
        host_ms = (time.perf_counter() - h0) * 1e3 / steps
        e1.record()
        state['t'] = t0 + steps
        return e0, e1, host_ms

    with torch.inference_mode():
        for _ in range(warm):
            proc.step(frames_dev[state['t']])
            state['t'] += 1
        # ---- timed region 1: device-resident inputs, the reference's call signature ----
        barrier()
        stop, samples = threading.Event(), []
        th = threading.Thread(target=nvsmi_sampler, args=(stop, samples, dev.index or 0), daemon=True)
        th.start()
        launches0 = K_.LAUNCH_COUNT
        if args.phase_timing:
            K_.phase_timing(True)
        marks, host_dev = device_arm(K, False, True, keep_last=bool(args.dump_outputs))
        barrier()
        stop.set(); th.join()
        launches = K_.LAUNCH_COUNT - launches0
        prof, K_.PROFILE = K_.PROFILE, None
        if args.phase_timing:
            K_.phase_timing(False)
            ph = [p for p in (K_.phase_times(i) for i in range(min(K, 60))) if p]
            if ph:
                n = min(len(p) for p in ph)
                res['phases'] = [sum(p[i] for p in ph) / len(ph) for i in range(n)]
                log('[phases] affinity plan, ms per launch: ' + ' '.join(f'{x:.3f}' for x in res['phases']))
        ms_total = marks[0].elapsed_time(marks[-1])
        per_step = [marks[i].elapsed_time(marks[i + 1]) for i in range(K)]
        kernel_ms = {}
        for name, a, b in prof:
            kernel_ms.setdefault(name, []).append(a.elapsed_time(b))
        # ---- timed region 2: end to end through the public API with host buffers ----
        barrier()
        e0, e1, host_e2e = e2e_arm(K, False)
        barrier()
        ms_e2e = e0.elapsed_time(e1)
        # ---- extension (not the reference signature): step(..., next_image=...) = encoder look-ahead ----
        look = None
        if use_graphs and not args.no_lookahead:
            for _ in range(4):                                  # the second encoder capture slot
                proc.step(frames_dev[state['t']], next_image=frames_dev[state['t'] + 1])
                state['t'] += 1
            barrier()
            lm, lh = device_arm(K, True, False)
            barrier()
            le0, le1, leh = e2e_arm(K, True)
            barrier()
            look = {'ms_total': lm[0].elapsed_time(lm[-1]), 'ms_e2e': le0.elapsed_time(le1)}
            log(f'[rank {rank}] look-ahead arms: device {look["ms_total"] / K:.2f} ms/step (host enqueue {lh:.2f}), '
                f'e2e {look["ms_e2e"] / K:.2f} ms/step (host enqueue {leh:.2f})')
    # ---- the north star's own stream configuration on the same model: 480p, 3 objects, ~10k-key memory (6 memory frames),
    # drop-in step(image), device-resident frames; every rank runs it (N streams), timed like the headline ----
    ns_ms, ns_tokens, ns_steps = 0.0, 0, 0
    if args.workload == 'cfg2' and not args.no_northstar:
        try:
            wl_ns = WORKLOADS['northstar']
            proc_ns = InferenceCore(net, cfg=make_cfg(wl_ns), use_cuda_graphs=use_graphs)
            ns_steps = min(K, 100)
            with torch.inference_mode():
                proc_ns.step(frames_dev[0], mask.to(dev), objects=objs)
                for key, shr, vals in synthetic_bank_chunks(wl_ns):
                    proc_ns.memory.work_mem.add(key.to(dev), {o: vals[:, i].to(dev) for i, o in enumerate(objs)},
                                                shr.to(dev), None, as_permanent='no')
                ns_tokens = proc_ns.memory.work_mem.size(0)
                t = 1
                for _ in range(warm):
                    proc_ns.step(frames_dev[t]); t += 1
                barrier()
                n0, n1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                n0.record()
                for _ in range(ns_steps):
                    proc_ns.step(frames_dev[t]); t += 1
                n1.record()
                barrier()
                ns_ms = n0.elapsed_time(n1)
            del proc_ns
        except Exception as e:                                   # never lose the headline to this extra arm
            log(f'[northstar stream] failed: {type(e).__name__}: {e}')
            ns_ms, ns_steps = 0.0, 0
    times = torch.tensor([ms_total, ms_e2e] + ([look['ms_total'], look['ms_e2e']] if look else [0.0, 0.0]) + [ns_ms],
                         dtype=torch.float64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(times, op=torch.distributed.ReduceOp.MAX)
    ms_total, ms_e2e = float(times[0]), float(times[1])
    if ns_steps:
        res['northstar_stream'] = {
            'what': 'the same model on BASELINE.json north_star\'s stream: 480p, 3 objects, ~10k-key working memory '
                    '(6 memory frames), InferenceCore.step(image) with device-resident frames, all ranks (max time over ranks)',
            'value': world * ns_steps / (float(times[4]) * 1e-3), 'unit': 'frames/s', 'ms_per_step': float(times[4]) / ns_steps,
            'steps': ns_steps, 'memory_tokens': ns_tokens, 'n_gpus': world}
        log(f'[northstar stream] {res["northstar_stream"]}')
    if look:
        look = {'ms_total': float(times[2]), 'ms_e2e': float(times[3])}
    log(f'[rank {rank}] host enqueue time per step: device arm {host_dev:.2f} ms, e2e arm {host_e2e:.2f} ms')
    res.update(ms_total=ms_total, ms_e2e=ms_e2e, per_step=per_step, kernel_ms=kernel_ms, launches=launches,
               n_tokens=n_tokens, clocks=summarize_clocks(samples), h2d=frames_pin[0].numel() * 4, d2h=host_out.numel(),
               host_ms=[host_dev, host_e2e], lookahead=look, untimed=warm, image_levels=K_.image_level_launches(),
               epilogues=net.conv_epilogues.report() if hasattr(net, 'conv_epilogues') else None,
               glue=net.glue_dispatch.report() if hasattr(net, 'glue_dispatch') else None)
    # ---- how selective the candidate filter is on this bank (one extra untimed frame; explains `roofline`) ----
    try:
        K_.KEEP_LAST_WORKSPACE = True
        with torch.inference_mode():
            proc.step(frames_dev[state['t']])
            state['t'] += 1
        torch.cuda.synchronize(dev)
        cnt = K_.last_candidate_counts()
        if cnt is not None:
            c = cnt.float().flatten()
            res['candidates'] = {'per_query_mean': float(c.mean()), 'per_query_p50': float(c.median()),
                                 'per_query_max': float(c.max()), 'of_tokens': n_tokens, 'top_k': wl['top_k']}
    finally:
        K_.KEEP_LAST_WORKSPACE = False
    # ---- in-run parity check: ONE frame re-computed by the CPU oracle from the live state ----
    if rank == 0 and world == 1 and not args.no_parity_check:
        try:
            res['parity'] = parity_check(proc, cfg, frames[state['t']], dev)
        except Exception as e:                                 # noqa: BLE001 -- reported, never hidden
            import traceback
            traceback.print_exc()
            res['parity'] = {'error': f'{type(e).__name__}: {e}'[:300]}
    return res


def dump_outputs(out_dir, outputs):
    """What the headline arm's last timed step returned to its caller -- InferenceCore.step's per-object probabilities
    [1 + objects, H, W] -- as float32 .npy files, for comparing two builds output for output on the same seeded inputs."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        a = t.detach().float().cpu().numpy()
        assert a.nbytes <= 64 * 2**20, (name, a.shape)
        np.save(os.path.join(out_dir, f'{name}.npy'), a)
        log(f'[dump] {name}: {a.shape} float32 -> {out_dir}')


def parity_check(proc, cfg, frame, dev):
    """The oracle (CPU restatement of the reference, dense [N,HW] affinity) re-computes the next frame from the state the
    CUDA path is in after the timed region -- the 413 100-token bank, i.e. the tcgen05 filter plan, the key-image path and
    the ring arena as the bench ran them -- and the segment() logits are compared.  The top-k sets are compared per
    query; where they differ, the CUDA choice is checked against the float64 direct-form ground truth (a near-tie the
    reference's fp32 three-term expansion cannot resolve) and adopted by the oracle, as in the teacher-forced tests."""
    import cutie_b200.kernels as K_
    from oracle.cpu_core import OracleCore
    from oracle.state_sync import ForegroundReconciler, SelectionReconciler, export_state_to_oracle
    t0 = time.perf_counter()
    oc = export_state_to_oracle(proc, OracleCore(make_net(cfg), cfg))     # un-optimised CPU copy of the same weights
    rec, fgr = SelectionReconciler(cfg.top_k, max_frac=0.05), ForegroundReconciler()
    oc.selection_hook, oc.fg_hook = rec, fgr
    orig, orig_aux = K_.affinity_topk, K_.qt_aux_mask

    def spy(*a, **k):
        out = orig(*a, **k)
        rec.gpu_idx = out[0].clone()
        return out

    def spy_aux(*a, **k):
        out = orig_aux(*a, **k)
        fgr.gpu_fg.append(out[1].clone())
        return out
    K_.affinity_topk, K_.qt_aux_mask = spy, spy_aux
    graphs = proc.use_cuda_graphs
    proc.use_cuda_graphs = False          # this one frame runs the same kernels eagerly so that the foreground maps can be read
    try:
        with torch.inference_mode():
            proc.step(frame.to(dev))
            torch.cuda.synchronize(dev)
            threads = torch.get_num_threads()
            torch.set_num_threads(usable_cpus())
            oc.step(frame)
            torch.set_num_threads(threads)
    finally:
        K_.affinity_topk, K_.qt_aux_mask = orig, orig_aux
        proc.use_cuda_graphs = graphs
    diff = float((proc.last_logits.cpu() - oc.last_logits).abs().max())
    out = {'max_abs_logit_diff': diff, 'within_1e-3': diff < 1e-3, 'queries': rec.queries,
           'topk_set_equal': rec.flips == 0, 'topk_sets_differing': rec.flips,
           'differing_sets_valid_vs_float64': True,            # SelectionReconciler raises if one is not
           'foreground_pixels_near_tied_and_adopted': fgr.flips, 'foreground_pixels': fgr.pixels,
           'memory_tokens': proc.memory.work_mem.size(0), 'seconds': time.perf_counter() - t0,
           'what': 'one teacher-forced frame after the timed region: CUDA path vs oracle/cpu_core.py from the same live state'}
    log(f'[parity] {out}')
    return out


def northstar_read_bench(dev, iters=50):
    """BASELINE.json north_star size of the fused memory read: 480p queries (1620), 3 objects, 10 000 keys -- SURVEY.md
    section 8(d): 39.1 MB algorithmic, HBM-bound (6.0 us at the measured copy bandwidth).  The read = cutie_affinity_topk
    (FP16 image plan: sample, threshold, filter, re-rank) + cutie_readout_gather, timed with CUDA events over `iters`
    back-to-back reads of a seeded synthetic bank.  The bank (2.6 MB of keys + 30.7 MB of values) fits the 126 MB L2 and
    is NOT flushed between reads: the denominator stays the HBM roofline of the algorithmic bytes, as the north star
    states it, and the line says so."""
    import cutie_b200.kernels as K_
    N, Q, K, top_k = 10000, 1620, 3, 30
    g = torch.Generator().manual_seed(3)
    key = torch.randn(1, N, 64, generator=g).to(dev)
    shr = (1 + torch.randn(1, N, generator=g) ** 2).to(dev)
    vals = tuple(torch.randn(1, N, 256, generator=g).to(dev) for _ in range(K))
    qk = torch.randn(1, 64, Q, generator=g).to(dev)
    qe = torch.sigmoid(torch.randn(1, 64, Q, generator=g)).to(dev)
    img = torch.zeros(1, K_.key_image_tiles(N), K_.KEY_IMAGE_FLOATS, device=dev)
    K_.bank_key_image(key, shr, 0, N, img)
    seg = [K_.BankSegment(key, shr, vals, img, 0)]
    with torch.inference_mode():
        for _ in range(5):
            idx, w, _ = K_.affinity_topk(seg, qk, qe, top_k)
            out = K_.readout_gather(idx, w, seg)
        torch.cuda.synchronize(dev)
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        l0 = K_.LAUNCH_COUNT
        e0.record()
        for _ in range(iters):
            idx, w, _ = K_.affinity_topk(seg, qk, qe, top_k, seed_idx=idx)       # steady state: last read's winners seed this one
        e1.record()
        for _ in range(iters):
            out = K_.readout_gather(idx, w, seg)
        e2.record()
        torch.cuda.synchronize(dev)
        K_.phase_timing(True)                                                    # per-launch breakdown (separate, untimed reads)
        for _ in range(8):
            K_.affinity_topk(seg, qk, qe, top_k, seed_idx=idx)
        torch.cuda.synchronize(dev)
        ph = [p for p in (K_.phase_times(i) for i in range(8)) if p]
        K_.phase_timing(False)
        phases = [sum(p[i] for p in ph) / len(ph) for i in range(min(len(p) for p in ph))] if ph else None
    launches = (K_.LAUNCH_COUNT - l0) / iters
    t_topk, t_gather = e0.elapsed_time(e1) / iters, e1.elapsed_time(e2) / iters
    bytes_alg = N * 65 * 4 + min(N, Q * top_k) * K * 256 * 4 + Q * 128 * 4 + Q * K * 256 * 4
    peaks = {'hbm_gbs': 6650.0}
    pk = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(pk):
        peaks = json.load(open(pk))
    ms = t_topk + t_gather
    ach = bytes_alg / (ms * 1e-3) / 1e9
    return {'what': '480p queries, 3 objects, 10 000 keys: cutie_affinity_topk + cutie_readout_gather', 'bound': 'hbm',
            'algorithmic_bytes': bytes_alg, 'ms': ms, 'affinity_topk_ms': t_topk, 'readout_gather_ms': t_gather,
            'launches_per_read': launches, 'affinity_phases_ms': phases, 'achieved': ach, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
            'frac': ach / peaks['hbm_gbs'], 'l2': 'bank fits L2 and is not flushed between reads (stated)',
            'roofline_time_us': bytes_alg / (peaks['hbm_gbs'] * 1e9) * 1e6}


def conv_roofline_bench(dev, iters=40):
    """The convolution kernel that now carries most of the step (cutie_conv_tc, tcgen05 3xTF32 implicit GEMM) on the layers
    it runs at cfg 2, timed alone with CUDA events (L2-warm, back to back): fp32-equivalent TFLOP/s = 2 NB H W Cout Cin k^2 /
    time; the tensor pipe executes 3 TF32 MMAs per product, so the tensor-bound ceiling of the fp32-equivalent figure is the
    measured dense bf16 throughput / 2 (TF32 rate) / 3."""
    import cutie_b200.kernels as K_
    peaks = {'bf16_tflops': 1650.0}
    pk = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(pk):
        peaks = json.load(open(pk))
    ceiling = peaks['bf16_tflops'] / 2 / 3
    layers = [('PixelFFN / fuser 3x3 256->256 @30x54 x3 objects', 3, 256, 256, 30, 54, 3, False),
              ('sensory update 3x3 512->768 @30x54 x3', 3, 512, 768, 30, 54, 3, False),
              ('decoder 3x3 128->128 @120x216 x3', 3, 128, 128, 120, 216, 3, False),
              ('ResNet-50 layer3 3x3 256->256 @30x54 (channels-last, shared tiles)', 1, 256, 256, 30, 54, 3, True),
              ('ResNet-50 layer3 1x1 1024->256 @30x54 (channels-last, shared tiles)', 1, 1024, 256, 30, 54, 1, True),
              ('ResNet-50 layer1 1x1 64->256 @120x216 + residual (channels-last)', 1, 64, 256, 120, 216, 1, True)]
    out = []
    g = torch.Generator().manual_seed(5)
    with torch.inference_mode():
        for name, NB, Cin, Cout, H, W, k, cl in layers:
            x = torch.randn(NB, Cin, H, W, generator=g).to(dev)
            z = torch.randn(NB, Cout, H, W, generator=g).to(dev)
            if cl:
                x, z = x.contiguous(memory_format=torch.channels_last), z.contiguous(memory_format=torch.channels_last)
            w = (torch.randn(Cout, Cin, k, k, generator=g) * 0.02).to(dev)
            b = torch.randn(Cout, generator=g).to(dev)
            img = K_.conv_weight_image(w)
            cnt = torch.zeros(8192, dtype=torch.int32, device=dev)
            for _ in range(4):
                K_.conv_tc(x, img, b, Cout, ksize=k, residual=z, relu_out=True, counters=cnt)
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                K_.conv_tc(x, img, b, Cout, ksize=k, residual=z, relu_out=True, counters=cnt)
            e1.record()
            torch.cuda.synchronize(dev)
            us = e0.elapsed_time(e1) / iters * 1e3
            flops = 2.0 * NB * H * W * Cout * Cin * k * k
            nbytes = 4.0 * (x.numel() + 2 * z.numel() + 2 * w.numel())
            out.append({'layer': name, 'us': us, 'fp32_equivalent_tflops': flops / us / 1e6, 'frac_of_3xtf32_ceiling': flops / us / 1e6 / ceiling,
                        'hbm_view_gbs': nbytes / us / 1e3})
    return {'kernel': 'cutie_conv_tc (csrc/conv_tc.cu)', 'bound': 'tensor', 'unit': 'TFLOP/s (fp32-equivalent)',
            'peak': ceiling, 'peak_source': 'MEASURED_PEAKS.json bf16_tflops (burst: kernel timed alone) / 2 (TF32) / 3 (three MMAs per product)',
            'achieved': max(o['fp32_equivalent_tflops'] for o in out), 'frac': max(o['frac_of_3xtf32_ceiling'] for o in out),
            'layers': out, 'note': 'host-launched back to back: layers shorter than ~25 us are launch-bound here (inside the '
                                   'frame they replay from CUDA graphs)'}


# ---------------------------------------------------------------------------------------------------
def run_cpu_port(args, wl, max_seconds, steps, warmup):
    """The reference's algorithm on the host cores as restated by oracle/cpu_core.py (pinned to the reference by
    tests/test_oracle_golden.py): same weights, same synthetic video, same pre-filled bank.  kind = "port"."""
    from oracle.cpu_core import OracleCore
    from oracle.synth import synthetic_video
    cfg = make_cfg(wl)
    net = make_net(cfg)
    frames, mask = synthetic_video(warmup + steps + 2, wl['H'], wl['W'], wl['K'], seed=0)
    objs = list(range(1, wl['K'] + 1))
    oc = OracleCore(net, cfg)
    t_begin = time.perf_counter()
    with torch.inference_mode():
        oc.step(frames[0], mask, objects=objs)
        ks, ss, vs = [oc.work.k[0]], [oc.work.s[0]], {o: [oc.work.v[o]] for o in objs}
        for key, shr, vals in synthetic_bank_chunks(wl):
            ks.append(key), ss.append(shr)
            for i, o in enumerate(objs):
                vs[o].append(vals[:, i])
        oc.work.k[0], oc.work.s[0] = torch.cat(ks, -1), torch.cat(ss, -1)
        for o in objs:
            oc.work.v[o] = torch.cat(vs[o], -1)
        del ks, ss, vs
        log(f'[cpu] bank prefilled: {oc.work.size(0)} tokens; threads={torch.get_num_threads()}')
        per_frame = []
        t = 1
        for i in range(warmup + steps):
            if per_frame and (time.perf_counter() - t_begin) + max(per_frame) > max_seconds and i >= warmup + 1:
                break
            t0 = time.perf_counter()
            oc.step(frames[t]); t += 1
            dt = time.perf_counter() - t0
            if i >= warmup:
                per_frame.append(dt)
            log(f'[cpu] frame {i} {"(warmup) " if i < warmup else ""}{dt:.2f} s')
    return per_frame


def run_cpu_reference(args, wl, max_seconds, steps, warmup, threads):
    """The UNMODIFIED reference (baseline/_ref) on the host cores, in a child process (baseline/ref_bench_child.py).
    Returns (per-frame seconds, info) or (None, why) when no reference tree travelled with the repo."""
    from oracle import ref_harness as rh
    if not rh.available():
        return None, 'no reference tree (baseline/_ref is created by __graft_entry__.build() where /root/reference exists)'
    job = dict(H=wl['H'], W=wl['W'], K=wl['K'], mem_frames=wl['mem_frames'], top_k=wl['top_k'], steps=steps, warmup=warmup,
               max_seconds=max_seconds, threads=threads)
    env = dict(os.environ, CUTIE_REFERENCE_ROOT=rh.REF_ROOT)
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'baseline', 'ref_bench_child.py'), json.dumps(job)], env=env,
                       stdout=subprocess.PIPE, stderr=None, text=True, timeout=max_seconds * 4 + 900)
    if r.returncode != 0:
        return None, f'reference child exited {r.returncode}'
    out = json.loads(r.stdout.strip().splitlines()[-1])
    return out['per_frame_s'], out


def reference_arm(args, wl, config):
    """bench.py --impl reference: the reference's own implementation of the path on the box's host cores."""
    cores = usable_cpus()
    torch.set_num_threads(cores)
    budget = max(args.cpu_seconds, 60.0)
    per, info = run_cpu_reference(args, wl, budget, args.steps, min(args.warmup, 1), cores)
    kind, note = 'reference', None
    calib = None
    if not per:
        log(f'[reference arm] {info}; timing the oracle port instead')
        kind, note = 'port', str(info)
        per = run_cpu_port(args, wl, budget, args.steps, min(args.warmup, 1))
    elif not args.no_port_calibration:
        # how the oracle port (the in-run cpu_baseline of the other arm) compares with the real thing on this box
        pp = run_cpu_port(args, wl, 60.0, 2, 1)
        calib = {'port_frames_per_s': len(pp) / sum(pp), 'reference_frames_per_s': len(per) / sum(per), 'port_frames': len(pp)}
    fps = len(per) / sum(per)
    line = {'impl': 'reference', 'metric': METRIC, 'value': fps, 'unit': 'frames/s', 'n_gpus': args.gpus,
            'steps': len(per), 'warmup': min(args.warmup, 1), 'ms_per_step': 1000 * sum(per) / len(per),
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': config,
            'cpu_baseline': {'value': fps, 'unit': 'frames/s', 'cores': cores, 'kind': kind,
                             'sample': f'{len(per)} full frame(s) of the same workload (time-bounded; {args.steps} requested) '
                                       + ('through the unmodified reference (baseline/_ref) InferenceCore.step'
                                          if kind == 'reference' else 'through oracle/cpu_core.py'),
                             'note': note, 'port_calibration': calib},
            'e2e': {'value': fps, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    emit(line)


# ---------------------------------------------------------------------------------------------------
def sharded_read_bench(rank, world, dev):
    """BASELINE.json configs[4] on the N ranks of the scaling run: 1080p queries (8160), 10 objects (rounded up to a
    multiple of N), a 50 000-key bank sharded 50 000/N keys per rank; local top-k -> NCCL all-gather of (similarity, global
    index) candidates -> merge -> local partial readout -> NCCL all-reduce (replicated result) or reduce-scatter over
    objects (object-sharded continuation).  Asserts bit-identity of the selection and weights with rank 0's unsharded read."""
    import torch.distributed as dist
    import cutie_b200.kernels as K_
    from cutie_b200.inference.sharded import shard_bounds, sharded_topk
    n_total, Q, K, top_k, B = 50000, 8160, 10, 30, 1
    K = -(-K // world) * world                                   # reduce-scatter over objects needs K % N == 0
    g = torch.Generator().manual_seed(7)
    key = torch.randn(B, n_total, 64, generator=g)
    shr = 1 + torch.randn(B, n_total, generator=g) ** 2
    qk = torch.randn(B, 64, Q, generator=g).to(dev)
    qe = torch.sigmoid(torch.randn(B, 64, Q, generator=g)).to(dev)
    lo, hi = shard_bounds(n_total, world, rank)
    gl = torch.Generator().manual_seed(100 + rank)
    vals_local = [torch.randn(B, hi - lo, 256, generator=gl).to(dev) for _ in range(K)]
    key_l, shr_l = key[:, lo:hi].to(dev).contiguous(), shr[:, lo:hi].to(dev).contiguous()
    img = torch.zeros(B, K_.key_image_tiles(hi - lo), K_.KEY_IMAGE_FLOATS, device=dev)      # as the runtime's arenas keep it
    K_.bank_key_image(key_l, shr_l, 0, hi - lo, img)
    seg = K_.BankSegment(key_l, shr_l, tuple(vals_local), img, 0)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    res = {'keys': n_total, 'keys_per_rank': hi - lo, 'queries': Q, 'objects': K, 'ranks': world}
    with torch.inference_mode():
        def one(mode):
            e = [ev() for _ in range(4)]
            marks = []
            e[0].record()
            idx_l, w_l, idx, w = sharded_topk([seg], lo, n_total, qk, qe, top_k, marks=marks)
            e[1].record()
            e += [e[0]] + marks + [e[1]]           # [4..7]: begin, after local top-k, after all-gather, after merge
            part = K_.readout_gather(idx_l, w_l, [seg])          # [B, K, 256, Q] partial sums over this rank's winners
            e[2].record()
            if mode == 'all_reduce':
                dist.all_reduce(part, op=dist.ReduceOp.SUM)
                out = part
            else:
                out = torch.empty(K // world * 256 * Q, device=dev)     # this rank's K/N objects of the summed readout
                dist.reduce_scatter_tensor(out, part[0].contiguous().view(-1), op=dist.ReduceOp.SUM)
            e[3].record()
            return e, idx, w, out
        for mode in ('all_reduce', 'reduce_scatter'):
            for _ in range(3):
                one(mode)
            dist.barrier()
            torch.cuda.synchronize(dev)
            t = [[] for _ in range(6)]
            for _ in range(10):
                e, idx, w, out = one(mode)
                torch.cuda.synchronize(dev)
                for i in range(3):
                    t[i].append(e[i].elapsed_time(e[i + 1]))
                for i in range(3):
                    t[3 + i].append(e[4 + i].elapsed_time(e[5 + i]))
            tm = torch.tensor([sum(x) / len(x) for x in t], dtype=torch.float64, device=dev)
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            res[mode] = {'topk_allgather_merge_ms': float(tm[0]), 'local_gather_ms': float(tm[1]),
                         'collective_ms': float(tm[2]), 'total_ms': float(tm[:3].sum()),
                         'local_topk_ms': float(tm[3]), 'candidate_allgather_ms': float(tm[4]), 'merge_ms': float(tm[5])}
        res['allgather_bytes_per_rank'] = int(idx.numel() * 8)
        res['readout_bytes'] = int(B * K * 256 * Q * 4)
        # bit-identity with the unsharded read (rank 0 holds the whole key bank for the check)
        ok = torch.ones(1, device=dev)
        if rank == 0:
            full = K_.BankSegment(key.to(dev), shr.to(dev), ())
            ridx, rw, _ = K_.affinity_topk([full], qk, qe, top_k)
            ok[0] = float(torch.equal(idx, ridx) and torch.equal(w, rw))
        dist.broadcast(ok, 0)
        res['bit_identical_to_unsharded'] = bool(ok.item())
    res['limiting'] = max(('local_topk_ms', 'candidate_allgather_ms', 'merge_ms', 'local_gather_ms', 'collective_ms'),
                          key=lambda k: res['reduce_scatter'][k])
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='cfg2', choices=sorted(WORKLOADS))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-parity-check', action='store_true')
    ap.add_argument('--no-port-calibration', action='store_true')
    ap.add_argument('--no-optimize', action='store_true', help='skip CUTIE.optimize_for_inference()')
    ap.add_argument('--no-cudnn-benchmark', action='store_true', help='cuDNN heuristics instead of its autotuner')
    ap.add_argument('--phase-timing', action='store_true', help='per-launch device times inside cutie_affinity_topk')
    ap.add_argument('--no-graphs', action='store_true', help='eager launches only (no CUDA-graph frame regions)')
    ap.add_argument('--no-lookahead', action='store_true', help='skip the extension arm step(..., next_image=...)')
    ap.add_argument('--no-sharded-read', action='store_true', help='skip the key-sharded read benchmark at N > 1')
    ap.add_argument('--no-northstar', action='store_true', help='skip the north-star-size memory-read micro-benchmark')
    ap.add_argument('--cpu-seconds', type=float, default=150.0)
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the last timed step\'s outputs (InferenceCore.step probabilities) as DIR/<name>.npy')
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    HW = tokens_per_frame(wl)
    config = base_config(args, wl, world)

    if args.impl == 'reference':
        if rank == 0:
            reference_arm(args, wl, config)
        return

    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device: there is no CPU fallback for the product path '
                         '(use --impl reference for the CPU arm)')
    dev = torch.device('cuda', local)
    torch.cuda.set_device(dev)
    if world > 1:
        torch.distributed.init_process_group('nccl', device_id=dev)
    res = run_ours(args, wl, rank, world, dev)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res.pop('outputs'))
    conv_roof = None
    if rank == 0 and not args.no_northstar:
        try:
            conv_roof = conv_roofline_bench(dev)
            log(f'[conv] {conv_roof}')
        except Exception as e:                                 # noqa: BLE001 -- reported, never hidden
            conv_roof = {'error': f'{type(e).__name__}: {e}'[:300]}
    northstar = None
    if rank == 0 and not args.no_northstar:
        try:
            northstar = northstar_read_bench(dev)
            log(f'[northstar] {northstar}')
        except Exception as e:                                   # noqa: BLE001 -- reported in the line, never hidden
            import traceback
            traceback.print_exc()
            northstar = {'error': f'{type(e).__name__}: {e}'[:300]}
    sharded = None
    if world > 1 and not args.no_sharded_read:
        try:
            sharded = sharded_read_bench(rank, world, dev)
        except Exception as e:                                   # noqa: BLE001 -- reported in the line, never hidden
            import traceback
            traceback.print_exc()
            sharded = {'error': f'{type(e).__name__}: {e}'[:300]}
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        torch.set_num_threads(usable_cpus())
        per = run_cpu_port(args, wl, max_seconds=40.0, steps=1, warmup=1)
        cpu = {'value': len(per) / sum(per), 'unit': 'frames/s', 'cores': torch.get_num_threads(), 'kind': 'port',
               'sample': f'{len(per)} full frame of the same workload (same weights, same pre-filled bank) through '
                         f'oracle/cpu_core.py, after one untimed warm-up frame; `bench.py --impl reference` times the '
                         f'unmodified reference (baseline/_ref) and calibrates this port against it'}
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    if rank != 0:
        return
    peaks = {'hbm_gbs': 6650.0, 'bf16_tflops_sustained': 1400.0, 'src': 'fallback'}
    pk = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(pk):
        peaks = dict(json.load(open(pk)), src='measured')
    N = res['n_tokens']
    K = args.steps
    scan = res['kernel_ms'].get('affinity_topk', [])
    scan_ms = sum(scan) / len(scan) if scan else None
    flops = 2.0 * N * 128 * HW                       # SURVEY.md 8(d): one K=128 contraction [mk^2|mk].[-qe;2qk.qe]
    bytes_alg = N * 65 * 4 + HW * 128 * 4 + HW * 32 * 8
    gather = res['kernel_ms'].get('readout_gather', [])
    gather_ms = sum(gather) / len(gather) if gather else None
    gather_bytes = min(N, HW * wl['top_k']) * wl['K'] * 256 * 4 + HW * wl['K'] * 256 * 4 + HW * 32 * 8
    tensor_bound = flops / (peaks['bf16_tflops_sustained'] * 1e12) > bytes_alg / (peaks['hbm_gbs'] * 1e9)
    traffic, traffic_note = None, None
    tj = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')       # dram bytes of one `ncu --set full` capture (per launch)
    if os.path.exists(tj) and args.workload == 'cfg2':
        t = json.load(open(tj))
        traffic, traffic_note = t.get('affinity_topk_dram_bytes'), t.get('note')
    roof = None
    if scan_ms:
        if tensor_bound:
            ach = flops / (scan_ms * 1e-3) / 1e12
            roof = {'bound': 'tensor', 'kernel': 'cutie_affinity_topk (tcgen05 candidate filter over the key operand image + '
                                                 'exact fp32 re-rank; csrc/affinity*.cu)',
                    'achieved': ach, 'peak': peaks['bf16_tflops_sustained'], 'unit': 'TFLOP/s',
                    'frac': ach / peaks['bf16_tflops_sustained'], 'traffic': traffic, 'traffic_note': traffic_note,
                    'peak_source': f"{peaks['src']} bf16 sustained (kernel timed inside a long step)",
                    'algorithmic_flops_per_launch': flops, 'avg_launch_ms': scan_ms,
                    'hbm_view': {'algorithmic_bytes': bytes_alg, 'achieved_gbs': bytes_alg / (scan_ms * 1e-3) / 1e9,
                                 'frac': bytes_alg / (scan_ms * 1e-3) / 1e9 / peaks['hbm_gbs']}}
        else:
            ach = bytes_alg / (scan_ms * 1e-3) / 1e9
            roof = {'bound': 'hbm', 'kernel': 'cutie_affinity_topk', 'achieved': ach, 'peak': peaks['hbm_gbs'],
                    'unit': 'GB/s', 'frac': ach / peaks['hbm_gbs'], 'traffic': None,
                    'peak_source': f"{peaks['src']} copy bandwidth", 'algorithmic_bytes_per_launch': bytes_alg,
                    'avg_launch_ms': scan_ms}
        if gather_ms:
            roof['readout_gather'] = {'bound': 'hbm', 'algorithmic_bytes': gather_bytes, 'avg_launch_ms': gather_ms,
                                      'achieved_gbs': gather_bytes / (gather_ms * 1e-3) / 1e9,
                                      'frac': gather_bytes / (gather_ms * 1e-3) / 1e9 / peaks['hbm_gbs']}
    kshare = {k: {'avg_ms': sum(v) / len(v), 'p50_ms': sorted(v)[len(v) // 2], 'max_ms': max(v),
                  'calls_per_step': len(v) / K, 'share_of_step': sum(v) / res['ms_total']}
              for k, v in res['kernel_ms'].items()}
    fps = world * K / (res['ms_total'] * 1e-3)
    fps_e2e = world * K / (res['ms_e2e'] * 1e-3)
    line = {'metric': METRIC, 'value': fps, 'unit': 'frames/s', 'n_gpus': world, 'steps': K, 'warmup': args.warmup,
            'ms_per_step': res['ms_total'] / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic', 'config': config, 'clocks': res['clocks'],
            'e2e': {'value': fps_e2e, 'unit': 'frames/s', 'h2d_bytes_per_step': res['h2d'],
                    'd2h_bytes_per_step': res['d2h'], 'ms_per_step': res['ms_e2e'] / K},
            'gpu_launches': res['launches'], 'roofline': roof, 'cpu_baseline': cpu,
            'parity_check': res.get('parity'), 'latency_ms': percentiles(res['per_step']),
            'untimed_steps_before_timed_region': res['untimed'],
            'api': 'InferenceCore.step(image) -- the reference signature (scripting_demo.py / eval_vos.py unchanged)',
            'with_encoder_lookahead': None if not res['lookahead'] else {
                'what': 'extension step(image, next_image=...): the next frame\'s encoder graph on a side stream; NOT the '
                        'reference signature, reported beside the headline',
                'value': world * K / (res['lookahead']['ms_total'] * 1e-3),
                'e2e': world * K / (res['lookahead']['ms_e2e'] * 1e-3), 'unit': 'frames/s'},
            'kernels': kshare,
            'host_enqueue_ms_per_step': {'device_arm': res['host_ms'][0], 'e2e_arm': res['host_ms'][1]},
            'affinity_phases_ms': res.get('phases'), 'affinity_candidates': res.get('candidates'),
            'key_image_levels': res['image_levels'],
            'build': {'cuda_graphs': not args.no_graphs, 'optimize_for_inference': not args.no_optimize,
                      'cudnn_benchmark': not args.no_cudnn_benchmark, 'cudnn_allow_tf32': False, 'matmul_allow_tf32': False,
                      'conv_epilogues': res['epilogues'], 'glue_dispatch': res['glue'],
                      'qt_chain': __import__('cutie_b200.model.object_transformer', fromlist=['QT_CHAIN']).QT_CHAIN},
            'roofline_northstar': northstar, 'northstar_stream': res.get('northstar_stream'), 'roofline_conv': conv_roof,
            'sharded_read': sharded}
    emit(line)


if __name__ == '__main__':
    main()
