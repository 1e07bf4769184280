#!/usr/bin/env python
"""Benchmark of the cross-attention heat-map hot path (BASELINE.json metric: heat-map px/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload sd21|sd21_768|sdxl|sdxl70|sd15] [--prompts P]
                    [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): random-init SD-2.1-base UNet shapes, 64x64 latent, 77 tokens, bf16, the 15 traced
cross-attention layers of one denoising step. A bench "step" is one pass of the hot path over one step's Q/K:
13.80 M accumulated heat-map px (SURVEY.md section 8d: sum over traced layers of heads*77*h*w).

One JSON line is printed by rank 0:
  value         px/s with Q/K already resident in HBM: one persistent `daam_accumulate` launch per step (all 15
                layers), K steps timed with CUDA events between barriers, max over ranks, x N ranks (weak scaling).
                Inputs exceed L2: the steps rotate over R independent resident prompt sets (accumulators + Q/K).
  roofline      the accumulate kernel against the measured HBM copy bandwidth (MEASURED_PEAKS.json), algorithmic bytes.
  e2e           the same metric through the public API -- `with trace(pipe): pipe(prompt, K steps);
                compute_global_heat_map()` on the cross-attention skeleton of the UNet -- with the pipeline inputs in
                pinned HOST memory copied H2D every step and results read D2H inside the timed region.
  cpu_baseline  the oracle's port of the reference hot path (rows a3+a4+a6) timed on this box's host cores on a bounded
                sample of the same Q/K shapes.
  hook_overhead hooked vs un-hooked forward of a full-cost synthetic UNet (resnets, self-attention, feed-forward), ms/step.

`--impl reference` times the reference's own CPU implementation of the path instead (the oracle's op-for-op port of
daam/trace.py's hook, since the Python reference cannot travel to the GPU box) through the same pipeline API on CPU.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'heatmap px/s (layers x steps x tokens)'
UNIT = 'px/s'
TOKENS = 77


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# Libraries (NCCL banners, cuDNN logs) may write to fd 1; the driver expects exactly one JSON line on stdout. Everything
# this process prints to fd 1 is sent to stderr, and the JSON line alone goes to the real stdout at the end.
_REAL_STDOUT = None


def capture_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + '\n').encode()
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


# --------------------------------------------------------------------------------------------------------------------
# workload description
# --------------------------------------------------------------------------------------------------------------------
def traced_layers(workload: str):
    """(hw, heads, head_dim) of every traced layer in the reference's layer_idx order (SURVEY.md section 8)."""
    if workload == 'sd21':
        shapes = [(256, 20)] * 3 + [(1024, 10)] * 3 + [(4096, 5)] * 3 + [(4096, 5)] * 2 + [(1024, 10)] * 2 + [(256, 20)] * 2
        return [(hw, h, 64) for hw, h in shapes]
    if workload == 'sd21_768':   # the 768-pixel SD-2.1: 96x96 latent, 9216 / 2304 / 576 query positions (partial 128-pixel tiles)
        shapes = [(576, 20)] * 3 + [(2304, 10)] * 3 + [(9216, 5)] * 3 + [(9216, 5)] * 2 + [(2304, 10)] * 2 + [(576, 20)] * 2
        return [(hw, h, 64) for hw, h in shapes]
    if workload == 'sdxl':   # 60 layers (default trace, no mid block): up 3x10 @32^2, 3x2 @64^2; down 2x2 @64^2, 2x10 @32^2
        shapes = [(1024, 20)] * 30 + [(4096, 10)] * 6 + [(4096, 10)] * 4 + [(1024, 20)] * 20
        return [(hw, h, 64) for hw, h in shapes]
    if workload == 'sdxl70':   # BASELINE configs[4]: "all 70 cross-attn layers traced" = the 60 above + the mid block's 10
        # (located only with the tracer's locate_middle_block switch; reference: daam/trace.py:34-35, daam/hook.py:110-114,
        # where the mid block comes last in layer order)
        return traced_layers('sdxl') + [(1024, 20, 64)] * 10
    if workload == 'sd15':   # SD-1.x: 8 heads everywhere, head dims 160 / 80 / 40
        shapes = [(256, 160)] * 3 + [(1024, 80)] * 3 + [(4096, 40)] * 3 + [(4096, 40)] * 2 + [(1024, 80)] * 2 + [(256, 160)] * 2
        return [(hw, 8, d) for hw, d in shapes]
    raise ValueError(workload)


def px_per_step(layers, n_prompts=1):
    return n_prompts * sum(h * TOKENS * hw for hw, h, _ in layers)


def literal_px_per_step(layers, n_prompts=1, x=None):
    x = x or (96 if max(hw for hw, _, _ in layers) == 9216 else 64)
    return n_prompts * len(layers) * TOKENS * x * x      # BASELINE-literal "layers x tokens x 64^2"


def algorithmic_bytes_per_step(layers, n_prompts=1, esize=2):
    """SURVEY.md section 8d: Q + K in the config dtype, fp32 accumulator read + write (conditional half only)."""
    return n_prompts * sum(h * hw * d * esize + h * TOKENS * d * esize + h * TOKENS * hw * 4 * 2 for hw, h, d in layers)


def measured_peak():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        with open(path) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


def recorded_traffic(workload):
    """dram bytes per launch of the accumulate kernel from the committed ncu capture, if there is one."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'accumulate_traffic.json')) as f:
            return json.load(f).get(workload)
    except Exception:
        return None


# --------------------------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi, during the timed regions)
# --------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ('clocks.sm,clocks.max.sm,power.draw,utilization.gpu,clocks_event_reasons.hw_slowdown,'
              'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
              'clocks_event_reasons.sw_power_cap')

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={index}', f'--query-gpu={self.FIELDS}',
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(',')]))

    def stop(self, windows):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'note': 'nvidia-smi unavailable'}
        time.sleep(0.15)
        self.proc.terminate()
        inside = [r for t, r in self.rows if any(a <= t <= b for a, b in windows)] or [r for _, r in self.rows]
        sm = sorted(float(r[0]) for r in inside if r[0].replace('.', '').isdigit())
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({n for r in inside for n, v in zip(names, r[4:8]) if v.lower().startswith('active')})
        mx = [float(r[1]) for r in inside if r[1].replace('.', '').isdigit()]
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(inside)}


# --------------------------------------------------------------------------------------------------------------------
# distributed helpers
# --------------------------------------------------------------------------------------------------------------------
class Dist:
    def __init__(self, n_gpus: int):
        import torch.distributed as dist
        self.world = int(os.environ.get('WORLD_SIZE', '1'))
        self.rank = int(os.environ.get('RANK', '0'))
        self.local_rank = int(os.environ.get('LOCAL_RANK', '0'))
        self.dist = dist
        if self.world > 1:
            os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
            torch.cuda.set_device(self.local_rank)
            dist.init_process_group('nccl', device_id=torch.device('cuda', self.local_rank))
        else:
            torch.cuda.set_device(0)
        if n_gpus != self.world:
            log(f'[bench] --gpus {n_gpus} but WORLD_SIZE {self.world}: launch with torchrun for N > 1; using {self.world}')

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def max_ms(self, ms: float) -> float:
        if self.world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device='cuda')
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


# --------------------------------------------------------------------------------------------------------------------
# legs
# --------------------------------------------------------------------------------------------------------------------
def build_sets(layers, n_prompts, dtype, n_sets, seed):
    """R independent resident prompt sets: per layer Q [2P, hw, H*64], K [2P, 77, H*64] and the fp32 accumulators."""
    from daam_b200 import ops
    g = torch.Generator(device='cuda').manual_seed(seed)
    sets = []
    for _ in range(n_sets):
        descs, keep = [], []
        for hw, heads, d in layers:
            q = torch.randn(2 * n_prompts, hw, heads * d, generator=g, device='cuda', dtype=torch.float32).to(dtype)
            k = torch.randn(2 * n_prompts, TOKENS, heads * d, generator=g, device='cuda', dtype=torch.float32).to(dtype)
            acc = ops.new_accumulator(n_prompts, heads, hw, 'cuda')
            descs.append(ops.make_layer_desc(q, k, acc, heads, d ** -0.5))
            keep.append((q, k, acc))
        sets.append((ops.pack(descs), keep))
    return sets


def leg_value(args, layers, dtype, D: Dist, windows):
    """K steps (one persistent launch per traced-layer pack each) between CUDA events: barrier + synchronize, K timed
    steps, synchronize + barrier; the time is the max over ranks. The launches are queued behind a short spin kernel so
    that the device executes them back to back: the figure is device throughput, not host launch pacing (8 Python
    processes share one host at N=8).

    Also returns the accumulators of the prompt set the last timed step added into: what the caller of the path gets."""
    from daam_b200 import _native, ops
    n_sets, _ = value_sets(layers, args.prompts)               # working set >= 320 MB > 126 MB L2
    sets = build_sets(layers, args.prompts, dtype, n_sets, 1234 + D.rank)
    stream = torch.cuda.current_stream()
    flags = _native.ACC_AUTO | _native.ACC_EARLY_LOADS       # Q/K are resident inputs: complete long before any launch
    for i in range(args.warmup):
        ops.accumulate(sets[i % n_sets][0], 'cuda', stream, flags)
    torch.cuda.synchronize()
    gate_cycles = int(max(2.0, args.steps * 0.04) * 1.9e6)     # ~max(2 ms, 40 us per launch) at 1.9 GHz
    launches0 = _native.launch_count()
    step = args.warmup
    D.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    torch.cuda._sleep(gate_cycles)
    e0.record(stream)
    for _k in range(args.steps):
        ops.accumulate(sets[step % n_sets][0], 'cuda', stream, flags)
        step += 1
    e1.record(stream)
    torch.cuda.synchronize()
    D.barrier()
    torch.cuda.synchronize()
    windows.append((t0, time.time()))
    launches = _native.launch_count() - launches0
    mine = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device='cuda')
    if D.world > 1:
        allr = torch.empty(D.world, dtype=torch.float64, device='cuda')
        D.dist.all_gather_into_tensor(allr, mine)
    else:
        allr = mine
    ms = float(allr.max())
    stats = {'steps': args.steps, 'us_per_step_max_over_ranks': round(ms / args.steps * 1e3, 3),
             'per_rank_us_per_step': [{'rank': r, 'us': round(float(allr[r]) / args.steps * 1e3, 3)}
                                      for r in range(D.world)]}
    # sanity: the timed work really accumulated (softmax rows sum to 1 -> each head gained hw per visit)
    q, k, acc = sets[0][1][0]
    visits = len(range(0, step, n_sets))
    got = float(acc[0, 0].double().sum())
    assert abs(got - visits * acc.shape[-1]) < 1e-3 * got, (got, visits)
    last = [acc for _, _, acc in sets[(step - 1) % n_sets][1]]
    return ms, launches, n_sets, stats, last


def leg_e2e(args, spec, dtype, D: Dist, windows, cuda_graph=True):
    """Public API on the cross-attention skeleton: host-resident pipeline inputs, H2D/D2H every step. With
    ``cuda_graph`` the pipeline replays the step's device work (UNet + the tracer's kernel) from a CUDA graph."""
    from daam_b200 import trace
    from daam_b200.distributed import gather_heat_maps
    from daam_b200.testing.synthetic import make_pipeline
    mid = args.workload == 'sdxl70'
    prompts = ['a photo of a dog chasing a red ball on the beach at sunset'] * args.prompts
    prompt_arg = prompts[0] if args.prompts == 1 else prompts

    def generate(seed, steps, timed):
        pipe = make_pipeline(spec, body='skeleton', dtype=dtype, device='cuda', seed=seed, init_on_device=True,
                             cuda_graph=cuda_graph)
        with trace(pipe, batch_prompts=args.prompts > 1, locate_middle_block=mid) as tc:
            pipe(prompt_arg, num_inference_steps=max(3, args.warmup))     # also captures the step graph
            tc.compute_global_heat_map()
            torch.cuda.synchronize()
            if not timed:
                pipe(prompt_arg, num_inference_steps=steps)
                return [tc.compute_global_heat_map(prompt_idx=i).heat_maps for i in range(args.prompts)], None
            D.barrier()
            torch.cuda.synchronize()
            t0 = time.time()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            pipe(prompt_arg, num_inference_steps=steps)
            maps = [tc.compute_global_heat_map(prompt_idx=i).heat_maps for i in range(args.prompts)]
            if D.world > 1:   # the one optional collective: finished maps to every rank (1.26 MB per prompt)
                allmaps = gather_heat_maps(maps, args.prompts * D.world, maps[0].shape[-1])
            else:
                allmaps = torch.stack([m for m in maps])
            out_h = allmaps.to('cpu', non_blocking=False)          # D2H of the result
            e1.record()
            torch.cuda.synchronize()
            D.barrier()
            torch.cuda.synchronize()
            windows.append((t0, time.time()))
            return maps, (e0.elapsed_time(e1), pipe.h2d_bytes_per_step, pipe.d2h_bytes_per_step, out_h)

    maps, (ms_local, h2d, d2h_step, out_h) = generate(D.rank, args.steps, True)
    ms = D.max_ms(ms_local)
    d2h = d2h_step + out_h.numel() * 4 / max(1, args.steps) / max(1, D.world)
    assert torch.isfinite(out_h).all() and float(out_h.sum()) > 0
    # gather ORDER check (untimed): prompt j of rank r must sit at row r + j * world. Rank 0 re-generates rank 1's first
    # prompt itself (same seed -> same weights and inputs; every kernel on the path is deterministic) and compares.
    order = None
    if D.world > 1 and D.rank == 0 and cuda_graph:
        try:
            same_own = all(torch.equal(out_h[j * D.world][:m.shape[0]], m.cpu()) for j, m in enumerate(maps))
            foreign, _ = generate(1, args.steps, False)
            f = foreign[0].cpu()
            err = float((out_h[1][:f.shape[0]] - f).abs().max() / f.abs().max())
            differs = float((out_h[0][:f.shape[0]] - f).abs().max() / f.abs().max())
            order = {'own_rows_bit_equal': bool(same_own), 'rank1_prompt0_rel_err_vs_recomputation_on_rank0': err,
                     'rank0_vs_rank1_maps_rel_diff': differs,
                     'ok': bool(same_own and err < 1e-3 and differs > 10 * max(err, 1e-6))}
        except Exception as e:      # the check must never cost the run its number
            order = {'ok': False, 'error': repr(e)}
        if not order['ok']:
            log(f'[bench] WARNING: gather order check failed: {order}')
    return ms, h2d, d2h, order, out_h


def leg_hook_overhead(args, spec, dtype, windows):
    """Hooked vs un-hooked forward of the full-cost synthetic UNet, CUDA-event timed, median over steps."""
    from daam_b200 import trace
    from daam_b200.testing.synthetic import make_pipeline
    pipe = make_pipeline(spec, body='full', dtype=dtype, device='cuda', seed=0, init_on_device=True)
    n = 20
    spec_ = pipe.unet.spec
    lat = torch.randn(2, spec_.in_channels, spec_.sample_size, spec_.sample_size, device='cuda', dtype=dtype)
    emb = torch.randn(2, spec_.tokens, spec_.cross_attention_dim, device='cuda', dtype=dtype)
    t_dev = torch.full((1,), 500.0, device='cuda')

    def forwards(k):
        """Per-forward device times (CUDA events) of k forwards."""
        times = []
        for i in range(k):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            pipe.unet(lat, t_dev, emb)
            b.record()
            times.append((a, b))
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in times]

    def median(ts):
        ts = sorted(ts)
        return ts[len(ts) // 2]

    def run(k):
        return median(forwards(k))

    t0 = time.time()
    rounds, per_round = 4, 10
    with torch.no_grad():
        run(5)
        mid = args.workload == 'sdxl70'
        # un-hooked and hooked forwards in alternating rounds (host jitter and clock drift hit both sides alike); the
        # figure is the difference of the medians over all forwards of each side
        unhooked_ts, hooked_ts = [], []
        for _ in range(rounds):
            unhooked_ts += forwards(per_round)
            with trace(pipe, launch='step', locate_middle_block=mid) as tc:
                run(3)
                hooked_ts += forwards(per_round)
                tc.synchronize()
        base, res = median(unhooked_ts), {'step': median(hooked_ts)}
        for mode in ('overlap', 'layer'):
            with trace(pipe, launch=mode, locate_middle_block=mid) as tc:
                run(5)
                res[mode] = run(n)
                tc.synchronize()
        # the same comparison with the forward replayed from a CUDA graph (no host launch cost on either side)
        def graphed():
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                pipe.unet(lat, t_dev, emb)
            ts = []
            for _ in range(3):
                g.replay()
            for _ in range(n):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                g.replay()
                b.record()
                ts.append((a, b))
            torch.cuda.synchronize()
            ts = sorted(a.elapsed_time(b) for a, b in ts)
            return ts[len(ts) // 2]

        gres = {}
        try:
            gres['unhooked'] = graphed()
            with trace(pipe, locate_middle_block=mid) as tc:
                run(2)                       # eager steps allocate the slabs before capture
                gres['hooked'] = graphed()
                tc.synchronize()
        except Exception as e:
            gres['error'] = repr(e)
    windows.append((t0, time.time()))
    graph = {}
    if 'hooked' in gres:
        graph = {'graph_unhooked_ms_per_step': round(gres['unhooked'], 4), 'graph_hooked_ms_per_step': round(gres['hooked'], 4),
                 'graph_overhead_pct': round(100 * (gres['hooked'] - gres['unhooked']) / gres['unhooked'], 3)}
    elif 'error' in gres:
        graph = {'graph_error': gres['error']}
    return {**graph, 'unhooked_ms_per_step': round(base, 4),
            'hooked_ms_per_step': round(res['step'], 4), 'overhead_ms_per_step': round(res['step'] - base, 4),
            'overhead_pct': round(100 * (res['step'] - base) / base, 3),
            'hooked_layer_mode_ms_per_step': round(res['layer'], 4),
            'hooked_overlap_mode_ms_per_step': round(res['overlap'], 4),
            'model': f'{spec.name} full-body synthetic UNet, CFG batch 2, {str(dtype).split(".")[-1]}, medians of '
                     f'{rounds * per_round} un-hooked and {rounds * per_round} hooked forwards in {rounds} alternating rounds'}


def pick_cpu_threads(step_fn, budget_s=20.0):
    """Give the CPU arm its best shot: torch's intra-op pool at the thread count that runs one step of the path fastest
    on this box. Candidates stop at 32 threads (the path's ops are small: on the many-core GPU hosts 64+ threads only
    lose time to oversubscription -- 16 of 128 won in round 1) and the probe stops at `budget_s` of wall clock."""
    cores = os.cpu_count() or 1
    cands = sorted({min(c, cores) for c in (8, 16, 32)})
    best, best_t, t_start = cands[0], float('inf'), time.time()
    for c in cands:
        torch.set_num_threads(c)
        if c == cands[0]:
            step_fn()                  # first touch: page in weights, start the pool
        t = time.time()
        step_fn()
        dt = time.time() - t
        if dt < best_t:
            best, best_t = c, dt
        if time.time() - t_start > budget_s:
            break
    torch.set_num_threads(best)
    return best


def leg_cpu_baseline(layers, budget_s=12.0):
    """Oracle port of the hot-path stages on the host cores: baddbmm+softmax (a3), unravel (a4), per-head update (a6)."""
    from oracle import daam_oracle as O
    g = torch.Generator().manual_seed(0)
    qs = [torch.randn(2, hw, h * d, generator=g) for hw, h, d in layers]
    ks = [torch.randn(2, TOKENS, h * d, generator=g) for hw, h, d in layers]
    store = O.OracleHeatMaps()

    def one_step():
        for i, ((hw, h, d), q, k) in enumerate(zip(layers, qs, ks)):
            maps = O.port_layer_step(q, k, h, d ** -0.5)
            for head, m in enumerate(maps):
                store.update(1, i, head, m)

    pick_cpu_threads(one_step)
    one_step()
    t0, n = time.time(), 0
    while True:
        one_step()
        n += 1
        if time.time() - t0 > budget_s or n >= 2000:
            break
    dt = time.time() - t0
    return {'value': px_per_step(layers) * n / dt, 'unit': UNIT, 'cores': torch.get_num_threads(), 'kind': 'port',
            'sample': f'{n} steps x {len(layers)} layers of the same Q/K shapes, fp32 (reference CPU dtype), '
                      f'stages a3+a4+a6 (oracle/daam_oracle.py port_layer_step + update), {dt:.1f} s'}


# --------------------------------------------------------------------------------------------------------------------
# reference arm
# --------------------------------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference's own hook path through the pipeline API (`oracle/` is the only thing executed: OracleTrace, the
    op-for-op port of daam/trace.py's hooks that tests/test_oracle_vs_reference.py pins bit-equal to the verbatim
    reference). Default: on this box's host cores in fp32 -- the contract's reference arm. ``--ref-device cuda`` runs
    the same torch-eager reference hooks on the GPU in the pipeline dtype instead (what a user of the reference gets on
    this box; a secondary figure recorded under profiles/, never what the driver's ratio is built on)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from daam_b200.testing.synthetic import make_pipeline
    from oracle import daam_oracle as O
    spec, layers = workload_spec(args.workload), traced_layers(args.workload)
    on_gpu = args.ref_device == 'cuda'
    dtype = {'bf16': torch.bfloat16, 'fp16': torch.float16, 'fp32': torch.float32}[args.dtype] if on_gpu else torch.float32
    pipe = make_pipeline(spec, body='skeleton', dtype=dtype, device=args.ref_device, seed=0, init_on_device=on_gpu)
    prompts = ['a photo of a dog chasing a red ball on the beach at sunset'] * args.prompts
    if args.prompts != 1:
        raise SystemExit('the reference traces one prompt per generation (daam/trace.py:172-173): use --prompts 1')
    prompt = prompts[0]
    budget = 150.0
    sync = torch.cuda.synchronize if on_gpu else (lambda: None)
    kwargs = {'locate_middle_block': True} if args.workload == 'sdxl70' else {}
    with torch.no_grad(), O.OracleTrace(pipe, **kwargs) as ot:
        if not on_gpu:
            pick_cpu_threads(lambda: pipe(prompt, num_inference_steps=1))
        t = time.time()
        pipe(prompt, num_inference_steps=1)
        ot.compute_global_heat_map()
        sync()
        step_cost = time.time() - t
        warm = min(args.warmup, max(0, int(20.0 / step_cost) - 1))
        if warm:
            pipe(prompt, num_inference_steps=warm)
        steps = max(1, min(args.steps, int(budget / step_cost)))
        sync()
        t0 = time.time()
        pipe(prompt, num_inference_steps=steps)
        sync()
        t_steps = time.time() - t0
        maps = ot.compute_global_heat_map().cpu()
        dt = time.time() - t0
    assert torch.isfinite(maps.float()).all()
    ms = dt / steps * 1e3
    value = px_per_step(layers) * steps / dt
    where = (f'on the GPU ({torch.cuda.get_device_name(0)}, torch eager, {args.dtype})' if on_gpu
             else f'on {torch.get_num_threads()} host threads, fp32')
    sample = (f'{steps} of the requested {args.steps} steps (bounded to ~{budget:.0f} s; the path has no step-dependent '
              f'cost) of the {spec.name} cross-attention skeleton {where} through OracleTrace (port of '
              f'daam/trace.py hooks), + one compute_global_heat_map; hooked forward {t_steps / steps * 1e3:.1f} ms/step')
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': args.dtype if on_gpu else 'f32', 'data': 'synthetic',
        'config': shared_config(args, layers, int(os.environ.get('WORLD_SIZE', '1'))),
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': 0 if on_gpu else torch.get_num_threads(),
                         'kind': 'port', 'sample': sample, 'device': args.ref_device, 'steps_timed': steps},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    emit(line)


DUMP_BYTES = 63_000_000   # data of all dumped arrays together, .npy headers aside: under 64 MB


def dump_outputs(out_dir, arrays):
    """Writes each tensor of ``arrays`` (name -> tensor) as ``<out_dir>/<name>.npy`` in float32. When they exceed
    DUMP_BYTES together, each is replaced by the same share of its elements at positions drawn from a fixed seed (the
    same positions on every run), flattened."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = sum(t.numel() for t in arrays.values()) * 4
    share = min(1.0, DUMP_BYTES / total)
    for i, (name, t) in enumerate(arrays.items()):
        t = t.detach().float()
        if share < 1.0:
            idx = torch.randint(t.numel(), (int(t.numel() * share),), generator=torch.Generator().manual_seed(i))
            t = t.flatten()[idx.sort().values.to(t.device)]
        np.save(os.path.join(out_dir, f'{name}.npy'), t.cpu().numpy())
    log(f'[bench] wrote {len(arrays)} arrays to {out_dir}' + (f' ({share:.3f} of each, seeded sample)' if share < 1 else ''))


def workload_spec(workload):
    from daam_b200.testing.synthetic import SD15_SPEC, SD21_768_SPEC, SD21_SPEC, SDXL_SPEC
    return {'sd21': SD21_SPEC, 'sd21_768': SD21_768_SPEC, 'sdxl': SDXL_SPEC, 'sdxl70': SDXL_SPEC, 'sd15': SD15_SPEC}[workload]


def workload_name(args):
    base = {'sd15': 'random-init SD-1.5 UNet shapes (8 heads, head dims 40/80/160), 64x64 latent, 77 tokens, 15 traced '
                    'cross-attn layers/step',
            'sd21': 'random-init SD-2.1-base UNet shapes, 64x64 latent, 77 tokens, 15 traced cross-attn layers/step',
            'sd21_768': 'random-init SD-2.1 (768-pixel) UNet shapes, 96x96 latent, 77 tokens, 15 traced cross-attn layers/step',
            'sdxl': 'random-init SDXL UNet shapes, 128x128 latent, 77 tokens, 60 traced cross-attn layers/step',
            'sdxl70': 'random-init SDXL UNet shapes, 128x128 latent, 77 tokens, all 70 cross-attn layers traced/step '
                      '(mid block included)'}
    return f'{base[args.workload]}, {args.prompts} prompt(s)/GPU, {args.dtype}'


def value_sets(layers, prompts):
    set_bytes = algorithmic_bytes_per_step(layers, prompts) - px_per_step(layers, prompts) * 4   # accumulators once
    return max(2, -(-int(320e6) // max(1, set_bytes))), set_bytes


def shared_config(args, layers, world):
    """The `config` object: identical for both arms of a run (the reference arm runs `on your arm's config`)."""
    n_sets, set_bytes = value_sets(layers, args.prompts)
    return {
        'workload': workload_name(args), 'px_per_step': px_per_step(layers, args.prompts),
        'px_definition': 'sum over traced layers of heads*77*h*w',
        'literal_px_per_step': literal_px_per_step(layers, args.prompts),
        'l2': f'inputs larger than L2: steps rotate over {n_sets} resident prompt sets '
              f'({n_sets * set_bytes / 1e6:.0f} MB of accumulators+Q/K vs 126 MB L2), no flush',
        'launch': 'one persistent kernel per step per pack of <= 32 traced layers',
        'timing': f'value: K={args.steps} steps between barrier+synchronize, CUDA events, max over ranks; launches '
                  f'queued behind a spin kernel so host pacing is not timed',
        'parallelism': f'prompts sharded, dp{world}',
    }


# --------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50)       # BASELINE configs[1]: 50 denoising steps
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='daam_b200', choices=['daam_b200', 'reference'])
    ap.add_argument('--workload', default='sd21', choices=['sd21', 'sd21_768', 'sdxl', 'sdxl70', 'sd15'])
    ap.add_argument('--prompts', type=int, default=1, help='prompts per GPU traced together (batch_prompts mode)')
    ap.add_argument('--dtype', default=None, choices=['bf16', 'fp16', 'fp32'])
    ap.add_argument('--ref-device', default='cpu', choices=['cpu', 'cuda'],
                    help='--impl reference only: where the reference hooks run (cpu = the contract\'s reference arm)')
    ap.add_argument('--skip-overhead', action='store_true')
    ap.add_argument('--skip-cpu', action='store_true')
    ap.add_argument('--skip-eager', action='store_true', help='skip the eager (no CUDA graph) e2e leg')
    ap.add_argument('--skip-e2e', action='store_true', help='kernel legs only (profiling runs)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what they computed as DIR/<name>.npy (float32, <= 64 MB): the '
                         'accumulators of the last timed step\'s prompt set and the e2e leg\'s heat maps (rank 0)')
    args = ap.parse_args()
    if args.dump_outputs and args.impl != 'daam_b200':
        ap.error('--dump-outputs writes the outputs of --impl daam_b200')
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dtype is None:   # sd15: the reference's default load
        args.dtype = {'sd21': 'bf16', 'sd21_768': 'bf16', 'sdxl': 'fp16', 'sdxl70': 'fp16', 'sd15': 'fp32'}[args.workload]
    args.warmup = max(3, args.warmup)
    capture_stdout()

    if args.impl == 'reference':
        run_reference(args)
        return

    from daam_b200 import _native
    dtype = {'bf16': torch.bfloat16, 'fp16': torch.float16, 'fp32': torch.float32}[args.dtype]
    spec = workload_spec(args.workload)
    layers = traced_layers(args.workload)
    D = Dist(args.gpus)
    _native.load()
    sampler = ClockSampler(D.local_rank) if D.rank == 0 else None
    windows = []

    with torch.no_grad():
        ms, launches, n_sets, value_stats, last_accs = leg_value(args, layers, dtype, D, windows)
        outputs = {f'accumulator_layer{i:02d}': acc for i, acc in enumerate(last_accs)}
        e2e_ms = eager_ms = float('nan')
        h2d = d2h = 0
        order = None
        if not args.skip_e2e:
            e2e_ms, h2d, d2h, order, outputs['e2e_heat_maps'] = leg_e2e(args, spec, dtype, D, windows, cuda_graph=True)
            if not args.skip_eager:
                eager_ms = leg_e2e(args, spec, dtype, D, windows, cuda_graph=False)[0]
        if args.dump_outputs and D.rank == 0:
            dump_outputs(args.dump_outputs, outputs)
        del outputs, last_accs
        overhead = None
        if not args.skip_overhead:       # every rank measures its own GPU (all ranks share the host's cores)
            try:
                overhead = leg_hook_overhead(args, spec, dtype, windows)
            except Exception as e:   # reported, never silently dropped
                overhead = {'error': repr(e)}
            if D.world > 1 and 'overhead_ms_per_step' in overhead:
                worst = torch.tensor([overhead['overhead_ms_per_step'], overhead['hooked_ms_per_step'],
                                      overhead['unhooked_ms_per_step']], dtype=torch.float64, device='cuda')
                D.dist.all_reduce(worst, op=D.dist.ReduceOp.MAX)
                overhead['max_over_ranks'] = {'overhead_ms_per_step': round(float(worst[0]), 4),
                                              'hooked_ms_per_step': round(float(worst[1]), 4),
                                              'unhooked_ms_per_step': round(float(worst[2]), 4), 'ranks': D.world}
    D.barrier()
    if D.rank != 0:
        D.close()
        return
    clocks = sampler.stop(windows)
    cpu = None
    if not args.skip_cpu and D.world == 1:
        cpu = leg_cpu_baseline(layers)

    n = D.world
    px = px_per_step(layers, args.prompts)
    esize = 4 if args.dtype == 'fp32' else 2
    bytes_step = algorithmic_bytes_per_step(layers, args.prompts, esize)
    peak, peak_src = measured_peak()
    achieved = bytes_step / (ms / args.steps * 1e-3) / 1e9        # GB/s per GPU (per-rank launch duration, max over ranks)
    traffic = recorded_traffic(args.workload) if args.dtype == 'bf16' and args.prompts == 1 else None
    e2e = None
    if not args.skip_e2e:
        e2e = {'value': px * args.steps * n / (e2e_ms * 1e-3), 'unit': UNIT, 'h2d_bytes_per_step': h2d,
               'd2h_bytes_per_step': d2h, 'ms_per_step': e2e_ms / args.steps,
               'eager_value': None if args.skip_eager else px * args.steps * n / (eager_ms * 1e-3),
               'eager_ms_per_step': None if args.skip_eager else eager_ms / args.steps,
               'what': 'with trace(pipe): pipe(prompt, K steps) on the cross-attn skeleton UNet (to_q/to_k/to_v, SDPA, '
                       'to_out + fused heat-map kernel), pinned-host inputs H2D every step, + compute_global_heat_map '
                       '(+ all_gather when N>1) + D2H of the maps; the pipeline replays the step from a CUDA graph '
                       '(eager_*: same without graph replay, host-launch bound)'}
        if order is not None:
            e2e['gather_order_check'] = order
        if overhead and 'hooked_ms_per_step' in overhead:
            # the hook-overhead half of the metric, on the FULL-cost UNet (resnets, self-attention, feed-forward):
            # un-hooked vs hooked forward, and the px/s a full-body generation sustains at that step time
            worst = overhead.get('max_over_ranks', overhead)
            e2e['hook_overhead'] = {
                'unhooked_ms_per_step': worst['unhooked_ms_per_step'], 'hooked_ms_per_step': worst['hooked_ms_per_step'],
                'overhead_ms_per_step': worst['overhead_ms_per_step'],
                'overhead_pct': round(100 * worst['overhead_ms_per_step'] / worst['unhooked_ms_per_step'], 3),
                'graph_overhead_pct': overhead.get('graph_overhead_pct'), 'ranks': n,
                'full_body_value': px * n / (worst['hooked_ms_per_step'] * 1e-3), 'model': overhead.get('model')}
    line = {
        'metric': METRIC, 'value': px * args.steps * n / (ms * 1e-3), 'unit': UNIT, 'n_gpus': n, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': args.dtype, 'data': 'synthetic',
        'config': shared_config(args, layers, n),
        'clocks': clocks,
        'e2e': e2e,
        'gpu_launches': launches,
        'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                     'traffic': traffic.get('steady') if isinstance(traffic, dict) else traffic,
                     'traffic_isolated_launch': traffic.get('isolated') if isinstance(traffic, dict) else None,
                     'traffic_note': traffic.get('note') if isinstance(traffic, dict) else None,
                     'kernel': 'daam accumulate (softmax(QK^T)->unravel->+=)',
                     'algorithmic_bytes_per_launch': bytes_step, 'peak_source': peak_src,
                     'timing': value_stats},
        'cpu_baseline': cpu,
        'hook_overhead': overhead,
    }
    emit(line)
    D.close()


if __name__ == '__main__':
    main()
