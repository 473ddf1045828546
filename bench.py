"""bench.py — tiles/s (and 4K images/s) of the PatchFusion hot path, Depth-Anything-vitl, 4K, P49 (cai_mode m2).

    python bench.py --gpus 1 --steps K --warmup W                      (this build, CUDA path through the C ABI)
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...                               (reference algorithm on the host cores)
    python bench.py ... --dump-outputs DIR          (also save the last timed step's depth canvas as DIR/depth.npy)

A step = one pass of the hot path over one synthetic 4K image per rank: coarse branch + G2L once, 49 tiles through
fine branch + guided fusion, stitch.  `value`: ranks process independent images (weak scaling, no data-path
collective).  `tile_sharded`: a second timed region where ONE image's tiles are sharded over the ranks with a single
NCCL all-gather of the per-rank prediction blocks (strong scaling of one image, BASELINE configs[2]).
Prints ONE JSON line (rank 0).
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

F_TILE = {'vits': 360.0e9, 'vitb': 1133.9e9, 'vitl': 4029.8e9}     # algorithmic FLOPs / tile   (BASELINE.md §2)
F_IMAGE = {'vits': 139.5e9, 'vitb': 404.1e9, 'vitl': 1343.5e9}     # coarse + G2L once per image


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tflops_sustained=d['bf16_tflops_sustained'], tflops_burst=d['bf16_tflops'], hbm=d['hbm_gbs'],
                    source='measured (MEASURED_PEAKS.json)')
    return dict(tflops_sustained=1400.0, tflops_burst=1590.0, hbm=6650.0, source='fallback (B200_PROFILING.md)')


class ClockSampler:
    QUERY = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(['nvidia-smi', '-i', str(index), '--query-gpu=' + self.QUERY,
                                       '--format=csv,noheader,nounits', '-lms', '200'], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None
        atexit.register(self._kill)         # a run that fails before stop() must not leave nvidia-smi polling

    def _kill(self):
        if self.p is not None and self.p.poll() is None:
            self.p.kill()

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[])
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(', ') for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, reasons = [], set()
        for r in rows:
            try:
                sm.append(float(r[1]))
                out['sm_max_mhz'] = float(r[2])
                for name, v in zip(['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'], r[4:8]):
                    if v.strip().lower().startswith('active'):
                        reasons.add(name)
            except Exception:
                pass
        if sm:
            sm.sort()
            out['sm_mhz'] = sm[len(sm) // 2]
        out['reasons'] = sorted(reasons)
        return out


def build_inputs(encoder, seed=0):
    from patchfusion_b200.configs import depth_anything_patchfusion
    from patchfusion_b200.params import synthetic_state_dict
    cfg = depth_anything_patchfusion(encoder, image_raw_shape=(2160, 3840), patch_split_num=(4, 4))
    sd = synthetic_state_dict(cfg, seed=seed)
    return cfg, sd


def _cpu_tile_runner(encoder, cfg, sd):
    """oracle state for timing single tiles of the 4K P49 workload on the host (fixed per-image work done once)."""
    from oracle import pf_oracle as po
    g = torch.Generator().manual_seed(1)
    img = torch.rand(1, 3, 2160, 3840, generator=g)
    orc = po.Oracle(sd, cfg)
    P = cfg['patch_process_shape']
    tc = po.prepare_tile_cfg((2160, 3840), (4, 4), P)
    st = {}

    def fixed():
        with torch.no_grad():
            lr = orc.resizer(img)
            t0 = time.time()
            st['cd'], st['cf'] = orc.coarse(lr)
            st['g2l'] = po.g2l_all(sd, st['cf'], cfg['guided_fusion'])
            return time.time() - t0

    def tile(r):
        with torch.no_grad():
            t0 = time.time()
            orc.tiles(img, [(540 * (r % 4), 960)], st['cd'], st['cf'], st['g2l'], 1, tc)
            return time.time() - t0

    return fixed, tile


def pick_threads(tile, candidates=None):
    """torch CPU kernels stop scaling (and regress) well before all threads on these hosts: time ONE WHOLE TILE (fine
    branch + fusion) at 32 / 64 / all threads after a warm-up tile and keep the fastest."""
    n = os.cpu_count() or 8
    cands = sorted(set(min(n, c) for c in (candidates or (32, 64, n))))
    torch.set_num_threads(cands[0])
    tile(0)                                     # warm-up (oneDNN primitive creation, allocator)
    best, best_t, probe = cands[0], None, {}
    for t in cands:
        torch.set_num_threads(t)
        dt = tile(1)
        probe[t] = dt
        if best_t is None or dt < best_t:
            best, best_t = t, dt
    return best, probe


def cpu_baseline(encoder, cfg, sd, threads=None, reps=1, n_tiles=49):
    """The oracle (a port of the reference algorithm) on the host cores: the per-image fixed work (coarse branch +
    G2L) once, then `reps` micro-batches of ONE tile (fine branch + fusion); bounded sample, not the product path.
    value = the P49-image-equivalent rate n_tiles / (t_fixed + n_tiles * t_tile)."""
    fixed, tile = _cpu_tile_runner(encoder, cfg, sd)
    torch.set_num_threads(min(os.cpu_count() or 8, 64))
    t_fixed = fixed()
    probe = None
    if threads is None:
        threads, probe = pick_threads(tile)
    torch.set_num_threads(threads)
    ts = [tile(2 + r) for r in range(reps)]
    t_tile = sum(ts) / len(ts)
    value = n_tiles / (t_fixed + n_tiles * t_tile)
    return dict(value=value, unit='tiles/s', cores=threads, kind='port',
                sample='%s: per-image fixed work (coarse + G2L) once = %.1f s, then %d x 1 tile (fine branch + fusion, '
                       'p=1) of the 4K P%d workload on %d of %d host threads (whole-tile probe %s); value = %d / (fixed '
                       '+ %d x mean tile time)' % (encoder, t_fixed, reps, n_tiles, threads, os.cpu_count(),
                                                    {k: round(v, 2) for k, v in (probe or {}).items()}, n_tiles, n_tiles),
                s_per_tile=t_tile, s_fixed_per_image=t_fixed, tile_times=ts)


def gpu_eager_baseline(encoder, cfg, sd, dev, n_tiles=49):
    """The reference algorithm (oracle port) in eager PyTorch on ONE B200 with the reference's own GPU flags
    (`estimator/utils/misc.py:24-26`: cudnn.benchmark=True; torch defaults otherwise = true-fp32 matmul, TF32 cuDNN
    convolutions): coarse + G2L once, then the 16 tiles of the first regular pass in micro-batches of 4 (the
    reference's default process_num).  G2L is hoisted out of the micro-batch loop (the reference recomputes it per
    micro-batch), so this baseline is FASTER than the real reference."""
    from oracle import pf_oracle as po
    old = (torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32 = True, True
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        sdc = {k: v.to(dev) for k, v in sd.items()}
        orc = po.Oracle(sdc, cfg)
        img = torch.rand(1, 3, 2160, 3840, generator=torch.Generator().manual_seed(1)).to(dev)
        P = cfg['patch_process_shape']
        tc = po.prepare_tile_cfg((2160, 3840), (4, 4), P)
        raws = [t[0] for t in po.tile_plan(tc, P, 'm1')[0]]

        def timed(fn):
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn()
            e1.record()
            torch.cuda.synchronize(dev)
            return e0.elapsed_time(e1) / 1e3, r

        with torch.no_grad():
            lr = orc.resizer(img)

            def fixed():
                cd, cf = orc.coarse(lr)
                return cd, cf, po.g2l_all(sdc, cf, cfg['guided_fusion'])

            fixed()                                             # warm-up (cudnn.benchmark autotuning)
            t_fixed, (cd, cf, g2l) = timed(fixed)
            orc.tiles(img, raws[:4], cd, cf, g2l, 4, tc)        # warm-up micro-batch
            t_tiles, _ = timed(lambda: orc.tiles(img, raws, cd, cf, g2l, 4, tc))
        t_tile = t_tiles / len(raws)
        return dict(value=n_tiles / (t_fixed + n_tiles * t_tile), unit='tiles/s', kind='port (oracle on cuda, eager)',
                    flags='cudnn.benchmark=True, cudnn.allow_tf32=True (TF32 convs), matmul fp32',
                    sample='coarse + G2L once (%.3f s) + 16 tiles (m1 pass) in micro-batches of 4 (%.3f s); value = '
                           '%d / (fixed + %d x s_per_tile), G2L hoisted' % (t_fixed, t_tiles, n_tiles, n_tiles),
                    s_per_tile=t_tile, s_fixed_per_image=t_fixed, p16_images_per_s=1.0 / (t_fixed + t_tiles))
    finally:
        torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
        torch.cuda.empty_cache()


def dram_traffic(kernel_key):
    """DRAM bytes per output pixel of the dominant launch shape, from the ncu --set full capture summarised under
    profiles/ by tools/summarize_profiles.py (profiles/dram_traffic.json); None when no capture is committed."""
    p = os.path.join(ROOT, 'profiles', 'dram_traffic.json')
    if not os.path.exists(p):
        return None, None
    d = json.load(open(p)).get(kernel_key)
    if not d:
        return None, None
    return d['bytes_per_unit'], d.get('source')


def lib_summary(records):
    out = {}
    for fam, label, fl, ms in records:
        d = out.setdefault(fam, dict(ms=0.0, flops=0.0, launches=0))
        d['ms'] += ms
        d['flops'] += fl
        d['launches'] += 1
    return out


def shard_plan_info(model, n_tiles, world):
    """How the single image's tiles were distributed in the tile_sharded region (mirrors PatchFusion.forward)."""
    from patchfusion_b200.parallel import tile_plan, shard_counts, block_rows
    owner = world > 1 and model.shard_coarse == 'owner'
    plan = tile_plan(n_tiles, world, model.owner_cost_tiles) if owner else None
    rows = block_rows(n_tiles, world, plan)
    coll = '1 all_gather_into_tensor of [%d, 392, 518] fp32 prediction blocks per image' % rows
    if owner:
        coll = '1 broadcast of rank 0\'s packed coarse depth + 6 coarse maps + 6 G2L maps, then ' + coll
    return dict(coarse_stage='rank 0 computes + broadcasts, takes %.1f tiles less' % model.owner_cost_tiles if owner
                else 'replicated on every rank', tiles_per_rank=shard_counts(n_tiles, world, plan),
                collective=coll, tiles_on_busiest_rank=rows)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--encoder', default='vitl')
    ap.add_argument('--cai-mode', default='m2')
    ap.add_argument('--process-num', type=int, default=9)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--profile', action='store_true', help='per-kernel-family time table to stderr')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the depth canvas of the last timed step (rank 0) to DIR/depth.npy, float32')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs needs --impl b200')
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    # torchrun pins OMP_NUM_THREADS=1: give the host-side weight synthesis / packing a fair share of the cores
    torch.set_num_threads(max(1, min(16, (os.cpu_count() or 8) // max(world, 1))))
    enc = args.encoder
    n_tiles = {'m1': 16, 'm2': 49}[args.cai_mode]
    workload = 'Depth-Anything-%s PatchFusion, 4K (2160x3840), P%d (%s, 4x4 split), %d image/rank/step' % (
        enc, n_tiles, args.cai_mode, 1)

    if args.impl == 'reference':
        if rank != 0:
            return
        cfg, sd = build_inputs(enc)
        warm = 2                            # CPU: the thread probe runs a warm-up tile + one tile per candidate count
        cb = cpu_baseline(enc, cfg, sd, reps=args.steps, n_tiles=n_tiles)
        ms = cb['s_per_tile'] * 1e3
        v = cb['value']
        print(json.dumps(dict(
            impl='reference', metric='tiles/s', value=v, unit='tiles/s', n_gpus=args.gpus, steps=args.steps,
            warmup=warm, ms_per_step=ms, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32',
            data='synthetic', config=dict(workload=workload, note='each step = 1 tile (bounded sample) on host cores; '
                                          'value includes the per-image fixed work amortised over the image'),
            cpu_baseline=cb, e2e=dict(value=v, unit='tiles/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0),
            gpu_launches=0)))
        return

    # keep stdout clean for the single JSON line: libraries (NCCL's version banner, ...) that write to fd 1 during
    # the run are sent to stderr; the descriptor is restored right before the result is printed
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    from patchfusion_b200 import lib
    from patchfusion_b200.model import PatchFusion
    dev = torch.device('cuda', local)
    torch.cuda.set_device(dev)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=dev)
    cfg, sd = build_inputs(enc)
    model = PatchFusion(cfg)
    model.load_state_dict(sd, strict=True)
    model = model.to(dev).eval()
    g = torch.Generator().manual_seed(100 + rank)
    host_img = torch.rand(1, 3, 2160, 3840, generator=g).pin_memory()
    RH, RW = model.tile_cfg['patch_reensemble_shape']
    host_out = torch.empty((1, 1, RH, RW), dtype=torch.float32).pin_memory()

    def step(img_dev):
        # images-per-rank (weak scaling): independent images, no data-path collective
        lr = model.make_lr(img_dev)
        y, _ = model(mode='infer', image_lr=lr, image_hr=img_dev, cai_mode=args.cai_mode, process_num=args.process_num)
        return y

    local_step = step
    # tiles-per-rank (SURVEY.md §8e, BASELINE configs[2]): ONE image (the same on every rank), tile i -> rank i % world,
    # one all-gather of the per-rank prediction blocks, deterministic stitch on every rank
    shared_img = torch.rand(1, 3, 2160, 3840, generator=torch.Generator().manual_seed(7)).to(dev)

    def sharded_step():
        lr = model.make_lr(shared_img)
        y, _ = model(mode='infer', image_lr=lr, image_hr=shared_img, cai_mode=args.cai_mode,
                     process_num=args.process_num, shard=(rank, world) if world > 1 else None)
        return y

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    img_dev = host_img.to(dev, non_blocking=True)
    for _ in range(max(args.warmup, 3)):
        step(img_dev)

    # end-to-end: every step copies its image from pinned host memory (99.5 MB) and reads its depth canvas back
    # (13 MB).  Plain user-level double buffering around the public call: the H2D of step i+1 runs on a copy stream
    # while step i computes; nothing is skipped and the timed region ends with a full synchronise.
    copy_stream = torch.cuda.Stream()
    dbuf = [torch.empty_like(img_dev) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]
    e2e_i = [0]

    def e2e_step():
        i = e2e_i[0] % 2
        e2e_i[0] += 1
        cur = torch.cuda.current_stream()
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(freed[i])
            dbuf[i].copy_(host_img, non_blocking=True)
            ready[i].record(copy_stream)
        cur.wait_event(ready[i])
        y = step(dbuf[i])
        freed[i].record(cur)
        host_out.copy_(y, non_blocking=True)

    sampler = ClockSampler(local) if rank == 0 else None
    last = [None]

    def timed_step():
        last[0] = None                      # free the previous canvas first, as a caller that drops it would
        last[0] = step(img_dev)

    l0 = lib.launch_count() + model.graph_launches
    ms_dev = timed(timed_step, args.steps)
    launches = lib.launch_count() + model.graph_launches - l0
    depth_out = last[0].cpu() if args.dump_outputs and rank == 0 else None
    last[0] = None
    ms_e2e = timed(e2e_step, args.steps)
    for _ in range(3):
        sharded_step()
    ms_shard = timed(sharded_step, args.steps)
    clocks = sampler.stop() if sampler else {}

    # roofline pass: per-launch CUDA events around every kernel of one more step (not part of the timed value)
    prof_records = None
    if rank == 0:
        lib.PROFILER = lib.Profiler()       # eager, single stream: events inside the library around every launch
        local_step(img_dev)                 # warm the eager path (workspaces, tensor maps)
        torch.cuda.synchronize()
        lib.PROFILER.start()
        local_step(img_dev)                 # no collective here: only rank 0 runs this pass
        torch.cuda.synchronize()
        prof_records = lib.PROFILER.stop()  # (kernel, label, flops, ms)
        lib.PROFILER = None
    barrier()

    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    tiles_per_step = n_tiles * world
    tps = tiles_per_step * args.steps / (ms_dev / 1e3)
    tps_e2e = tiles_per_step * args.steps / (ms_e2e / 1e3)
    if rank != 0:
        return
    pk = peaks()
    fam = lib_summary(prof_records)
    total_ms = sum(v['ms'] for v in fam.values())
    halo = fam.get('pf_conv3_halo_kernel', dict(ms=1e-9, flops=0.0, launches=0))
    gall_ms = halo['ms'] + fam.get('pf_gemm_kernel', dict(ms=0.0))['ms']
    gall_fl = halo['flops'] + fam.get('pf_gemm_kernel', dict(flops=0.0))['flops']
    # dominant kernel = pf_conv3_halo_kernel; its heaviest launch shape = guided_fusion.up_conv_list.4 conv1
    # (3x3, [32,256,256] -> 544 channels @392x518), timed per launch with CUDA events on the launching stream
    big = max((r for r in prof_records if r[0] == 'pf_conv3_halo_kernel'), key=lambda r: r[2])
    same = [r for r in prof_records if r[0] == 'pf_conv3_halo_kernel' and r[2] == big[2]]
    ms_launch = sum(r[3] for r in same) / len(same)
    ach = big[2] / (ms_launch / 1e3) / 1e12
    rows_launch = big[2] / (2.0 * 9 * 544 * 544)
    # DRAM bytes of this launch shape: dram__bytes_read.sum + dram__bytes_write.sum of the committed ncu --set full
    # capture, stored per output pixel in profiles/dram_traffic.json by tools/summarize_profiles.py (None if absent)
    bpp, traffic_src = dram_traffic('pf_conv3_halo_kernel/up_conv_list.4.conv1')
    traffic = bpp * rows_launch if bpp is not None else None
    roof = dict(bound='tensor', achieved=ach, peak=pk['tflops_sustained'], unit='TFLOP/s',
                frac=ach / pk['tflops_sustained'], traffic=traffic, traffic_source=traffic_src,
                kernel='pf_conv3_halo_kernel (tcgen05 halo-tile 3x3 conv; %d launches/step, %.1f%% of step kernel '
                       'time); launch = up_conv_list.4 conv1 [32,256,256]->544 @392x518 x %d tiles, %.3f ms'
                       % (halo['launches'], 100.0 * halo['ms'] / total_ms, round(rows_launch / (392 * 518)), ms_launch),
                algorithmic_bytes=rows_launch * (544 + 544) * 2.0 + 544 * 9 * 576 * 2.0,
                peak_source=pk['source'] + ', sustained bf16',
                all_gemm_tflops=gall_fl / (gall_ms / 1e3) / 1e12, all_gemm_share=gall_ms / total_ms,
                whole_step_tflops=(tps / world * F_TILE[enc] + tps / world / n_tiles * F_IMAGE[enc]) / 1e12)
    prof = fam
    if args.profile:
        # per launch-shape table (label -> launches, ms, TF/s), slowest first
        by = {}
        for f_, lab, fl, ms_ in prof_records:
            d_ = by.setdefault(lab, [0, 0.0, 0.0])
            d_[0] += 1; d_[1] += ms_; d_[2] += fl
        rows_ = sorted(by.items(), key=lambda kv: -kv[1][1])
        for k_, v in rows_:
            sys.stderr.write('%-64s %5d x %8.3f ms %8.1f TF/s\n' % (k_, v[0], v[1], v[2] / max(v[1], 1e-9) / 1e9))
        for k_, v in sorted(prof.items(), key=lambda kv: -kv[1]['ms']):
            sys.stderr.write('%-26s %8.2f ms %6d launches %8.1f TF/s\n' % (k_, v['ms'], v['launches'],
                                                                         v['flops'] / max(v['ms'], 1e-9) / 1e9))
    cb = ge = None
    plan_info = shard_plan_info(model, n_tiles, world)
    if not args.no_cpu_baseline and world == 1:
        del model
        torch.cuda.empty_cache()
        ge = gpu_eager_baseline(enc, cfg, sd, dev, n_tiles=n_tiles)
        cb = cpu_baseline(enc, cfg, sd, reps=1, n_tiles=n_tiles)
    ms_img_single = ms_dev / args.steps                  # one image on one GPU (replica mode, same run)
    ms_img_shard = ms_shard / args.steps
    tile_sharded = dict(ms_per_image=ms_img_shard, tiles_per_s=n_tiles / (ms_img_shard / 1e3), n_gpus=world,
                        single_gpu_ms_per_image=ms_img_single, speedup_vs_single_gpu=ms_img_single / ms_img_shard,
                        efficiency_vs_n1=ms_img_single / ms_img_shard / world,
                        **plan_info)
    out = dict(
        metric='tiles/s', value=tps, unit='tiles/s', n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3),
        ms_per_step=ms_dev / args.steps, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='bf16',
        data='synthetic', images_per_s=tps / n_tiles,
        config=dict(workload=workload, process_num=args.process_num, weights='seeded random init (no checkpoints offline)',
                    l2='working set >> L2: 1.5 GB bf16 weights + ~GBs of activations streamed every step'),
        e2e=dict(value=tps_e2e, unit='tiles/s', h2d_bytes_per_step=host_img.numel() * 4,
                 d2h_bytes_per_step=host_out.numel() * 4),
        gpu_launches=launches, clocks=clocks, roofline=roof, cpu_baseline=cb, gpu_eager_baseline=ge,
        tile_sharded=tile_sharded)
    if depth_out is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, 'depth.npy'), depth_out.numpy())
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(out), flush=True)


if __name__ == '__main__':
    main()
