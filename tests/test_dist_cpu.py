"""world_size-2 gloo run on CPU: frame-sharded processing (refvsr_b200/dist.py) with the input-halo
exchange equals the single-process stream bit for bit."""
import os
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_plan_segments():
    from refvsr_b200.dist import plan_segments
    assert plan_segments(32, 9, 8) == [(0, 9), (9, 18), (18, 27), (27, 32), (32, 32), (32, 32), (32, 32), (32, 32)]
    assert plan_segments(64, 9, 4) == [(0, 18), (18, 36), (36, 54), (54, 64)]
    assert plan_segments(5, 2, 2) == [(0, 4), (4, 5)]
    with pytest.raises(ValueError):
        plan_segments(10, None, 2)


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    torch.set_num_threads(2)
    from oracle.oracle_ops import OracleOps
    from refvsr_b200.dist import exchange_halo, gather_frames, plan_segments, run_sharded
    from util import build_case
    spec, cfg, net, lrs, refs, golden = build_case('small_t3_32x48', 'cpu', ops=OracleOps(), b200_precision='fp32')
    T, n = spec['T'], lrs.shape[0]
    plan = plan_segments(n, cfg.reset_branch, world)
    f0, f1 = plan[rank]
    fl, first = exchange_halo(lrs[f0:f1].clone(), plan, rank, T // 2)      # each rank starts with ITS frames only
    fr, _ = exchange_halo(refs[f0:f1].clone(), plan, rank, T // 2)
    assert torch.equal(fl, lrs[first:first + fl.shape[0]])
    res = list(run_sharded(net, fl, fr, first, (f0, f1), n, T))
    allf = gather_frames(res, plan, rank, (3, 4 * spec['h'], 4 * spec['w']), 'cpu')
    if rank == 0:
        q.put([f.numpy() for f in allf])
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_equals_single_stream():
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    from oracle.oracle_ops import OracleOps
    from refvsr_b200.synth import sliding_windows
    from util import build_case
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    sharded = q.get(timeout=600)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    spec, cfg, net, lrs, refs, golden = build_case('small_t3_32x48', 'cpu', ops=OracleOps(), b200_precision='fp32')
    nthr = torch.get_num_threads()
    torch.set_num_threads(2)          # same as the workers: oneDNN's summation order depends on the thread count
    try:
        single = [net(wl, wr, first)['result'][0].numpy() for k, wl, wr, first in sliding_windows(lrs, refs, spec['T'])]
    finally:
        torch.set_num_threads(nthr)
    assert len(sharded) == len(single) == 4
    for a, b in zip(sharded, single):
        assert np.array_equal(a, b), 'segment-sharded output must be bit identical to the continuous stream'


# ---------------------------------------------------------------------------------------------------------------------
# BASELINE configs[3]: frame sharding finer than the reset segments, forward state handed from rank to rank
# ---------------------------------------------------------------------------------------------------------------------
def test_plan_frames_and_chain_pieces():
    from refvsr_b200.dist import chain_pieces, plan_frames
    plan = plan_frames(32, 8)
    assert plan == [(4 * r, 4 * r + 4) for r in range(8)]                    # all 8 GPUs busy on a 32-frame clip
    assert chain_pieces((0, 4), 9) == [(0, 4, True)]
    assert chain_pieces((8, 12), 9) == [(8, 9, False), (9, 12, True)]       # tail of chain 0, head of chain 1
    assert chain_pieces((16, 20), 9) == [(16, 18, False), (18, 20, True)]
    assert chain_pieces((4, 8), 9) == [(4, 8, False)]
    assert plan_frames(10, 3) == [(0, 4), (4, 7), (7, 10)]


def _frame_worker(rank, world, port, q, reset_branch, nframes):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    torch.set_num_threads(2)
    from oracle.oracle_ops import OracleOps
    from refvsr_b200.dist import exchange_halo, gather_frames, plan_frames, run_clip_frame_sharded
    from refvsr_b200.synth import make_clip
    from util import build_case
    spec, cfg, net, _, _, _ = build_case('small_t7_24x32', 'cpu', ops=OracleOps(), b200_precision='fp32', reset_branch=reset_branch)
    lrs, refs = make_clip(nframes, spec['h'], spec['w'], 1, seed=31)
    T = spec['T']
    plan = plan_frames(nframes, world)
    f0, f1 = plan[rank]
    fl, first = exchange_halo(lrs[f0:f1].clone(), plan, rank, T // 2)
    fr, _ = exchange_halo(refs[f0:f1].clone(), plan, rank, T // 2)
    timing = {}
    res = run_clip_frame_sharded(net, fl, fr, first, plan, rank, timing=timing)
    allf = gather_frames(res, plan, rank, (3, 4 * spec['h'], 4 * spec['w']), 'cpu')
    logs = [None] * world
    dist.all_gather_object(logs, timing.get('log'))
    # after a sharded clip the module serves ordinary windowed calls again
    w0 = net(lrs[[0, 0, 0, 0, 1, 2, 3]].unsqueeze(0), refs[[0, 0, 0, 0, 1, 2, 3]].unsqueeze(0), True)['result']
    if rank == 0:
        q.put(([f.numpy() for f in allf], logs, w0[0].numpy()))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize('world,reset_branch,nframes', [(3, 4, 10), (2, 9, 8)])
def test_frame_sharded_clip_equals_single_stream(world, reset_branch, nframes):
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    from oracle.oracle_ops import OracleOps
    from refvsr_b200.synth import make_clip, sliding_windows
    from util import build_case
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 31500 + (os.getpid() * 7 + world) % 2000
    procs = [ctx.Process(target=_frame_worker, args=(r, world, port, q, reset_branch, nframes)) for r in range(world)]
    for p in procs:
        p.start()
    sharded, logs, w0 = q.get(timeout=900)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    spec, cfg, net, _, _, _ = build_case('small_t7_24x32', 'cpu', ops=OracleOps(), b200_precision='fp32', reset_branch=reset_branch)
    lrs, refs = make_clip(nframes, spec['h'], spec['w'], 1, seed=31)
    nthr = torch.get_num_threads()
    torch.set_num_threads(2)          # same as the workers: oneDNN's summation order depends on the thread count
    try:
        single = [net(wl, wr, first)['result'][0].numpy() for k, wl, wr, first in sliding_windows(lrs, refs, spec['T'])]
        net.Network.reset_state()
        w0_single = net(lrs[[0, 0, 0, 0, 1, 2, 3]].unsqueeze(0), refs[[0, 0, 0, 0, 1, 2, 3]].unsqueeze(0), True)['result'][0].numpy()
    finally:
        torch.set_num_threads(nthr)
    assert len(sharded) == len(single) == nframes
    for k, (a, b) in enumerate(zip(sharded, single)):
        assert np.array_equal(a, b), f'frame {k}: frame-sharded output must be bit identical to the single stream'
    assert np.array_equal(w0, w0_single)
    if world == 3:          # (0,4) head only | (4,7) head, sends | (7,10): head piece [8,10) first, then receives for frame 7
        assert [e[0] for e in logs[0] if e[0] in ('recv', 'send')] == []
        assert ('send', 2) in logs[1] and ('recv', 1) in logs[2]
        kinds2 = [e for e in logs[2] if e[0] in ('forward', 'recv')]
        assert kinds2[0] == ('forward', 8, 10, True) and kinds2[1] == ('recv', 1) and kinds2[2] == ('forward', 7, 8, False)
    else:
        assert ('send', 1) in logs[0] and ('recv', 0) in logs[1]


def _halo_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    sys.path.insert(0, ROOT)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from refvsr_b200.dist import exchange_halo, plan_segments
    plan = plan_segments(5, 9, world)                 # [(0,5), (5,5), (5,5)]: ranks 1 and 2 own nothing (ADVICE r1: used to hang)
    frames = torch.arange(5, dtype=torch.float32).view(5, 1)
    f0, f1 = plan[rank]
    out, first = exchange_halo(frames[f0:f1].clone(), plan, rank, 3)
    q.put((rank, out.flatten().tolist(), first))
    dist.barrier()
    dist.destroy_process_group()


def test_exchange_halo_with_empty_ranks():
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 33500 + os.getpid() % 2000
    procs = [ctx.Process(target=_halo_worker, args=(r, 3, port, q)) for r in range(3)]
    for p in procs:
        p.start()
    got = sorted(q.get(timeout=120) for _ in range(3))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert got[0] == (0, [0.0, 1.0, 2.0, 3.0, 4.0], 0) and got[1][1] == [] and got[2][1] == []
