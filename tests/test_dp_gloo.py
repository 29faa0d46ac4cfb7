"""world_size-2 gloo test (CPU) of the data-parallel host logic: per-rank losses with the global
completeness denominator, summed over ranks through FlatGrads.all_reduce, reproduce the
global-batch gradients of the reference loss (oracle)."""
import os
import sys

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, out):
    for p in (ROOT, os.path.join(ROOT, "action-detection_b200")):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from oracle import ssn_oracle as O
    from ssn_b200.dp import FlatGrads, shard_loss_config, completeness_denominator
    torch.manual_seed(0)
    K, M, D, videos = 5, 3, 16, 64            # 64 global videos: int(65.28) = 65 != 2 * int(32.64)
    n = videos * 8
    g = torch.Generator().manual_seed(1)
    course, stpp = torch.randn(n, D, generator=g), torch.randn(n, D * M, generator=g)
    ptype = torch.tensor([0, 1, 1, 1, 1, 1, 1, 2]).repeat(videos)
    target = torch.randint(1, K + 1, (n,), generator=g); target[ptype == 2] = 0
    rtarget = torch.randn(n, 2, generator=g)

    def make_heads():
        gg = torch.Generator().manual_seed(2)
        return [torch.nn.Parameter(torch.randn(s, generator=gg) * 0.3) for s in ((K + 1, D), (K + 1,), (K, D * M), (K,), (2 * K, D * M), (2 * K,))]

    def loss_of(hp, rows, comp_denom=None):
        F = torch.nn.functional
        ra = F.linear(course[rows], hp[0], hp[1]); rc = F.linear(stpp[rows], hp[2], hp[3])
        rr = F.linear(stpp[rows], hp[4], hp[5]).view(-1, K, 2)
        pt, tg, rt = ptype[rows], target[rows], rtarget[rows]
        ai = ((pt == 0) | (pt == 2)).nonzero().view(-1); ci = ((pt == 0) | (pt == 1)).nonzero().view(-1); ri = (pt == 0).nonzero().view(-1)
        la = F.cross_entropy(ra[ai], tg[ai])
        lr = O.classwise_regression_loss(rr[ri], tg[ri], rt[ri])
        if comp_denom is None:
            lc = O.completeness_loss(rc[ci], tg[ci], 1, 7)
        else:   # same OHEM selection, explicit denominator (what ssnb_heads_cfg.comp_denom carries)
            c3 = rc[ci].view(-1, 7, K); l3 = tg[ci].view(-1, 7)
            pos = O.OHEMHingeLoss.apply(c3[:, :1].reshape(-1, K), l3[:, :1].reshape(-1), 1, 1.0, 1)
            neg = O.OHEMHingeLoss.apply(c3[:, 1:].reshape(-1, K), l3[:, 1:].reshape(-1), -1, 0.17, 6)
            lc = (pos + neg) / comp_denom
        return la + 0.1 * lc + 0.1 * lr

    # global reference
    ref = make_heads()
    loss_of(ref, torch.arange(n)).sum().backward()
    # sharded: rank r owns videos [r*V/2, (r+1)*V/2)
    hp = make_heads()
    fg = FlatGrads(hp, "cpu")
    per = n // world
    comp_denom, scale = shard_loss_config(videos, world)
    assert completeness_denominator(videos) == 129 and comp_denom == 64.5   # 2 * (32 + int(32.64)) = 128 would be wrong
    (loss_of(hp, torch.arange(rank * per, (rank + 1) * per), comp_denom) * scale).sum().backward()
    fg.all_reduce()
    err = max(float((a.grad - b.grad).abs().max() / (b.grad.abs().max() + 1e-12)) for a, b in zip(hp, ref))
    out[rank] = err
    dist.destroy_process_group()


def free_port():
    """a TCP port nothing on this host listens on (a fixed one can be taken by another job on a shared host)"""
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_dp_two_ranks_match_global_batch():
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, free_port(), out), nprocs=world, join=True)
    assert len(out) == world
    for r in range(world):
        assert out[r] < 1e-5, dict(out)
