"""H-sharded single-pair mode on the GPU (hshard.hot_path_steps): N virtual ranks on one device against the un-sharded
forward of the same network and against the oracle; with >= 2 GPUs also one process per GPU over both transports
(first green on B200: round 2, 1 and 2 GPUs).  The plan itself is verified on CPU in test_hshard_plan.py."""
import os

import pytest
import torch

pytestmark = [pytest.mark.gpu]


@pytest.mark.parametrize("world", [2, 3])
def test_virtual_ranks_match_unsharded_forward_and_oracle(world):
    import dcanet_b200 as d
    from oracle import dcanet_oracle as O
    hs = d.hshard
    maxdisp, H4, W4 = 48, 24, 40
    feats = O.synth_features(0, 1, H4, W4, shift=2)
    sd = O.calibrate_state_dict(O.synth_state_dict(0), feats, maxdisp)
    with torch.no_grad():
        ref4, refpv = O.hot_path(sd, *feats, maxdisp=maxdisp)
    net = d.GwcNet(maxdisp)
    own = net.state_dict()
    own.update(sd)
    net.load_state_dict(own)
    net = net.cuda().eval()
    dev = [f.cuda() for f in feats]
    with torch.no_grad():
        full4, fullpv = net.hot_path(*dev)
        sh4, shpv = hs.hot_path_forward_virtual(net.packed(), *dev, world=world)
    torch.cuda.synchronize()
    assert sh4.shape == full4.shape and shpv.shape == fullpv.shape
    # same kernels on row slabs; only the summation order of S[b,k] and the tile decomposition differ
    assert float((sh4 - full4).abs().max()) <= 0.01
    err = (sh4.cpu() - ref4).abs()
    assert float(err.max()) <= 0.05 and float(err.mean()) <= 0.01          # north_star tolerance
    assert float((shpv.cpu() - refpv).abs().max()) <= 1e-3


def _rank_main(rank, world, port, transport, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    import dcanet_b200 as d
    from oracle import dcanet_oracle as O
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    maxdisp, H4, W4 = 48, 24, 40
    feats = O.synth_features(0, 1, H4, W4, shift=2)
    sd = O.calibrate_state_dict(O.synth_state_dict(0), feats, maxdisp)
    net = d.GwcNet(maxdisp)
    own = net.state_dict()
    own.update(sd)
    net.load_state_dict(own)
    net = net.cuda().eval()
    mine = [d.hshard.owned_rows(f, world, rank).cuda() for f in feats]
    with torch.no_grad():
        for _ in range(3):               # several forwards: staging parity and the arrival counters carry over
            pred4, pv = net.hot_path_hsharded(*mine, rank=rank, world=world, transport=transport)
        for peer in d.hshard._PEERS.values():
            peer.check()
        full4, fullpv = net.hot_path(*[f.cuda() for f in feats])
    torch.cuda.synchronize()
    want4 = d.hshard.owned_rows(full4, world, rank, dim=2, scale=4)
    q.put((rank, float((pred4 - want4).abs().max())))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("transport", ["nccl", "p2p"])
def test_two_gpus_match_unsharded_forward(transport):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import socket
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_main, args=(r, 2, port, transport, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for rank, err in res:
        assert err <= 0.01, (rank, err)
