"""GPU (>= 2 devices): multi-GPU result exchange by peer stores (sharding.PeerResultExchange + the heads epilogue
of the persistent FCN kernel) - after a barrier every rank's gather buffer holds BOTH ranks' decoded results,
bit-identical to a local forward of the same inputs, and the epoch flags count the forwards.
Runs on a machine with two or more GPUs (`python -m pytest tests/test_gpu_peer.py -m gpu`); skipped on one GPU."""
import os
import socket
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, ret):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["FCN_MEGA"] = "1"
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from frustum_convnet_b200 import config, synth
        from frustum_convnet_b200.det_base import PointNetDet
        from frustum_convnet_b200.sharding import PeerResultExchange, pack_outputs
        cfg, w = config.load_workload("car")
        sd = synth.make_state_dict(w["arch"], 3, "KITTI", seed=7)

        def model():
            m = PointNetDet(3, num_vec=3)
            m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()})
            m.precision, m.use_cuda_graph, m.copy_outputs = 1, True, False
            return m.to(dev).eval()

        B, slots = 4, 2
        datas = [synth.make_frustums("car", B, seed=500 + r, max_depth=17.5) for r in range(world)]
        ins = [{k: torch.from_numpy(v).to(dev) for k, v in d.items()} for d in datas]
        T = [datas[0]["center_ref%d" % (i + 1)].shape[2] for i in range(4)]
        m = model()
        eng = m.engine()
        n_blk = B * T[1] * (2 + 3 + 1 + 3 + 12 + 3)
        ex = PeerResultExchange(slots, n_blk, dev)
        streams = [torch.cuda.Stream(device=dev) for _ in range(slots)]
        k_alloc = [0]

        def alloc(n, device):
            v = ex.local_block(k_alloc[0])
            k_alloc[0] += 1
            return v
        eng.out_alloc = alloc
        plans = []
        for st in streams:
            with torch.cuda.stream(st):
                plans.append(eng.plan(B, datas[0]["point_cloud"].shape[2], T))
        eng.out_alloc = None
        for k, pl in enumerate(plans):
            blocks, flags = ex.peer_targets(k)
            pl.set_peer_outputs(blocks, flags)
        nrep = 3
        for rep in range(nrep):
            for k, st in enumerate(streams):
                with torch.cuda.stream(st):
                    m(ins[rank])
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        # local recomputation of every rank's result on a fresh model (no peer outputs)
        m2 = model()
        data_ok = True
        for r in range(world):
            want = pack_outputs([o.clone() for o in m2(ins[r])])
            for k in range(slots):
                data_ok = data_ok and bool(torch.equal(ex.gathered(k)[r], want))
        fl = ex.flags.cpu().numpy()
        # every plan ran nrep replays + the eager warm-up pass of its graph capture
        ret[rank] = (data_ok, fl.tolist(), nrep + 1)
        ex.close()
    finally:
        dist.destroy_process_group()


def test_peer_store_exchange_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(2, port, ret), nprocs=2, join=True)
    for r in range(2):
        data_ok, flags, want = ret.get(r)
        assert data_ok, "rank %d: gathered blocks differ from the local recomputation" % r
        assert all(f == want for row in flags for f in row), (r, flags, want)
