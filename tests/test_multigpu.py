"""Multi-GPU product path on real hardware (needs >= 2 B200s: `python -m pytest tests/test_multigpu.py -m gpu`).

ShardedOptimizer.reconstruct_batch over a 2-rank NCCL group: ONE mixed-class object list, class-sorted shard,
per-rank persistent kernel, result records stored by the solve step straight into rank 0's HBM over NVLink
(CUDA IPC) -- must equal the single-GPU result of the same list BIT FOR BIT, for both exchange mechanisms,
with ragged shards, an empty shard and a soft-failed object in the list.
"""
import os
import socket
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _make_list(n, with_bad=True):
    from dsp_slam_b200 import synth
    clss = [("cars", "chairs")[(i * 5) % 3 == 0] for i in range(n)]
    sizes = [(300, 129, 700, 64, 1000, 333, 128, 513, 5, 900, 2048, 256)[i % 12] for i in range(n)]
    objs = [synth.make_object(200 + i, m, cls=c) for i, (m, c) in enumerate(zip(sizes, clss))]
    ins = [dict(t_cam_obj=o["t_cam_obj_init"], pts=o["pts"], class_id=(0 if c == "cars" else 1)) for o, c in zip(objs, clss)]
    if with_bad and n > 3:
        ins[3] = dict(ins[3], pts=np.zeros((0, 3), np.float32))          # unusable detection -> per-object soft failure
    return ins


def _worker(rank, world, port, out_dir, n_obj):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    import json
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from dsp_slam_b200.optimizer import Optimizer
    from dsp_slam_b200.distributed import ShardedOptimizer
    G = os.path.join(ROOT, "tests", "golden")
    cfg = json.load(open(os.path.join(ROOT, "dsp_slam_b200", "configs", "config_kitti.json")))
    opt = Optimizer(os.path.join(G, "decoder_cars.npz"), cfg, device=rank, sdf_only=True,
                    extra_decoders=[os.path.join(G, "decoder_chairs.npz")])
    ins = _make_list(n_obj)
    out = {}
    for mech in ("peer", "nccl"):
        sh = ShardedOptimizer(opt, exchange=mech)
        assert sh.exchange == mech
        for rep in range(3):                                   # several steps: slot-set parity + acknowledgements
            res = sh.reconstruct_batch(ins)
        everyone = sh.reconstruct_batch(ins, all_ranks=True)
        assert len(everyone) == n_obj
        if rank == 0:
            out[mech] = res
            for a_, b_ in zip(res, everyone):
                assert a_.is_good == b_.is_good
                if a_.is_good:
                    np.testing.assert_array_equal(a_.t_cam_obj, b_.t_cam_obj)
        elif mech == "peer":
            assert res is None
        sh.close()
    if rank == 0:
        single = opt.reconstruct_batch(ins)                    # the same list on ONE GPU
        np.savez(os.path.join(out_dir, "cmp.npz"),
                 good_single=np.array([r.is_good for r in single]),
                 **{f"good_{m}": np.array([r.is_good for r in out[m]]) for m in out},
                 **{f"T_{m}": np.stack([r.t_cam_obj if r.is_good else np.zeros((4, 4), np.float32) for r in out[m]]) for m in out},
                 **{f"z_{m}": np.stack([r.code if r.is_good else np.zeros(64, np.float32) for r in out[m]]) for m in out},
                 T_single=np.stack([r.t_cam_obj if r.is_good else np.zeros((4, 4), np.float32) for r in single]),
                 z_single=np.stack([r.code if r.is_good else np.zeros(64, np.float32) for r in single]),
                 status_single=np.array([r.status for r in single]))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("n_obj", [13, 1])
def test_sharded_equals_single_gpu_bit_for_bit(tmp_path, n_obj):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path), n_obj), nprocs=2, join=True)
    d = np.load(tmp_path / "cmp.npz")
    if n_obj > 3:
        assert not d["good_single"][3] and d["status_single"][3] == 5       # DSPGN_ST_BAD_INPUT, neighbours unaffected
        assert d["good_single"].sum() == n_obj - 1
    for m in ("peer", "nccl"):
        np.testing.assert_array_equal(d[f"good_{m}"], d["good_single"])
        np.testing.assert_array_equal(d[f"T_{m}"], d["T_single"])
        np.testing.assert_array_equal(d[f"z_{m}"], d["z_single"])
