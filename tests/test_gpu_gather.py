"""The C-ABI keypoint gather (casa_comm_init / casa_allgather_points_overlapped) on two GPUs: shards voted on their
own devices and gathered by the library's NCCL path equal the unsharded single-GPU result bit for bit.  The NCCL id
travels over a gloo process group: the gather itself needs no torch collective (SURVEY.md 8b export list)."""
import os
import socket

import numpy as np
import pytest

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, out_dir):
    import torch.distributed as dist

    from casapose_b200 import sharding, synthetic
    from casapose_b200.pose_estimation import ransac_voting_layer_all_masks

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    n_images = 4
    d = synthetic.make_frames(n_images, 120, 160, (1, 5, 6), variant="easy")
    s, e = sharding.shard_bounds(n_images, rank, world)
    mask = torch.from_numpy(d["mask"][s:e]).to(dev)
    vertex = torch.from_numpy(d["vertex"][s:e]).to(dev)
    g = sharding.AbiGather((e - s, 3, 9, 2), dev, world, rank)
    results = []
    for step in range(3):  # three steps: the two result buffers alternate, the gathers overlap the next vote
        ransac_voting_layer_all_masks(mask, vertex, 64, seed=5 + step, image_offset=s, out=g.buffer(step))
        results.append(g.launch(step))
        if step:
            np.save(os.path.join(out_dir, "rank%d_step%d.npy" % (rank, step - 1)), results[step - 1].wait().cpu().numpy())
    np.save(os.path.join(out_dir, "rank%d_step2.npy" % rank), results[2].wait().cpu().numpy())
    torch.cuda.synchronize()
    g.close()
    dist.barrier()
    dist.destroy_process_group()


def test_two_gpu_gather_equals_single_gpu(cuda_lib, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp

    from casapose_b200 import synthetic
    from casapose_b200.pose_estimation import ransac_voting_layer_all_masks

    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    d = synthetic.make_frames(4, 120, 160, (1, 5, 6), variant="easy")
    mask, vertex = torch.from_numpy(d["mask"]).cuda(), torch.from_numpy(d["vertex"]).cuda()
    for step in range(3):
        whole = ransac_voting_layer_all_masks(mask, vertex, 64, seed=5 + step).cpu().numpy()
        for r in range(2):
            got = np.load(os.path.join(str(tmp_path), "rank%d_step%d.npy" % (r, step)))
            assert got.shape == whole.shape and np.array_equal(got, whole)
