"""N > 1 on GPUs: world_size-2 NCCL processes run the REAL transforms on their shard and gather
the augmented volumes to rank 0 (`parallel.gather_batch_to_root`, the one exchange the path
has).  Needs two GPUs: skipped on a single-GPU machine."""

import os
import socket
import warnings

import pytest
import torch

pytestmark = pytest.mark.gpu


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _pipeline(tio):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return tio.Compose([tio.Affine(scales=(0.9, 1.1), degrees=(-10, 10)), tio.ElasticDeformation(),
                            tio.BiasField(), tio.Blur(std=(0, 2)), tio.Noise(std=(0, 0.25)),
                            tio.Gamma(log_gamma=(-0.3, 0.3))], copy=False)


def _shard(tio, rank, n, device):
    g = torch.Generator().manual_seed(10 + rank)
    data = torch.rand((n, 1, 48, 64, 64), generator=g).to(device)
    seg = (torch.rand((n, 1, 48, 64, 64), generator=g) * 4).to(torch.int16).to(device)
    return tio.SubjectsBatch({
        "t1": tio.ImagesBatch(data, [tio.AffineMatrix() for _ in range(n)]),
        "seg": tio.ImagesBatch(seg, [tio.AffineMatrix() for _ in range(n)], image_class=tio.LabelMap)})


def _augment(tio, parallel, rank, n, device):
    parallel.seed_for_rank(100, rank)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return _pipeline(tio)(_shard(tio, rank, n, device))


def _worker(rank, world, port, counts, results):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import torchio_b200 as tio
        from torchio_b200 import parallel

        out = _augment(tio, parallel, rank, counts[rank], torch.device("cuda", rank))
        gathered = parallel.gather_batch_to_root(out)  # counts exchanged by all_gather (ragged shards)
        again = parallel.gather_batch_to_root(out, counts=counts,
                                              out=parallel.gather_buffers(out, counts) if rank == 0 else None)
        if rank == 0:
            assert all(torch.equal(gathered[k], again[k]) for k in gathered)
            # rank 1's block == what rank 1's seed and data give when recomputed here
            mine = _augment(tio, parallel, 1, counts[1], torch.device("cuda", 0))
            ok = all(torch.equal(gathered[k][counts[0]:], mine.images[k].data) for k in gathered)
            own = all(torch.equal(gathered[k][:counts[0]], out.images[k].data) for k in gathered)
            results.put((ok, own, {k: tuple(v.shape) for k, v in gathered.items()}))
        else:
            assert gathered is None and again is None
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_real_transforms_shard_and_nccl_gather_world2():
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    results = ctx.Queue()
    counts = [3, 2]
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, counts, results)) for r in range(2)]
    for p in procs:
        p.start()
    ok, own, shapes = results.get(timeout=300)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert ok and own
    assert shapes == {"t1": (5, 1, 48, 64, 64), "seg": (5, 1, 48, 64, 64)}
