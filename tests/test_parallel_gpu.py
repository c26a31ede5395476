"""GPU tests of the sharded-batch exchange: the pack kernel behind the C-ABI vs its plain-torch statement, and
(2+ GPUs) the whole sharded path over NCCL vs a single-GPU run of the same global batch."""
import os
import socket

import pytest
import torch

import parity_util as pu

pytestmark = pytest.mark.gpu


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("capacity", [3, 8])
def test_pack_kernel_matches_torch_statement(cuda_device, capacity):
    """mhmr_pack_records (one kernel, count read on the device) == parallel.pack_block_torch, bit for bit,
    both when the block has room (capacity 8 > 5 persons) and when it overflows (capacity 3: header reports 5
    detected / 3 packed)."""
    import ctypes

    from multihmr_b200 import _lib, parallel
    from multihmr_b200.model import _OUT_FIELDS, _Outputs

    case, sd, bm, x, K, idx = pu.build_inputs("s_224_S_forced")
    m = pu.build_engine(case, sd, bm, max_persons=16)
    t, P = m.forward_raw(x, K, idx=idx)
    assert P == 5
    lib = _lib.load()
    _, R = parallel.record_layout(m.num_betas, m.num_verts)
    block = torch.full((parallel.HEADER_WORDS + capacity * R,), 7.0, device=cuda_device)
    o = _Outputs(*[ctypes.c_void_p(t[n].data_ptr()) if t.get(n) is not None else None for n in _OUT_FIELDS])
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(lib.mhmr_pack_records(ctypes.byref(o), 16, m.num_betas, m.num_verts, 24, capacity,
                                     ctypes.c_void_p(block.data_ptr()), stream), "mhmr_pack_records")
    torch.cuda.synchronize()
    want = parallel.pack_block_torch(t, P, 24, capacity, m.num_betas, m.num_verts)
    assert torch.equal(block.view(torch.int32), want.view(torch.int32))
    lib.mhmr_record_block_bytes.restype = ctypes.c_int64
    assert lib.mhmr_record_block_bytes(m.num_betas, m.num_verts, capacity) == block.numel() * 4
    assert lib.mhmr_record_floats(m.num_betas, m.num_verts) == R


def _rank_main(rank, world, port, q):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from multihmr_b200 import parallel, synth
    from multihmr_b200.model import Model

    backbone, S, B, seed = "dinov2_vits14", 224, 4, 11
    sd = synth.make_state_dict(backbone, S, seed=seed, det_bias=-1.0)
    bm = synth.make_body_model(seed)
    x, K = synth.make_images(B, S, seed), synth.make_cameras(B, S, jitter=True, seed=seed)
    m = Model(backbone=backbone, img_size=S, max_batch=B, max_persons=128, body_model=bm, device=dev)
    m.load_state_dict(sd)
    # capacity 2 per rank: the natural detections overflow it, so the full-size second round runs too
    for cap in (None, 2):
        sm = parallel.ShardedModel(m, capacity=cap)
        recs, counts = sm(x, K, det_thresh=0.3, nms_kernel_size=3)
        if rank == 0:
            q.put((cap, counts, recs.cpu().numpy()))
        sm.gather.close()
    if rank == 0:  # single-GPU run of the whole batch on the same device
        t, P = m.forward_raw(x, K, det_thresh=0.3, nms_kernel_size=3)
        want = parallel.pack_block_torch(t, P, 0, 128, m.num_betas, m.num_verts)
        _, R = parallel.record_layout(m.num_betas, m.num_verts)
        q.put(("single", [P], want[parallel.HEADER_WORDS:].view(128, R)[:P].cpu().numpy()))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_forward_equals_single_gpu(cuda_device):
    """2 ranks over NCCL, image shards [0,2) and [2,4): the gathered persons are bit-identical to the single-GPU
    forward of the 4-image batch, in the same (b, y, x) order — images are independent units of Model.forward."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp

    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_main, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = [q.get(timeout=600) for _ in range(3)]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    res = {g[0]: g for g in got}
    single = torch.from_numpy(res["single"][2])
    assert single.shape[0] >= 4, "workload must produce detections on both shards"
    for cap in (None, 2):
        _, counts, recs = res[cap]
        recs = torch.from_numpy(recs)
        assert sum(counts) == single.shape[0] and min(counts) > 0
        assert torch.equal(recs, single), (cap, (recs - single).abs().max())
