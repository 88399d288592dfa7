"""GPU, world_size 2 over NCCL (skipped on single-GPU boxes): the crop scatter on hardware.  Rank 0 owns many mini-batch
groups, rank 1 few; `BatchedOCR._run_groups_dev` balances them with the GPU-to-GPU all_to_all (device canvases, no host
staging) and every rank must get back, for each of its own groups, exactly the ids / probabilities a single-rank run
(`_run_groups_dev_local` on the same records) produces - bit for bit, since a crop's result does not depend on which
GPU recognises it (same kernels, same padded width, same group)."""
import os
import socket
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from yomitoku_b200 import TextRecognizer
        from yomitoku_b200 import parallel as par
        from yomitoku_b200.data import crop_geometry
        from yomitoku_b200.pipeline import BatchedOCR
        from yomitoku_b200.synth import peaked_parseq_state_dict, synthetic_page
        from yomitoku_b200.text_recognizer import plan_mini_batches
        rec = TextRecognizer(model_name="parseq-tiny-dynw-v4", from_pretrained=False, device="cuda:%d" % rank,
                             dynamic_width=True, batch_bucketing=True)
        sd = peaked_parseq_state_dict(rec.model.state_dict())
        rec.model.load_state_dict(par.broadcast_state_dict(sd, "cuda"))
        ocr = BatchedOCR(None, rec, workers=1, device_crops=True)
        page, quads = synthetic_page(40 + rank)
        quads = quads[:160] if rank == 0 else quads[:15]          # skew: groups must move from rank 0 to rank 1
        geoms, keep = crop_geometry(page.shape, quads, rec._cfg.data.img_size, True, page=0)
        widths = geoms["canvas_w"].tolist()
        order = np.argsort(geoms["cw"]).tolist()
        plan = plan_mini_batches(widths, order, True, 16, None, None)
        padded, _ = rec._collate_widths(widths, plan)
        groups = [([widths[i] for i in b], [padded[i] for i in b], np.asarray(b, np.int64)) for b in plan]
        pages_dev = torch.from_numpy(np.ascontiguousarray(page))[None].cuda()
        ref = ocr._run_groups_dev_local(groups, geoms, pages_dev, None)
        x0 = dict(par.STATS)
        got = ocr._run_groups_dev(groups, geoms, pages_dev, None)
        moved = par.STATS["exchange_bytes_sent"] - x0["exchange_bytes_sent"]
        recvd = par.STATS["exchange_bytes_received"] - x0["exchange_bytes_received"]
        assert len(got) == len(ref) == len(groups)
        for (ids, probs, glen), (rid, rp, rg) in zip(got, ref):
            assert np.array_equal(ids, rid) and np.array_equal(probs, rp) and glen == rg
        assert (moved > 0) if rank == 0 else (recvd > 0), (rank, moved, recvd)      # rank 0 must hand groups to rank 1
        q.put((rank, "ok", moved))
    except Exception:  # pragma: no cover
        import traceback
        q.put((rank, "fail: " + traceback.format_exc(), None))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_crop_scatter_over_nccl_equals_single_rank():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    out = [q.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    for rank, status, _ in out:
        assert status == "ok", status
    print("[multirank] bytes moved by rank 0:", [o[2] for o in out if o[0] == 0])
