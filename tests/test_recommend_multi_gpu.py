"""Two-rank ``run.recommend``: users sharded like ``evaluate``'s impressions and the results all-gathered; every rank
returns exactly the single-process result.  Needs >= 2 GPUs; skipped otherwise."""
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _problem(device):
    import tinyrec.model_bert as mb
    import tinyrec.synth as synth
    n_news, H, D = 3000, 50, 256
    table = (torch.randn(n_news + 1, D, generator=torch.Generator().manual_seed(1)) * 0.1).to(device)
    hist, mask, _, _, _ = synth.eval_impressions(301, n_news, H, seed=2)     # odd: the shards are ragged
    args = synth.demo_args(user_log_length=H)
    ue = mb.UserEncoder(args)
    ue.load_state_dict(synth.user_encoder_state("", D, args.user_query_vector_dim, 3), strict=True)
    return ue.to(device).eval(), table, hist, mask


def _worker(rank, world, port, out):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    import tinyrec.run as trun
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    ue, table, hist, mask = _problem(dev)
    idx, score = trun.recommend(ue, table, hist, mask, 32, batch_size=64)
    torch.save(dict(idx=idx.cpu(), score=score.cpu()), f"{out}.{rank}")
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_recommend_equals_single_process(tmp_path):
    import torch.multiprocessing as mp
    import tinyrec.run as trun
    out = str(tmp_path / "rec.pt")
    mp.spawn(_worker, args=(2, 29557, out), nprocs=2, join=True)
    ue, table, hist, mask = _problem(torch.device("cuda", 0))
    idx, score = trun.recommend(ue, table, hist, mask, 32)
    for r in range(2):
        got = torch.load(f"{out}.{r}")
        assert torch.equal(got["idx"], idx.cpu())
        assert np.array_equal(got["score"].numpy().view(np.int32), score.cpu().numpy().view(np.int32))
