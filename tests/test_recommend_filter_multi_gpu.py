"""Two-rank ``run.recommend`` with a candidate pool, per-user exclusions and per-user categories: the pool and the news
categories are replicated, the exclusions and user categories sharded with the users, and every rank returns exactly
the single-process result.  Needs >= 2 GPUs; skipped otherwise."""
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
    n_news, H, D, n = 3000, 50, 256, 301        # odd: the shards are ragged
    table = (torch.randn(n_news + 1, D, generator=torch.Generator().manual_seed(1)) * 0.1).to(device)
    hist, mask, _, _, _ = synth.eval_impressions(n, n_news, H, seed=2)
    args = synth.demo_args(user_log_length=H)
    ue = mb.UserEncoder(args)
    ue.load_state_dict(synth.user_encoder_state("", D, args.user_query_vector_dim, 3), strict=True)
    rng = np.random.default_rng(3)
    filters = dict(candidates=rng.random(n_news + 1) < 0.4,
                   exclude=rng.integers(-5, n_news + 10, size=(n, 30)),
                   news_category=rng.integers(0, 18, size=n_news + 1),
                   user_categories=rng.random((n, 18)) < 0.5)
    return ue.to(device).eval(), table, hist, mask, filters


def _worker(rank, world, port, out):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    import tinyrec.run as trun
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    ue, table, hist, mask, filters = _problem(dev)
    idx, score = trun.recommend(ue, table, hist, mask, 32, batch_size=64, **filters)
    torch.save(dict(idx=idx.cpu(), score=score.cpu()), f"{out}.{rank}")
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_filtered_recommend_equals_single_process(tmp_path):
    import torch.multiprocessing as mp
    import tinyrec.run as trun
    out = str(tmp_path / "rec_filter.pt")
    mp.spawn(_worker, args=(2, 29561, out), nprocs=2, join=True)
    ue, table, hist, mask, filters = _problem(torch.device("cuda", 0))
    idx, score = trun.recommend(ue, table, hist, mask, 32, **filters)
    for r in range(2):
        got = torch.load(f"{out}.{r}")
        assert torch.equal(got["idx"], idx.cpu())
        assert np.array_equal(got["score"].numpy().view(np.int32), score.cpu().numpy().view(np.int32))
