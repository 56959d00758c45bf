"""Two-rank ``run.predict`` / ``run.predict_test``-style flow: impressions are sharded with ``par.shard_rows``, the ragged
per-rank scores and ranks all-gathered, and every rank returns exactly the single-process result; rank 0's prediction
file is byte-identical to the single-process file.  Needs >= 2 GPUs; skipped otherwise."""
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
    hist, mask, ptr, cand, _ = synth.eval_impressions(n, n_news, H, seed=2)
    args = synth.demo_args(user_log_length=H)
    ue = mb.UserEncoder(args)
    ue.load_state_dict(synth.user_encoder_state("", D, args.user_query_vector_dim, 3), strict=True)
    imp_ids = np.arange(n, dtype=np.int64) * 1000003
    return ue.to(device).eval(), table, hist, mask, ptr, cand, imp_ids


def _worker(rank, world, port, out):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    import tinyrec.run as trun
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    ue, table, hist, mask, ptr, cand, imp_ids = _problem(dev)
    score, rank_t = trun.predict(ue, table, hist, mask, ptr, cand, batch_size=64)
    torch.save(dict(score=score.cpu(), rank=rank_t.cpu()), f"{out}.{rank}")
    if rank == 0:
        trun.write_prediction(f"{out}.txt", imp_ids, ptr, rank_t)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_predict_equals_single_process(tmp_path):
    import torch.multiprocessing as mp
    import tinyrec.run as trun
    out = str(tmp_path / "predict.pt")
    mp.spawn(_worker, args=(2, 29571, out), nprocs=2, join=True)
    ue, table, hist, mask, ptr, cand, imp_ids = _problem(torch.device("cuda", 0))
    score, rank = trun.predict(ue, table, hist, mask, ptr, cand)
    for r in range(2):
        got = torch.load(f"{out}.{r}")
        assert torch.equal(got["rank"], rank.cpu())
        assert np.array_equal(got["score"].numpy().view(np.int32), score.cpu().numpy().view(np.int32))
    ref = str(tmp_path / "single.txt")
    trun.write_prediction(ref, imp_ids, ptr, rank)
    assert open(f"{out}.txt", "rb").read() == open(ref, "rb").read()
