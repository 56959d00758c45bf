"""One process per GPU over ``torch.distributed`` (NCCL on the B200 box, gloo in CPU tests):
the replacement for the reference's Horovod plumbing.

Reference: Tiny-NewsRec/utils.py:43-60 (``init_hvd_cuda``), run.py:142-149 (broadcast +
DistributedOptimizer(op=Average)), run.py:372-379 (eval sum all-reduce), streaming.py:40-58
(file sharding r, r+world, ...).  The path shards by impressions (training / eval) and by news
rows (table build); the only data-path collectives are the gradient all-reduce, the final table
all-gather and the 5-scalar metric reduction.
"""
import os

import torch
import torch.distributed as dist


def init_distributed(enable=True, backend=None):
    """-> (world, rank, local_rank), mirroring ``init_hvd_cuda`` (utils.py:43-60).  Reads the
    torchrun environment; a single process without it is world 1."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        nccl_defaults()
    if enable and world > 1 and not dist.is_initialized():
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local)
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        else:
            dist.init_process_group(backend)
    elif torch.cuda.is_available():
        torch.cuda.set_device(local)
    return world, rank, local


COMM_CTAS = 8


def nccl_defaults():
    """NCCL settings of the data-parallel train step; must run BEFORE the communicator is created.  The gradient
    exchange is ~59 MB per 7 ms step over NVSwitch: bandwidth is not the constraint, SM occupancy is -- the all-reduce
    shares the GPU with persistent GEMMs.  ``NCCL_MAX_CTAS`` caps a collective at COMM_CTAS CTAs, the number of SMs
    the GEMM grids leave free while exchanges are in flight (``tinyrec.optim.DistributedOptimizer``)."""
    os.environ.setdefault("NCCL_MAX_CTAS", str(COMM_CTAS))


def world_size():
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


def get_rank():
    return dist.get_rank() if dist.is_available() and dist.is_initialized() else 0


def shard_files(files, rank, world):
    """streaming.py:53-54: worker r reads files r, r+world, ..."""
    return [f for i, f in enumerate(files) if i % world == rank]


def shard_rows(n_rows, rank, world):
    """Contiguous row range of the news table owned by ``rank`` (table build, SURVEY.md section 8e)."""
    per = (n_rows + world - 1) // world
    lo = min(n_rows, rank * per)
    return lo, min(n_rows, lo + per)


def allreduce_sum_(t):
    if world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t


def allreduce_mean_(t):
    """hvd.allreduce(op=Average) semantics (run.py:145-149)."""
    w = world_size()
    if w > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        t.div_(w)
    return t


def reduce_eval_sums(local_count, local_sums):
    """run.py:372-379: total metric sums / total impression count (all impressions, skipped ones
    included).  local_sums: float64 [4] tensor; returns (mean float64 [4], total_count)."""
    buf = torch.cat([local_sums.double().reshape(4), torch.tensor([float(local_count)], dtype=torch.float64,
                                                                 device=local_sums.device)])
    allreduce_sum_(buf)
    total = float(buf[4].item())
    return buf[:4] / max(total, 1.0), int(total)


def allgather_rows(local_rows, n_rows):
    """Gather the per-rank ``[hi-lo, D]`` table shards (``shard_rows`` layout) into ``[n_rows, D]``."""
    w = world_size()
    if w == 1:
        return local_rows
    per = (n_rows + w - 1) // w
    D = local_rows.shape[1]
    pad = torch.zeros(per, D, device=local_rows.device, dtype=local_rows.dtype)
    pad[:local_rows.shape[0]] = local_rows
    out = torch.empty(w * per, D, device=local_rows.device, dtype=local_rows.dtype)
    dist.all_gather_into_tensor(out, pad)
    return out[:n_rows]


def allgather_ragged(local):
    """Concatenate every rank's 1-D ``local`` (lengths may differ) in rank order, on every rank: the lengths are
    gathered first, then the padded vectors in one ``all_gather_into_tensor``."""
    w = world_size()
    if w == 1:
        return local
    counts = torch.empty(w, device=local.device, dtype=torch.int64)
    dist.all_gather_into_tensor(counts, torch.tensor([local.numel()], device=local.device, dtype=torch.int64))
    counts = counts.tolist()
    per = max(counts)
    if per == 0:
        return local
    pad = torch.zeros(per, device=local.device, dtype=local.dtype)
    pad[:local.numel()] = local
    out = torch.empty(w * per, device=local.device, dtype=local.dtype)
    dist.all_gather_into_tensor(out, pad)
    return torch.cat([out[r * per:r * per + c] for r, c in enumerate(counts)])


class SymmetricGradBuffer:
    """The flat fp32 gradient buffer of a data-parallel model as a SYMMETRIC allocation (every rank's copy is mapped
    into every process over NVLink: ``torch.distributed._symmetric_memory``), plus a flag page, for the one-kernel
    peer-memory all-reduce ``tnr_allreduce_p2p``.  Construction is a collective (all ranks, same order, same size).
    ``available(...)`` says whether this process can use it; ``TNR_P2P_ALLREDUCE=0`` keeps NCCL."""

    def __init__(self, numel, device):
        import torch.distributed._symmetric_memory as symm
        from . import _lib
        self.world, self.rank = dist.get_world_size(), dist.get_rank()
        group = dist.group.WORLD
        try:
            symm.enable_symm_mem_for_group(group.group_name)
        except Exception:  # noqa: BLE001  (newer torch enables it implicitly)
            pass
        self.grad = symm.empty(numel, dtype=torch.float32, device=device)
        self.grad.zero_()
        self.grad_hdl = symm.rendezvous(self.grad, group)
        words = int(_lib.load().tnr_allreduce_p2p_flag_words())
        self.flags = symm.empty(words, dtype=torch.int32, device=device)
        self.flags.zero_()
        self.flags_hdl = symm.rendezvous(self.flags, group)
        self.ptrs_dev = int(self.grad_hdl.buffer_ptrs_dev)
        self.flags_dev = int(self.flags_hdl.buffer_ptrs_dev)
        # NVLS: the same buffer at a multicast address (reduce in the switch); 0 when the fabric has no multicast
        self.mc_ptr = 0
        if os.environ.get("TNR_NVLS", "1") != "0":
            try:
                self.mc_ptr = int(self.grad_hdl.multicast_ptr or 0)
            except Exception:  # noqa: BLE001
                self.mc_ptr = 0
        torch.cuda.synchronize(device)
        dist.barrier()                       # every rank's flag page is zero before anyone's first kernel

    @staticmethod
    def wanted():
        return (os.environ.get("TNR_P2P_ALLREDUCE", "1") != "0" and dist.is_available() and dist.is_initialized()
                and dist.get_world_size() > 1 and dist.get_backend() == "nccl")

    def all_reduce(self, lo, hi, n_ctas):
        """sum-all-reduce self.grad[lo:hi] in place on the current stream"""
        from . import ops
        ops.allreduce_p2p(self.ptrs_dev, self.mc_ptr, self.flags_dev, self.rank, self.world, lo, hi - lo, n_ctas)
