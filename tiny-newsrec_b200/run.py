"""Mode drivers: ``train`` / ``test`` / ``get_teacher_emb`` on the B200 path.

Same three modes, argument namespace (``parameters.py`` flags) and on-disk formats as the
reference's ``Tiny-NewsRec/run.py`` (:20 train, :219 test, :382 get_teacher_emb):
checkpoints are ``torch.save({'model_state_dict', 'category_dict', 'word_dict',
'subcategory_dict'}, model_dir/epoch-{n}.pt)`` (run.py:205-214), teacher tables are pickled
float32 ndarrays [N+1, D] (run.py:458-459).  What changes underneath: Horovod -> NCCL
(``tinyrec.parallel``), host batch assembly -> device gathers (``tinyrec.dataloader``), the
per-impression Python metric loop -> ``tnr_eval_metrics``, the single-GPU table build ->
row-sharded build + all-gather.

Text ingestion (news.tsv tokenisation, TF ``TextLineDataset`` streaming) is outside the hot
path (SURVEY.md section 2): callers hand in ``news_combined`` (int32 [N+1, 2L]) and an iterable
of behaviour lines or pre-parsed index arrays.
"""
import logging
import os
import random

import numpy as np
import torch

from . import checkpoint as ckpt
from . import dataloader as dl
from . import ops
from . import parallel as par
from .model_bert import Model
from .optim import Adam, DistributedOptimizer, broadcast_parameters


def apply_freeze_policy(model, trainable_layers, student=True):
    """run.py:98-112: teachers frozen; whole bert_model frozen except the listed encoder layers."""
    if student:
        for p in model.teachers.parameters():
            p.requires_grad = False
        bm = model.student.news_encoder.bert_model
    else:
        bm = model.news_encoder.bert_model
    for p in bm.parameters():
        p.requires_grad = False
    for i, layer in enumerate(bm.bert.encoder.layer):
        if i in trainable_layers:
            logging.info(f"finetune block {i}")
            for p in layer.parameters():
                p.requires_grad = True


def load_teacher_user_encoders(model, teacher_state_dicts):
    """run.py:61-70: keys ``user_encoder.*`` of teacher i -> ``teachers.{i}.*``."""
    sd = model.state_dict()
    loaded = []
    for i, tsd in enumerate(teacher_state_dicts):
        for k, v in tsd.items():
            if not k.startswith("user_encoder"):
                continue
            key = ".".join(["teachers", str(i)] + k.split(".")[1:])
            sd[key].copy_(v)
            loaded.append(key)
    return loaded


def load_student_from_first_stage(model, pretrained_state_dict):
    """run.py:76-85: every key starting with ``student`` is copied."""
    sd = model.state_dict()
    loaded = []
    for k, v in pretrained_state_dict.items():
        if k.startswith("student"):
            sd[k].copy_(v)
            loaded.append(k)
    return loaded


def accuracy(y_true, y_hat):
    """utils.py:79-83 (device scalar; no host sync)."""
    return (y_true == y_hat.argmax(dim=-1)).sum().float() / y_true.shape[0]


class _PinnedRing:
    """``depth`` slots of pinned host staging tensors: ``push(arrays)`` copies one batch of numpy arrays into the next
    slot and starts its host->device copies (``non_blocking``, on the current stream); a slot is reused only after
    the copies issued from it have completed (an event per slot), so the host can run ``depth - 1`` batches ahead
    of the device -- the job of the reference loader's producer thread (dataloader.py:85-116).  Without CUDA
    (``device='cpu'``: the host-logic tests) the arrays are passed through as tensors."""

    def __init__(self, device, depth=3):
        self.device = torch.device(device)
        self.depth, self.slots, self.k = depth, [], 0

    def push(self, arrays):
        if self.device.type != "cuda":
            return tuple(torch.from_numpy(np.ascontiguousarray(a)) for a in arrays)
        i_slot = self.k % self.depth
        self.k += 1
        if len(self.slots) <= i_slot:
            self.slots.append(dict(bufs=[None] * len(arrays), ev=None))
        slot = self.slots[i_slot]
        if slot["ev"] is not None:
            slot["ev"].synchronize()
        out = []
        for i, a in enumerate(arrays):
            a = np.asarray(a)
            buf = slot["bufs"][i]
            if buf is None or buf.dtype != torch.from_numpy(a[:0].reshape(-1)).dtype or buf.numel() < a.size:
                buf = slot["bufs"][i] = torch.empty(max(a.size, 1), dtype=torch.from_numpy(a[:0].reshape(-1)).dtype,
                                                    pin_memory=True)
            view = buf[:a.size].view(a.shape)
            np.copyto(view.numpy(), a)
            out.append(view.to(self.device, non_blocking=True))
        slot["ev"] = torch.cuda.Event()
        slot["ev"].record()
        return tuple(out)


class IndexBatches:
    """Re-iterable source of pre-parsed training impressions -> device index tensors (one pass per epoch).
    ``hist_idx`` int32 [n,H], ``hist_mask`` f32 [n,H], ``cand_idx`` int32 [n,K], ``label`` int64 [n].
    Rank r takes batches r, r+world, ... (impression sharding, streaming.py:53-54) of the first
    ``(n_batches // world) * world`` batches: every rank runs the SAME number of optimizer steps, so the per-step
    gradient all-reduces of the ranks always pair up (a ragged tail would hang NCCL)."""

    def __init__(self, hist_idx, hist_mask, cand_idx, label, batch_size, rank=0, world=1, device="cuda"):
        self.arr = (hist_idx, hist_mask, cand_idx, label)
        self.bs, self.rank, self.world, self.device = batch_size, rank, world, device
        self.ring = _PinnedRing(device)

    def __len__(self):
        return (self.arr[0].shape[0] // self.bs) // self.world

    def __iter__(self):
        for i in range(len(self)):
            b = i * self.world + self.rank
            sl = slice(b * self.bs, (b + 1) * self.bs)
            yield self.ring.push([a[sl] for a in self.arr])


class LineBatches:
    """Re-iterable source that parses ``behaviors_np{K}_*.tsv`` lines (dataloader.py:118-148) into index batches.
    ``lines``: a sequence of lines, or a zero-argument callable returning one (called once per epoch -- e.g. a
    shuffled re-read of the rank's files).  Rank r parses lines r, r+world, ... (streaming.py:53-54 applied to lines)
    and every rank stops after ``len(lines) // (world * batch_size)`` batches (equal step counts, see IndexBatches).
    The positive's slot ``label = randint(0, npratio)`` (dataloader.py:135) is drawn from ``Random(seed + epoch)``."""

    def __init__(self, lines, news_index, args, rank=0, world=1, device="cuda", seed=0):
        self.lines, self.news_index, self.args = lines, news_index, args
        self.rank, self.world, self.device, self.seed = rank, world, device, seed
        self.epoch = 0
        self.ring = _PinnedRing(device)

    def _materialise(self):
        lines = self.lines() if callable(self.lines) else self.lines
        return lines if hasattr(lines, "__len__") and hasattr(lines, "__getitem__") else list(lines)

    def __iter__(self):
        a = self.args
        H, K, bs = a.user_log_length, a.npratio + 1, a.batch_size
        lines = self._materialise()
        rng = random.Random(self.seed + self.epoch)
        self.epoch += 1
        n_batches = len(lines) // (self.world * bs)
        for b in range(n_batches):
            rows = [dl.parse_train_line(lines[(b * bs + j) * self.world + self.rank], self.news_index, H, a.npratio, rng)
                    for j in range(bs)]
            hist = np.array([r[0] for r in rows], dtype=np.int32)
            mask = np.array([r[1] for r in rows], dtype=np.float32)
            cand = np.array([r[2] for r in rows], dtype=np.int32).reshape(bs, K)
            lab = np.array([r[3] for r in rows], dtype=np.int64)
            yield self.ring.push([hist, mask, cand, lab])


def batches_from_lines(lines, news_index, args, rank=0, world=1, device="cuda", seed=0):
    """Kept name: returns the re-iterable ``LineBatches`` (sharded by rank, one pass per epoch)."""
    return LineBatches(lines, news_index, args, rank, world, device, seed)


class GraphedTrainStep:
    """The body of the reference train loop (run.py:178-197: forward, acc, zero_grad, backward, optimizer step)
    captured ONCE into a CUDA graph and replayed per batch: the ~100 kernel launches and ~40 small torch ops of a
    step become one graph launch (no launch gaps, no Python between kernels).  Inputs are copied into static device
    buffers; the dropout seed and the Adam step counter live on the device and advance inside the graph, so every
    replay is a new step.  Warm-up steps needed before the capture run on a snapshot that is restored afterwards:
    constructing this object does not train the model.

        step = GraphedTrainStep(model, optimizer, first_batch)
        total, distill, emb, target, score = step(history, mask, candidate, label, th_list, tc_list)

    With ``batcher`` (a ``tinyrec.dataloader.TrainBatcher``) the batch is the four INDEX tensors of the loader
    (hist_idx int32 [B,H], hist_mask f32 [B,H], cand_idx int32 [B,K], label int64 [B]) and the row gathers that
    assemble the model inputs from the device-resident tables (dataloader.py:129-144) run inside the graph: only
    ~7 KB of indices cross PCIe per step.

        step = GraphedTrainStep(model, optimizer, (hist_idx, hist_mask, cand_idx, label), batcher=batcher)
        total, distill, emb, target, score = step(hist_idx, hist_mask, cand_idx, label)

    ``step.stats`` (fp32 [3] on the device) accumulates [sum of total_loss, sum of utils.acc, steps] inside the
    graph (run.py:180-182); the returned tensors are static outputs overwritten by the next call."""

    def __init__(self, model, optimizer, batch, warmup=3, batcher=None):
        self.model, self.opt, self.batcher = model, optimizer, batcher
        inner = getattr(optimizer, "opt", optimizer)
        inner.make_capturable()
        self.static = self._clone(batch)
        st = model.train_state()
        inner.ensure_state()
        ne = model.student.news_encoder if hasattr(model, "student") else model.news_encoder
        drop = ne.drop_state(st.flat.data.device)
        self.stats = torch.zeros(3, device=st.flat.data.device, dtype=torch.float32)
        snap = dict(data=st.flat.data.clone(), grad=st.flat.grad.clone(), m=inner.m.clone(), v=inner.v.clone(),
                    vmax=inner.vmax.clone() if inner.vmax is not None else None, step=inner.step_dev.clone(),
                    seed=drop.seed.clone())
        cur = torch.cuda.current_stream()
        side = torch.cuda.Stream()
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for _ in range(max(1, warmup)):                # first-call work: workspaces, smem attributes, NCCL buffers
                self._eager(self.static)
        cur.wait_stream(side)
        torch.cuda.synchronize()
        launches0 = ops.stats.launches
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, capture_error_mode="thread_local"):
            self.out = self._eager(self.static)
        self.launches_per_step = ops.stats.launches - launches0
        # roll the warm-up steps back: parameters, optimizer state, step counter, dropout seed
        st.flat.data.copy_(snap["data"])
        st.flat.grad.copy_(snap["grad"])
        st.flat.refresh_shadow()
        inner.m.copy_(snap["m"])
        inner.v.copy_(snap["v"])
        if inner.vmax is not None:
            inner.vmax.copy_(snap["vmax"])
        inner.step_dev.copy_(snap["step"])
        drop.seed.copy_(snap["seed"])
        self.stats.zero_()
        torch.cuda.synchronize()

    def close(self):
        """Release the captured graph.  Call this before ``torch.distributed.destroy_process_group()``: the graph
        holds the NCCL all-reduce kernels of the step, and tearing the communicator down under a live graph hangs."""
        self.graph = None
        self.out = None
        torch.cuda.synchronize()

    @staticmethod
    def _clone(batch):
        dev = lambda t: t.detach().to("cuda", copy=True) if not t.is_cuda else t.detach().clone()  # noqa: E731
        return tuple([dev(t) for t in x] if isinstance(x, (list, tuple)) else dev(x) for x in batch)

    def _eager(self, batch):
        if self.batcher is not None:
            hist_idx, hist_mask, cand_idx, label = batch
            history, candidate, th, tc = self.batcher.assemble(hist_idx, cand_idx)
            batch = (history, hist_mask, candidate, label, th, tc)
        self.opt.zero_grad()
        out = self.model(*batch)
        out[0].backward()
        self.opt.step()
        out = tuple(o.detach() for o in out)
        self.stats[0] += out[0]
        self.stats[1] += accuracy(batch[3], out[4])
        self.stats[2] += 1.0
        return out

    def __call__(self, *batch):
        if len(batch) != len(self.static):
            raise TypeError(f"GraphedTrainStep takes {len(self.static)} inputs, got {len(batch)}")
        for dst, src in zip(self.static, batch):
            if isinstance(dst, list):
                for d, t in zip(dst, src):
                    d.copy_(t, non_blocking=True)
            else:
                dst.copy_(src, non_blocking=True)
        self.graph.replay()
        ops.bump_param_generation()          # the replay stepped the optimizer: cached parameter copies are stale
        return self.out


def build_kd_model(args):
    """run.py:54-88, :118-122: ``Model(args)`` (student encoder from ``args.model_name`` when set), the teachers'
    user encoders from ``args.teacher_ckpts``, the first-stage student from ``args.pretrain_model_path`` when
    ``args.use_pretrain_model``, then the whole model from ``model_dir/load_ckpt_name`` when given."""
    model = Model(args)
    tsds = []
    for path in (getattr(args, "teacher_ckpts", None) or []):
        tsds.append(torch.load(path, map_location="cpu")["model_state_dict"])
    loaded = load_teacher_user_encoders(model, tsds)
    if getattr(args, "use_pretrain_model", False):
        sd = torch.load(args.pretrain_model_path, map_location="cpu")["model_state_dict"]
        loaded += load_student_from_first_stage(model, sd)
    logging.info(f"{len(loaded)} loaded parameters, {len(model.state_dict()) - len(loaded)} initialized parameters")
    if getattr(args, "load_ckpt_name", None) is not None:
        path = os.path.join(args.model_dir, args.load_ckpt_name)                       # utils.get_checkpoint
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        ckpt.load_checkpoint(path, model)
        logging.info(f"Model loaded from {path}")
    return model


def train(args, news_combined, teacher_embs, batches, model=None, category_dict=None, subcategory_dict=None,
          word_dict=None, use_graph=True, history=None):
    """run.py:20-216.  ``batches``: a RE-ITERABLE source of (hist_idx, hist_mask, cand_idx, label) device tensors,
    iterated once per epoch (``IndexBatches`` / ``LineBatches``; both give every rank the same number of steps).
    ``teacher_embs``: the M [N+1, D] tables, or None to unpickle ``args.teacher_emb_paths`` (run.py:72-73).
    ``model`` None builds it the way run.py:54-122 does (``build_kd_model``).  Full batches run as one replayed CUDA
    graph each (``GraphedTrainStep`` with the loader's row gathers inside); ``use_graph=False`` or an odd-sized batch
    launches the same kernels eagerly.  ``history``: optional list; per step a dict of the five outputs' scalars and
    ``acc`` (device tensors) is appended.  Returns the trained model."""
    ops.check_history_length(args.user_log_length)
    world, rank, local = par.init_distributed(getattr(args, "enable_hvd", True))
    device = torch.device("cuda", local)
    if model is None:
        model = build_kd_model(args)
    if teacher_embs is None:
        teacher_embs = [ckpt.load_teacher_table(p) for p in args.teacher_emb_paths]
    model = model.to(device)
    apply_freeze_policy(model, list(args.bert_trainable_layer))
    optimizer = Adam(model, lr=args.lr, amsgrad=True)                       # run.py:134
    if world > 1:
        broadcast_parameters(model, root_rank=0)                            # run.py:142-143
        optimizer = DistributedOptimizer(optimizer)                         # run.py:144-149
    tables = dl.DeviceTables(news_combined, teacher_embs, device)
    K = args.npratio + 1
    batcher = dl.TrainBatcher(tables, args.batch_size, args.user_log_length, K)
    stats = torch.zeros(3, device=device, dtype=torch.float32)             # [LOSS, ACC, steps] of the epoch's eager steps
    gstep = None
    logging.info("Training...")
    try:
        for ep in range(getattr(args, "start_epoch", 0), args.epochs):
            stats.zero_()
            if gstep is not None:
                gstep.stats.zero_()
            n_steps = 0
            for cnt, (hist_idx, hist_mask, cand_idx, label) in enumerate(batches):
                if cnt > args.max_steps_per_epoch:                              # run.py:176 (runs max+1 steps)
                    break
                if use_graph and hist_idx.shape[0] == args.batch_size:
                    if gstep is None:
                        gstep = GraphedTrainStep(model, optimizer, (hist_idx, hist_mask, cand_idx, label), batcher=batcher)
                    out = gstep(hist_idx, hist_mask, cand_idx, label)
                    acc = None
                else:
                    history_t, candidate, th, tc = batcher.assemble(hist_idx, cand_idx) if hist_idx.shape[0] == args.batch_size \
                        else dl.TrainBatcher(tables, hist_idx.shape[0], args.user_log_length, K).assemble(hist_idx, cand_idx)
                    out = model(history_t, hist_mask, candidate, label, th, tc)
                    acc = accuracy(label, out[4].detach())
                    stats[0] += out[0].detach()
                    stats[1] += acc
                    stats[2] += 1.0
                    optimizer.zero_grad()
                    out[0].backward()
                    optimizer.step()
                n_steps += 1
                if history is not None:
                    if acc is None:
                        acc = accuracy(label, out[4].detach())
                    history.append(dict(epoch=ep, step=cnt, total=out[0].detach().clone(), distill=out[1].detach().clone(),
                                        emb=out[2].detach().clone(), target=out[3].detach().clone(), acc=acc.clone(),
                                        score=out[4].detach().clone()))
                if cnt % args.log_steps == 0 and cnt > 0:
                    loss_sum, acc_sum, _ = (stats + gstep.stats if gstep is not None else stats).tolist()
                    logging.info("[{}] Ed: {}, train_loss: {:.5f}, acc: {:.5f}".format(
                        rank, cnt * args.batch_size, loss_sum / cnt, acc_sum / cnt))
            if n_steps == 0:
                raise ValueError(f"epoch {ep + 1} produced no training steps: `batches` must be re-iterable and hold at "
                                 "least world x batch_size impressions")
            if rank == 0 and getattr(args, "model_dir", None):
                os.makedirs(args.model_dir, exist_ok=True)
                ckpt_path = os.path.join(args.model_dir, f"epoch-{ep + 1}.pt")
                ckpt.save_checkpoint(ckpt_path, model, category_dict, word_dict, subcategory_dict)       # run.py:205-214
                logging.info(f"Model saved to {ckpt_path}")
    finally:
        if gstep is not None:
            gstep.close()
    return model


@torch.no_grad()
def build_news_table(news_encoder, news_combined, batch_size=2048, device=None, sharded=True):
    """run.py:261-290 / :432-447: encode every row of ``news_combined`` (row 0 = pad news included).
    Rows are sharded contiguously over ranks and all-gathered at the end -> fp32 [N+1, D] on device."""
    device = device or next(news_encoder.parameters()).device
    nc = torch.as_tensor(np.ascontiguousarray(news_combined))
    n = nc.shape[0]
    world, rank = (par.world_size(), par.get_rank()) if sharded else (1, 0)
    lo, hi = par.shard_rows(n, rank, world)
    D = news_encoder.dense.weight.shape[0]
    out = torch.empty(hi - lo, D, device=device, dtype=torch.float32)
    tab = nc[lo:hi].to(device)
    for s in range(0, hi - lo, batch_size):
        x = tab[s:s + batch_size].to(torch.int64)           # torch.LongTensor(arr), run.py:276-277
        out[s:s + x.shape[0]] = news_encoder(x)
    return par.allgather_rows(out, n) if world > 1 else out


_EVAL_STAGING = {}


def _eval_staging(device, bs, H, nnz_max, n_slots):
    """Pinned + device staging slots of ``evaluate`` (cached per device, grown on demand) -> (slots, copy stream,
    per-impression metric buffer)."""
    need = (bs * H, bs * H, bs + 1, nnz_max, nnz_max)
    dts = (torch.int32, torch.float32, torch.int64, torch.int32, torch.int8)
    c = _EVAL_STAGING.get(device)
    if c is None or len(c["slots"]) < n_slots or any(a < b for a, b in zip(c["cap"], need)) or c["per"].shape[0] < bs:
        cap = tuple(max(int(m * 1.25) + 16, 1) for m in need)
        slots = [dict(pin=[torch.empty(m, dtype=dt, pin_memory=True) for m, dt in zip(cap, dts)],
                      dev=[torch.empty(m, dtype=dt, device=device) for m, dt in zip(cap, dts)], done=None)
                 for _ in range(n_slots)]
        c = _EVAL_STAGING[device] = dict(slots=slots, cap=cap, stream=torch.cuda.Stream(device=device),
                                         per=torch.empty(max(bs, 1), 5, device=device, dtype=torch.float64))
    return c["slots"][:n_slots], c["stream"], c["per"]


@torch.no_grad()
def evaluate(user_encoder, news_scoring, hist_idx, hist_mask, cand_ptr, cand_idx, labels, batch_size=16384,
             return_per_impression=False):
    """run.py:301-379 on the device.  Impressions are CSR-packed: ``cand_ptr`` int64 [n+1],
    ``cand_idx`` int32 [nnz], ``labels`` int8 [nnz]; rank r scores impressions r-th contiguous slice.
    Returns (mean [auc, mrr, ndcg5, ndcg10] over ALL impressions as the reference's final line does,
    total impression count)."""
    device = news_scoring.device
    n = hist_idx.shape[0]
    H = hist_idx.shape[1]
    ops.check_history_length(H)
    world, rank = par.world_size(), par.get_rank()
    lo, hi = par.shard_rows(n, rank, world)
    sums = torch.zeros(5, device=device, dtype=torch.float64)
    per_all = []
    ptr_h = np.asarray(cand_ptr)
    hist_idx, hist_mask = np.asarray(hist_idx), np.asarray(hist_mask)
    cand_idx, labels = np.asarray(cand_idx), np.asarray(labels)
    # Index batches go host -> pinned staging -> device on a copy stream, one batch ahead of the scoring kernels -- the
    # job of the reference's loader thread (dataloader.py:303-314), which used blocking copies.  The staging copy of a
    # batch (~10 MB of pageable numpy memory at the default batch size) is ONE multi-threaded native memcpy per array
    # (tnr_host_copy_mt: no Python threads, hence no GIL hand-offs); the slots (pinned + device buffers sized for the
    # largest batch of this shard) come from a per-process cache, so cudaHostAlloc is paid once, not per call.  Nothing
    # is read back until the final reduction.
    starts = np.arange(lo, hi, batch_size, dtype=np.int64)
    ends = np.minimum(starts + batch_size, hi)
    nb_total = len(starts)
    nnz_max = int((ptr_h[ends] - ptr_h[starts]).max()) if nb_total else 0
    counts = np.diff(ptr_h[lo:hi + 1])
    max_cs = np.maximum.reduceat(counts, starts - lo) if nb_total else np.zeros(0, dtype=np.int64)
    bs = int((ends - starts).max()) if nb_total else 0
    main = torch.cuda.current_stream(device)
    slots, copy_stream, per_buf = _eval_staging(device, bs, H, nnz_max, min(3, max(1, nb_total)))
    n_slots = len(slots)
    host_threads = max(1, min(8, (os.cpu_count() or 2) // 2))
    for slot in slots:
        slot["done"] = None

    def stage(k):
        s, e = int(starts[k]), int(ends[k])
        p0, p1 = int(ptr_h[s]), int(ptr_h[e])
        slot = slots[k % n_slots]
        if slot["done"] is not None:
            slot["done"].synchronize()                   # the kernels that read this slot's device buffers have finished
        nb, nz = e - s, p1 - p0
        pin = slot["pin"]
        ops.host_copy(pin[0], hist_idx[s:e], host_threads)
        ops.host_copy(pin[1], hist_mask[s:e], host_threads)
        np.subtract(ptr_h[s:e + 1], p0, out=pin[2][:nb + 1].numpy())
        ops.host_copy(pin[3], cand_idx[p0:p1], host_threads)
        ops.host_copy(pin[4], labels[p0:p1], host_threads)
        sizes = (nb * H, nb * H, nb + 1, nz, nz)
        with torch.cuda.stream(copy_stream):
            for d, p_, m in zip(slot["dev"], pin, sizes):
                d[:m].copy_(p_[:m], non_blocking=True)
            ready = torch.cuda.Event()
            ready.record(copy_stream)
        d = slot["dev"]
        return dict(nb=nb, slot=slot, max_c=int(max_cs[k]), ready=ready,
                    dev=(d[0][:nb * H].view(nb, H), d[1][:nb * H].view(nb, H), d[2][:nb + 1], d[3][:nz], d[4][:nz]))

    copy_stream.wait_stream(main)
    nxt = stage(0) if nb_total else None
    for k in range(nb_total):
        cur = nxt
        main.wait_event(cur["ready"])
        hi_t, hm_t, ptr_t, cand_t, lab_t = cur["dev"]
        if hasattr(user_encoder, "forward_gather"):  # news_scoring[log_ids] (dataloader.py:295) fused into the kernel
            user = user_encoder.forward_gather(news_scoring, hi_t, hm_t)
        else:
            user = user_encoder(dl.gather_history_vecs(news_scoring, hi_t), hm_t)
        per = torch.empty(cur["nb"], 5, device=device, dtype=torch.float64) if return_per_impression \
            else per_buf[:cur["nb"]]
        ops.eval_metrics(news_scoring, user, ptr_t, cand_t, lab_t, cur["max_c"], per, sums)
        done = torch.cuda.Event()
        done.record(main)
        cur["slot"]["done"] = done
        if return_per_impression:
            per_all.append(per)
        # the next batch is staged AFTER this batch's kernels are queued: the host copies overlap them
        nxt = stage(k + 1) if k + 1 < nb_total else None
    mean, total = par.reduce_eval_sums(hi - lo, sums[:4])
    if return_per_impression:
        return mean, total, torch.cat(per_all) if per_all else torch.zeros(0, 5, dtype=torch.float64)
    return mean, total


def doc_sim(news_scoring, n_pairs=1000000, rng=random):
    """run.py:292-299: mean cosine similarity of ``n_pairs`` random row pairs drawn from rows 1..N with
    ``random.randrange`` exactly as the reference draws them (pairs with i == j add nothing but still count in the
    mean).  The pair list is drawn on the host, the 2 x n_pairs row reads and cosines run in one kernel."""
    n = news_scoring.shape[0]
    pairs = np.empty((n_pairs, 2), dtype=np.int32)
    for k in range(n_pairs):
        pairs[k, 0] = rng.randrange(1, n)
        pairs[k, 1] = rng.randrange(1, n)
    total = torch.zeros(1, device=news_scoring.device, dtype=torch.float64)
    ops.doc_sim(news_scoring, torch.from_numpy(pairs).to(news_scoring.device), total)
    return float(total.item()) / n_pairs


def latest_checkpoint(directory):
    """utils.py:127-137: the ``epoch-{n}.pt`` with the largest n, or None."""
    if not directory or not os.path.exists(directory):
        return None
    found = {}
    for x in os.listdir(directory):
        try:
            found[int(x.split(".")[-2].split("-")[-1])] = x
        except (ValueError, IndexError):
            continue
    return os.path.join(directory, found[max(found)]) if found else None


def test(args, model, news_combined, hist_idx, hist_mask, cand_ptr, cand_idx, labels):
    """run.py:219-379: student news table, doc-sim diagnostic, then impression scoring with ``user_log_mask`` as in
    args.  ``model`` None: ``Model(args)`` loaded from ``model_dir/load_ckpt_name`` or the latest ``epoch-{n}.pt``
    (run.py:226-243) and broadcast from rank 0."""
    world, rank, local = par.init_distributed(getattr(args, "enable_hvd", True))
    if model is None:
        name = getattr(args, "load_ckpt_name", None)
        path = os.path.join(args.model_dir, name) if name is not None else latest_checkpoint(args.model_dir)
        if path is None or not os.path.exists(path):
            raise FileNotFoundError("No ckpt found")                                            # run.py:231
        model = Model(args)
        ckpt.load_checkpoint(path, model)
        logging.info(f"Model loaded from {path}")
        model = model.to(torch.device("cuda", local))
        if world > 1:
            broadcast_parameters(model, root_rank=0)                                            # run.py:246-247
    model.eval()
    news_scoring = build_news_table(model.student.news_encoder, news_combined, batch_size=args.batch_size * 16)
    logging.info("news scoring num: {}".format(news_scoring.shape[0]))
    if rank == 0 and getattr(args, "doc_sim", True):
        print(f"=== doc-sim: {doc_sim(news_scoring, getattr(args, 'doc_sim_pairs', 1000000))} ===")      # run.py:292-299
    mean, total = evaluate(model.student.user_encoder, news_scoring, hist_idx, hist_mask, cand_ptr, cand_idx, labels)
    if rank == 0:
        logging.info("[{}] Ed: {}: {}".format(rank, total, "\t".join("{:0.2f}".format(float(x) * 100) for x in mean)))
    return mean, total


def get_teacher_emb(args, teacher_state_dicts, news_combined, out_paths=None):
    """run.py:382-460: one [N+1, D] float32 table per teacher checkpoint, pickled like the reference.
    ``teacher_state_dicts`` None: the ``model_state_dict`` of every file in ``args.teacher_ckpts`` (run.py:419-421);
    ``out_paths`` None with ``args.teacher_emb_paths`` set: those paths (run.py:458-459)."""
    from .model_bert_2 import ModelBert
    world, rank, local = par.init_distributed(getattr(args, "enable_hvd", True))
    device = torch.device("cuda", local)
    if teacher_state_dicts is None:
        teacher_state_dicts = [torch.load(p_, map_location="cpu")["model_state_dict"] for p_ in args.teacher_ckpts]
        if out_paths is None:
            out_paths = getattr(args, "teacher_emb_paths", None)
    tables = []
    for i, tsd in enumerate(teacher_state_dicts):
        model = ModelBert(args)
        if tsd is not None:
            model.load_state_dict(tsd)
        model = model.to(device).eval()
        table = build_news_table(model.news_encoder, news_combined, batch_size=args.batch_size * 64)
        arr = table.cpu().numpy()
        logging.info("news scoring num: {}".format(arr.shape[0]))
        if rank == 0 and getattr(args, "doc_sim", False):
            print(f"=== doc-sim: {doc_sim(table, getattr(args, 'doc_sim_pairs', 1000000))} ===")      # run.py:449-456
        if out_paths is not None and rank == 0:
            ckpt.save_teacher_table(out_paths[i], arr)                                          # run.py:458-459
            logging.info(f"teacher embedding saved at {out_paths[i]}")
        tables.append(arr)
        del model
    return tables
