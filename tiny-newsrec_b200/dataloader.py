"""Device-resident batch assembly.

The reference assembles every batch on the host with numpy fancy indexing per impression and
ships the gathered token rows / teacher embeddings to the GPU
(Tiny-NewsRec/dataloader.py:118-172 train, :285-314 eval).  Here the tables live in HBM
(news tokens int32 [N+1, 2L] 38 MB, M teacher tables fp32 [N+1, D] 165 MB each) and only the
index arrays cross PCIe; the row gathers are the bit-exact kernels tnr_gather_rows_*.

Host-side index logic (id -> row, front padding, label insertion) keeps the reference
semantics: unknown id -> row 0; keep the last ``user_log_length`` clicks; left-pad with 0;
mask = [0..0, 1..1]; candidates = neg[:label] + pos + neg[label:].
"""
import random

import numpy as np
import torch

from . import ops
from ._lib import TinyRecError


def trans_to_nindex(nids, news_index):
    """dataloader.py:73-74"""
    get = news_index.get
    return [get(i, 0) for i in nids]


def pad_to_fix_len(x, fix_length, padding_front=True, padding_value=0):
    """dataloader.py:76-83"""
    n = len(x)
    keep = x[-fix_length:]
    fill = [padding_value] * (fix_length - n)
    ones = [1] * min(fix_length, n)
    zeros = [0] * (fix_length - n)
    if padding_front:
        return fill + keep, zeros + ones
    return keep + fill, ones + zeros


def parse_train_line(line, news_index, user_log_length, npratio, rng=random):
    """One ``behaviors_np{K}_*.tsv`` line -> (hist_idx, hist_mask, cand_idx, label)
    (dataloader.py:124-137)."""
    cols = line.decode("utf-8").split("\t") if isinstance(line, bytes) else line.split("\t")
    hist, mask = pad_to_fix_len(trans_to_nindex(cols[3].split(), news_index), user_log_length)
    pos = trans_to_nindex(cols[4].split(), news_index)
    neg = trans_to_nindex(cols[5].split(), news_index)
    label = rng.randint(0, npratio)
    return hist, mask, neg[:label] + pos + neg[label:], label


def parse_eval_line(line, news_index, user_log_length):
    """One ``behaviors_*.tsv`` line -> (hist_idx, hist_mask, cand_idx, labels) (dataloader.py:289-299)."""
    cols = line.decode("utf-8").split("\t") if isinstance(line, bytes) else line.split("\t")
    hist, mask = pad_to_fix_len(trans_to_nindex(cols[3].split(), news_index), user_log_length)
    imps = cols[4].split()
    cand = trans_to_nindex([i.split("-")[0] for i in imps], news_index)
    labels = [int(i.split("-")[1]) for i in imps]
    return hist, mask, cand, labels


def parse_test_line(line, news_index, user_log_length):
    """One ``behaviors.tsv`` line, labelled or not -> (imp_id, hist_idx, hist_mask, cand_idx).  MIND's test split lists
    bare candidate ids (``N123 N456``); a ``-0`` / ``-1`` label suffix, as in the dev split, is dropped, so a dev file
    gives the same arrays as its unlabeled copy."""
    cols = line.decode("utf-8").split("\t") if isinstance(line, bytes) else line.split("\t")
    hist, mask = pad_to_fix_len(trans_to_nindex(cols[3].split(), news_index), user_log_length)
    cand = trans_to_nindex([i[:-2] if i.endswith(("-0", "-1")) else i for i in cols[4].split()], news_index)
    return int(cols[0]), hist, mask, cand


def pack_test_lines(lines, news_index, user_log_length):
    """``parse_test_line`` over many lines (blank lines skipped) -> the arrays ``run.predict`` / ``run.predict_test``
    take: (imp_ids int64 [n], hist_idx int32 [n, H], hist_mask fp32 [n, H], cand_ptr int64 [n+1], cand_idx int32
    [nnz])."""
    rows = [parse_test_line(ln, news_index, user_log_length) for ln in lines if ln.strip()]
    H = user_log_length
    imp_ids = np.array([r[0] for r in rows], dtype=np.int64)
    hist = np.array([r[1] for r in rows], dtype=np.int32).reshape(len(rows), H)
    mask = np.array([r[2] for r in rows], dtype=np.float32).reshape(len(rows), H)
    cand_ptr = np.zeros(len(rows) + 1, dtype=np.int64)
    np.cumsum([len(r[3]) for r in rows], out=cand_ptr[1:])
    cand = np.fromiter((c for r in rows for c in r[3]), dtype=np.int32, count=int(cand_ptr[-1]))
    return imp_ids, hist, mask, cand_ptr, cand


class DeviceTables:
    """News token table and teacher embedding tables resident in HBM."""

    def __init__(self, news_combined, teacher_embs=(), device="cuda"):
        nc = torch.as_tensor(np.ascontiguousarray(news_combined))
        if nc.dtype != torch.int32:
            raise TinyRecError("news_combined must be int32 [N+1, 2L] (preprocess.py:49-53)")
        self.news = nc.to(device)
        self.teachers = [torch.as_tensor(np.ascontiguousarray(t), dtype=torch.float32).to(device) for t in teacher_embs]
        self.device = self.news.device


class TeacherViews(list):
    """The per-teacher [B, H, D] / [B, K, D] views ``TrainBatcher.assemble`` returns, remembering the buffer they are
    views of (``ext`` fp32 [M, B (H + K) + B, D]: history rows | candidate rows | room for the teachers' user vectors) --
    exactly the layout ``Model.forward`` keeps its teacher matrices in, so the model adopts it instead of copying."""
    ext = None


class TrainBatcher:
    """indices -> the six tensors ``Model.forward`` takes, gathered on the device by ONE kernel launch."""

    def __init__(self, tables, B, H, K):
        self.t, self.B, self.H, self.K = tables, B, H, K
        dev, W = tables.device, tables.news.shape[1]
        M = len(tables.teachers)
        D = tables.teachers[0].shape[1] if M else 4
        R = B * (H + K)
        self.tokens = torch.empty(R, W, device=dev, dtype=torch.int64)            # [history rows | candidate rows]
        self.history = self.tokens[:B * H].view(B, H, W)
        self.candidate = self.tokens[B * H:].view(B, K, W)
        self.ext = torch.zeros(max(M, 1), R + B, D, device=dev, dtype=torch.float32)
        self.th, self.tc = TeacherViews(), TeacherViews()
        for i in range(M):
            self.th.append(self.ext[i, :B * H].view(B, H, D))
            self.tc.append(self.ext[i, B * H:R].view(B, K, D))
        self.th.ext = self.tc.ext = self.ext
        self.M = M

    def assemble(self, hist_idx, cand_idx):
        """hist_idx int32 [B,H], cand_idx int32 [B,K] (CUDA) -> history, candidate, [th], [tc]."""
        if hist_idx.numel() != self.B * self.H or cand_idx.numel() != self.B * self.K:
            raise TinyRecError("TrainBatcher.assemble: index shapes do not match the batcher's (B, H, K)")
        ops.train_batch_gather(self.t.news, self.t.teachers, hist_idx.reshape(-1), cand_idx.reshape(-1), self.tokens,
                               [self.ext[i] for i in range(self.M)])
        return self.history, self.candidate, self.th, self.tc


def gather_history_vecs(news_scoring, hist_idx, out=None):
    """news_scoring fp32 [N+1, D] (CUDA), hist_idx int32 [B,H] -> log_vecs fp32 [B,H,D]
    (dataloader.py:295)."""
    B, H = hist_idx.shape
    D = news_scoring.shape[1]
    if out is None:
        out = torch.empty(B, H, D, device=news_scoring.device, dtype=torch.float32)
    ops.gather_rows_f32(news_scoring, hist_idx.reshape(-1), out.view(-1, D))
    return out
