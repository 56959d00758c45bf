"""Drop-in replacement for the reference's ``Tiny-NewsRec/model_bert.py`` on the B200 path.

Same class names, constructor arguments, forward signatures, sub-module attribute paths and
``state_dict`` keys as the reference (SURVEY.md section 8b), so ``run.py`` works by changing
``from model_bert import Model`` to ``from tinyrec.model_bert import Model``.  The modules
are parameter holders: the arithmetic runs in the sm_100a kernels of libtinyrec.so
(``tinyrec.engine`` / ``tinyrec.ops``); there is no PyTorch-op or CPU fallback.

Reference: Tiny-NewsRec/model_bert.py:8-34 (AttentionPooling), :103-137 (NewsEncoder),
:140-176 (UserEncoder), :179-205 (ModelBert), :208-244 (losses), :247-306 (Model);
tnlrv3/modeling.py:133-476,713-801 for the encoder parameter tree.
"""
import json

import torch
from torch import nn

from . import ops
from ._lib import TinyRecError
from .engine import F32, DropState, Encoder, FlatParams, _align8
from .synth import BERT_BASE

# ------------------------------------------------------------------------------------
# parameter-holder tree with the reference's attribute names
# ------------------------------------------------------------------------------------


class _Holder(nn.Module):
    def forward(self, *a, **k):  # pragma: no cover
        raise TinyRecError(f"{type(self).__name__} is a parameter holder; compute goes through the CUDA engine")


def _bert_init(module, std):
    """tnlrv3/modeling.py:41-51"""
    if isinstance(module, (nn.Linear, nn.Embedding)):
        module.weight.data.normal_(mean=0.0, std=std)
    elif isinstance(module, nn.LayerNorm):
        module.bias.data.zero_()
        module.weight.data.fill_(1.0)
    if isinstance(module, nn.Linear) and module.bias is not None:
        module.bias.data.zero_()


def load_bert_config(config_name, **over):
    cfg = dict(BERT_BASE, initializer_range=0.02)
    if config_name:
        with open(config_name, "r", encoding="utf-8") as f:
            cfg.update(json.load(f))
    cfg.update(over)
    return cfg


def _bert_layer(cfg):
    E, Fd, eps = cfg["hidden_size"], cfg["intermediate_size"], cfg["layer_norm_eps"]
    layer = _Holder()
    layer.attention = _Holder()
    layer.attention.self = _Holder()
    layer.attention.self.query = nn.Linear(E, E)
    layer.attention.self.key = nn.Linear(E, E)
    layer.attention.self.value = nn.Linear(E, E)
    layer.attention.output = _Holder()
    layer.attention.output.dense = nn.Linear(E, E)
    layer.attention.output.LayerNorm = nn.LayerNorm(E, eps=eps)
    layer.intermediate = _Holder()
    layer.intermediate.dense = nn.Linear(E, Fd)
    layer.output = _Holder()
    layer.output.dense = nn.Linear(Fd, E)
    layer.output.LayerNorm = nn.LayerNorm(E, eps=eps)
    return layer


def build_bert_model(cfg, num_layers):
    """Parameter tree of TuringNLRv3ForSequenceClassification (tnlrv3/modeling.py:713-723):
    ``bert.{embeddings,encoder.layer[i],pooler,rel_pos_bias}`` + ``classifier``.  The pooler and
    classifier are dead compute in the reference (model_bert.py:128-129 discards their
    outputs) but must exist so load_state_dict stays strict."""
    E = cfg["hidden_size"]
    m = _Holder()
    m.bert = _Holder()
    emb = _Holder()
    emb.word_embeddings = nn.Embedding(cfg["vocab_size"], E, padding_idx=0)
    emb.position_embeddings = nn.Embedding(cfg["max_position_embeddings"], E)
    emb.token_type_embeddings = nn.Embedding(cfg["type_vocab_size"], E)
    emb.LayerNorm = nn.LayerNorm(E, eps=cfg["layer_norm_eps"])
    m.bert.embeddings = emb
    m.bert.encoder = _Holder()
    m.bert.encoder.layer = nn.ModuleList([_bert_layer(cfg) for _ in range(num_layers)])
    m.bert.pooler = _Holder()
    m.bert.pooler.dense = nn.Linear(E, E)
    m.bert.rel_pos_bias = nn.Linear(cfg["rel_pos_bins"], cfg["num_attention_heads"], bias=False)
    m.classifier = nn.Linear(E, cfg.get("num_labels", 2))
    std = cfg.get("initializer_range", 0.02)
    m.apply(lambda mod: _bert_init(mod, std))
    return m


# ------------------------------------------------------------------------------------
# modules
# ------------------------------------------------------------------------------------
def precision_of(args):
    """``args.precision``: 'bf16' (the default: bf16 activations between the news-encoder kernels, TF32 user-encoder
    contractions, 1e-2 parity) or 'fp32' (fp32 news-encoder activations end to end and fp32-accurate user-encoder
    contractions, 1e-4 parity, inference only).  Reference args have no such field."""
    precision = getattr(args, "precision", "bf16")
    if precision not in ("bf16", "fp32"):
        raise TinyRecError(f"args.precision must be 'bf16' or 'fp32', got {precision!r}")
    return precision


class AttentionPooling(nn.Module):
    """model_bert.py:8-34.  Standalone ``forward`` handles fp32 [B, S, C] inputs (S <= 512)."""

    def __init__(self, emb_size, hidden_size):
        super().__init__()
        self.att_fc1 = nn.Linear(emb_size, hidden_size)
        self.att_fc2 = nn.Linear(hidden_size, 1)

    def forward(self, x, attn_mask=None):
        B, S, C = x.shape
        x = x.contiguous().float()
        mask = torch.ones(B, S, device=x.device, dtype=F32) if attn_mask is None else attn_mask.contiguous().float()
        out = torch.empty(B, C, device=x.device, dtype=F32)
        a = torch.empty(B, S, device=x.device, dtype=F32)
        ops.user_encoder_fwd(x.view(B * S, C), mask, self.att_fc1.bias, self.att_fc1.weight, self.att_fc1.bias,
                             self.att_fc2.weight.view(-1), self.att_fc2.bias, True, out, a, None, B, S)
        return out


class NewsEncoder(nn.Module):
    """model_bert.py:103-137 (``pooling='att'`` only; 'cls'/'mean' are out of scope, SURVEY.md section 2)."""

    def __init__(self, args, is_teacher=False, num_layers=None):
        super().__init__()
        if getattr(args, "pooling", "att") != "att":
            raise TinyRecError("only pooling='att' is on the supported hot path (demo.sh:28)")
        if getattr(args, "model_type", "tnlrv3") != "tnlrv3":
            raise TinyRecError("only model_type='tnlrv3' is supported (the reference's bert/roberta branch is broken)")
        if num_layers is None:
            num_layers = args.num_teacher_layers if is_teacher else args.num_student_layers
        self.pooling = args.pooling
        self.precision = precision_of(args)
        self.bert_config = load_bert_config(getattr(args, "config_name", None), num_hidden_layers=num_layers)
        self.bert_model = build_bert_model(self.bert_config, num_layers)
        model_name = getattr(args, "model_name", None)
        if model_name:
            # model_bert.py:114 ``model_class.from_pretrained(args.model_name, config=...)``: the encoder starts from the
            # UniLM / TNLRv3 ``.bin`` (layers beyond ``num_layers`` dropped, pooler / classifier keep their init).  A
            # name that cannot be loaded is an error -- silently training a random-init encoder is not a drop-in.
            import os
            from . import checkpoint
            if not os.path.isfile(model_name):
                raise TinyRecError(f"args.model_name={model_name!r} is not a file: pass the UniLM/TNLRv3 .bin the reference "
                                   "loads with from_pretrained, or model_name=None for a random-init encoder")
            missing, _ = checkpoint.load_unilm_bin(self.bert_model, model_name,
                                                   initializer_range=self.bert_config.get("initializer_range", 0.02))
            self.pretrained_missing_keys = missing
        self.attn = AttentionPooling(self.bert_config["hidden_size"], args.news_query_vector_dim)
        self.dense = nn.Linear(self.bert_config["hidden_size"], args.news_dim)
        self._engine = None
        self._flat = None           # set by the owning TrainState
        self._drop = None

    def drop_state(self, device):
        """Dropout state shared by every forward of this encoder (probabilities from the bert config;
        the reference's nn.Dropout modules, tnlrv3/modeling.py:177,223 + BertSelfOutput / BertOutput)."""
        if self._drop is None or self._drop.seed.device != device:
            c = self.bert_config
            self._drop = DropState(device, c.get("hidden_dropout_prob", 0.1), c.get("attention_probs_dropout_prob", 0.1))
        return self._drop

    def engine(self):
        if self._engine is None:
            self._engine = Encoder(self)
        return self._engine

    def forward(self, x, chunk=2048):
        """x int64 [n, 2L] (ids | mask) -> fp32 [n, news_dim].  Inference path (no autograd graph);
        training goes through ``Model`` / ``model_bert_2.ModelBert``."""
        if not x.is_cuda:
            raise TinyRecError("tinyrec NewsEncoder needs CUDA tensors (no CPU path)")
        eng = self.engine()
        if self.precision == "fp32":
            if self.training:
                raise TinyRecError("precision='fp32' is an inference mode (no fp32 dropout or backward kernels): "
                                   "call .eval() first")
            out = torch.empty(x.shape[0], eng.D, device=x.device, dtype=F32)
            for s in range(0, x.shape[0], chunk):
                eng.forward_fp32(x[s:s + chunk], out=out[s:s + chunk])
            return out
        flat = self._flat
        if flat is not None:
            if not flat.attached():
                flat = self._flat = None
            elif flat.stale():
                flat.refresh_shadow()
        n = x.shape[0]
        drop = None
        if self.training:                      # nn.Module semantics: dropout is active unless .eval() was called
            drop = self.drop_state(x.device)
        out = torch.empty(n, eng.D, device=x.device, dtype=F32)
        for s in range(0, n, chunk):
            if drop is not None:
                drop.advance()
            eng.forward(x[s:s + chunk], flat, out=out[s:s + chunk], drop=drop)
        return out


class MultiHeadSelfAttention(_Holder):
    """model_bert.py:63-100: parameter holder for W_Q / W_K / W_V (xavier-uniform weights, :73-76).
    The arithmetic is ``nrms_self_attention`` below (tnr_sgemm_nt + tnr_nrms_attn_fwd)."""

    def __init__(self, d_model, n_heads, d_k, d_v):
        super().__init__()
        if d_k != 16 or d_v != 16:
            raise TinyRecError("NRMS self-attention: d_k = d_v = 16 (as the reference hard-wires, model_bert.py:146)")
        self.d_model, self.n_heads, self.d_k, self.d_v = d_model, n_heads, d_k, d_v
        self.W_Q = nn.Linear(d_model, d_k * n_heads)
        self.W_K = nn.Linear(d_model, d_k * n_heads)
        self.W_V = nn.Linear(d_model, d_v * n_heads)
        for m in (self.W_Q, self.W_K, self.W_V):
            nn.init.xavier_uniform_(m.weight, gain=1)

    def stacked(self):
        """(W, b, stride_W, stride_b) for the batched (x3) projection GEMMs: the W_Q tensors themselves plus the
        element strides to W_K / W_V when the three parameters sit at a constant stride in memory (the flat training
        buffer keeps them contiguous), else a stacked [3, Dh, D] / [3, Dh] copy."""
        ws = [self.W_Q.weight, self.W_K.weight, self.W_V.weight]
        bs = [self.W_Q.bias, self.W_K.bias, self.W_V.bias]
        sw, sb = _const_stride(ws), _const_stride(bs)
        if sw is not None and sb is not None:
            return ws[0].detach(), bs[0].detach(), sw, sb
        Dh, D = ws[0].shape
        return (torch.stack([w.detach() for w in ws]).contiguous(), torch.stack([b.detach() for b in bs]).contiguous(),
                Dh * D, Dh)


def nrms_self_attention(mh, pad_doc, vecs, mask, use_mask, B, H, buf=None, fp32=False):
    """The NRMS front of ``UserEncoder.forward`` (model_bert.py:162-164, :169-173):
    vecs fp32 [B*H, D], mask fp32 [B, H] -> dict(xb = attention input, qkv [3, B*H, Dh], ctx [B*H, Dh],
    pool_mask = the mask the additive pooling applies: the log mask, or ones in the pad_doc branch).
    ``fp32``: the Q/K/V projections to fp32 accuracy (the attention itself is fp32 either way)."""
    R, D = vecs.shape
    Dh = mh.W_Q.weight.shape[0]
    dev = vecs.device
    buf = {} if buf is None else buf

    def get(name, *shape):
        t = buf.get(name)
        if t is None or tuple(t.shape) != shape:
            t = buf[name] = torch.empty(*shape, device=dev, dtype=F32)
        return t

    if use_mask:
        xb, pool_mask = vecs, mask
    else:
        xb = ops.nrms_blend_fwd(vecs, mask.reshape(-1), pad_doc.reshape(-1), get("xb", R, D))
        pool_mask = buf.get("ones")
        if pool_mask is None or tuple(pool_mask.shape) != (B, H):
            pool_mask = buf["ones"] = torch.ones(B, H, device=dev, dtype=F32)
    Wc, bc, sw, sb = mh.stacked()
    qkv = get("qkv", 3, R, Dh)
    ops.sgemm_nt(xb, Wc, bc, qkv, R, Dh, D, 3, 0, sw, sb, R * Dh, fp32=fp32)
    ctx = ops.nrms_attn_fwd(qkv, mask if use_mask else None, get("ctx", R, Dh), B, H)
    return dict(xb=xb, qkv=qkv, ctx=ctx, pool_mask=pool_mask, Wc=Wc, sw=sw)


class UserEncoder(nn.Module):
    """model_bert.py:140-176: additive attention over the clicked-news vectors (NAML), optionally behind
    the 16-dim-per-head self-attention (args.model == 'NRMS', :145-148).  With ``args.precision == 'fp32'`` every
    contraction of the forward is fp32-accurate (3xTF32 kernels; the flat TF32 scoring kernels are not used)."""

    def __init__(self, args):
        super().__init__()
        self.args = args
        self.precision = precision_of(args)
        self.nrms = getattr(args, "model", "NAML") == "NRMS"
        if self.nrms:
            self.multi_head_self_attn = MultiHeadSelfAttention(args.news_dim, args.num_attention_heads, 16, 16)
            self.attn = AttentionPooling(args.num_attention_heads * 16, args.user_query_vector_dim)
        else:
            self.attn = AttentionPooling(args.news_dim, args.user_query_vector_dim)
        self.pad_doc = nn.Parameter(torch.empty(1, args.news_dim).uniform_(-1, 1))

    def _packed_w1(self):
        """Packed TF32 image of att_fc1.weight (+ W1 pad_doc and the pad_doc logit) for the scoring kernels,
        re-packed when any of the parameters it is made from changes."""
        at = self.attn
        src = (at.att_fc1.weight, self.pad_doc, at.att_fc1.bias, at.att_fc2.weight)
        key = tuple((t.data_ptr(), t._version) for t in src) + (src[0].device, ops.param_generation)
        c = getattr(self, "_w1_pack", None)
        if c is None or c[0] != key:
            c = (key, ops.user_encoder_pack_w1(src[0].detach(), src[1].detach().view(-1), src[2].detach(),
                                               src[3].detach().view(-1)))
            object.__setattr__(self, "_w1_pack", c)
        return c[1]

    def _pool(self, v, idx, m, use_mask, B, H):
        """Additive pooling of v fp32 [B*H, D] (or table rows v[idx]) -> user fp32 [B, D]."""
        at = self.attn
        Q, D = at.att_fc1.weight.shape
        user = torch.empty(B, D, device=v.device, dtype=F32)
        a = torch.empty(B, H, device=v.device, dtype=F32)
        fp32 = self.precision == "fp32"
        if not fp32 and ops.user_encoder_score_supported(B, H, D, Q):   # scoring-sized batch: flat GEMM + pooling kernels
            return ops.user_encoder_score(v, idx, m, self.pad_doc.view(-1), self._packed_w1(), Q, at.att_fc1.bias,
                                          at.att_fc2.weight.view(-1), at.att_fc2.bias, use_mask, user, a, B, H)
        if idx is not None:
            return ops.user_encoder_fwd_gather(v, idx, m, self.pad_doc.view(-1), at.att_fc1.weight, at.att_fc1.bias,
                                               at.att_fc2.weight.view(-1), at.att_fc2.bias, use_mask, user, a, fp32=fp32)
        return ops.user_encoder_fwd(v, m, self.pad_doc.view(-1), at.att_fc1.weight, at.att_fc1.bias,
                                    at.att_fc2.weight.view(-1), at.att_fc2.bias, use_mask, user, a, None, B, H, fp32=fp32)

    def forward(self, news_vecs, log_mask=None):
        B, H, D = news_vecs.shape
        v = news_vecs.contiguous().float().view(B * H, D)
        m = log_mask.contiguous().float()
        use_mask = bool(self.args.user_log_mask)
        if self.nrms:
            fr = nrms_self_attention(self.multi_head_self_attn, self.pad_doc, v, m, use_mask, B, H,
                                     fp32=self.precision == "fp32")
            v, m, use_mask = fr["ctx"], fr["pool_mask"], True
        return self._pool(v, None, m, use_mask, B, H)

    def forward_gather(self, table, idx, log_mask):
        """``self(table[idx], log_mask)`` for the scoring loop (run.py:340-343, dataloader.py:292-301) with the
        gather fused into the user-encoder kernels: table fp32 [N+1, D], idx int32 [B, H] -> user fp32 [B, D]."""
        B, H = idx.shape
        if self.nrms:
            vecs = torch.empty(B * H, table.shape[1], device=table.device, dtype=F32)
            ops.gather_rows_f32(table, idx.reshape(-1), vecs)
            return self.forward(vecs.view(B, H, -1), log_mask)
        return self._pool(table, idx.contiguous(), log_mask.contiguous().float(), bool(self.args.user_log_mask), B, H)


# ------------------------------------------------------------------------------------
# training state shared by Model and model_bert_2.ModelBert
# ------------------------------------------------------------------------------------
class TrainState:
    """Flat parameter / gradient buffers + head workspaces of one trainable top-level model."""

    def __init__(self, news_encoder, user_encoder, teachers, transform, device):
        if getattr(news_encoder, "precision", "bf16") == "fp32":
            raise TinyRecError("the train step and Model.forward run the bf16 encoder; a news encoder with "
                               "precision='fp32' is for inference (NewsEncoder.forward, ModelBert.forward, table builds)")
        self.ne, self.ue, self.teachers, self.transform = news_encoder, user_encoder, teachers, transform
        self.enc = news_encoder.engine()
        self.enc.check_supported()
        enc_params = self.enc.trainable_order()
        at = user_encoder.attn
        head_all = [user_encoder.pad_doc, at.att_fc1.weight, at.att_fc1.bias, at.att_fc2.weight, at.att_fc2.bias]
        self.nrms = bool(getattr(user_encoder, "nrms", False))
        if self.nrms:      # [W_Q | W_K | W_V] and [b_Q | b_K | b_V] contiguous: one batched GEMM each way
            mh = user_encoder.multi_head_self_attn
            head_all += [mh.W_Q.weight, mh.W_K.weight, mh.W_V.weight, mh.W_Q.bias, mh.W_K.bias, mh.W_V.bias]
        head = [p for p in head_all if p.requires_grad]
        if head and len(head) != len(head_all):
            raise TinyRecError("the user encoder must be trainable or frozen as a whole")
        self.ue_trainable = bool(head)
        tparams = []
        for lin in transform:
            if lin.weight.requires_grad != lin.bias.requires_grad:
                raise TinyRecError("transform_matrix weight/bias must share requires_grad")
            if lin.weight.requires_grad:
                tparams += [lin.weight, lin.bias]
        self.tm_trainable = bool(tparams)
        if tparams and len(tparams) != 2 * len(transform):
            raise TinyRecError("transform_matrix modules must be trainable or frozen together")
        ordered = enc_params + head + tparams
        self.sig = tuple(id(p) for p in ordered)
        self.flat = FlatParams(ordered, device) if ordered else None
        self.head_begin = self.flat.off(head[0]) if head else (self.flat.off(tparams[0]) if tparams else (self.flat.numel if self.flat else 0))
        self.head_end = self.flat.numel if self.flat else 0
        self.stage = torch.zeros(max(self.head_end - self.head_begin, 1), device=device, dtype=F32)
        news_encoder._flat = self.flat
        self.hw = {}
        self.anchor = torch.zeros(1, device=device, requires_grad=True)
        self.comm_hook = None      # optional callable(flat) run at the end of backward (NCCL all-reduce)

    def valid(self, module):
        want = tuple(id(p) for p in _trainable_signature(module))
        if set(want) != set(self.sig):
            return False
        return self.flat is None or self.flat.attached()

    def _stage_view(self, p):
        o = self.flat.off(p) - self.head_begin
        return self.stage[o:o + p.numel()]

    def head_ws(self, B, H, K, M, D, Q, dev):
        key = (B, H, K, M)
        w = self.hw.get(key)
        if w is None:
            R = B * (H + K)
            mk = lambda *s: torch.empty(*s, device=dev, dtype=F32)  # noqa: E731
            w = dict(news=mk(R, D), user=mk(B, D), a=mk(B, H), e=mk(B, H, Q), ta=mk(max(M, 1), B, H), score=mk(B, K),
                     ue_scratch=mk(B * H * (Q + D)),
                     losses=torch.zeros(4 + 4 * B + 1, device=dev, dtype=F32), d_news=mk(R, D), d_user=mk(B, D),
                     T=mk(max(M, 1), R + B, D), TP=mk(max(M, 1), R + B, D), G=mk(max(M, 1), R + B, D))
            self.hw[key] = w
        return w

    # ---- one fused forward (+ eager head gradients) -------------------------------------------
    def step_forward(self, history, history_mask, candidate, label, th_list, tc_list, temperature, coef, use_mask,
                     want_grad, training=False):
        B, H, W = history.shape
        K = candidate.shape[1]
        M = len(th_list)
        dev = history.device
        flat = self.flat
        if flat is not None:
            if flat.stale():
                flat.refresh_shadow()
            if want_grad:
                flat.reattach_grads()
        x = _rows_of(history, candidate)
        D = self.enc.D
        Q = self.ue.attn.att_fc1.weight.shape[0]
        w = self.head_ws(B, H, K, M, D, Q, dev)
        R = B * (H + K)
        drop = None
        if training:
            drop = self.ne.drop_state(dev)
            drop.advance()
        news = self.enc.forward(x, flat, save=want_grad, out=w["news"], drop=drop)
        mask = history_mask.contiguous().float()
        label = label.contiguous()
        at = self.ue.attn
        T, TP, G = w["T"], w["TP"], w["G"]
        # teacher rows that the device loader already gathered into the [M, R + B, D] layout are used where they are
        ext = getattr(th_list, "ext", None)
        adopted = (M > 0 and ext is not None and ext is getattr(tc_list, "ext", None) and ext.is_cuda
                   and tuple(ext.shape) == tuple(T.shape) and ext.dtype == F32 and ext.is_contiguous())
        if adopted:
            T = ext
        pool_vecs, pool_mask, pool_use_mask = news[:B * H], mask, use_mask
        if self.nrms:       # self-attention in front of every pooling (model_bert.py:162-164, :171-173)
            nb = w.setdefault("nrms", [dict() for _ in range(1 + M)])
            fr = w["fr"] = nrms_self_attention(self.ue.multi_head_self_attn, self.ue.pad_doc, news[:B * H], mask, use_mask,
                                               B, H, nb[0])
            if fr["ctx"].shape[1] != D:
                raise TinyRecError("NRMS: num_attention_heads * 16 must equal news_dim (the click score is a dot product)")
            pool_vecs, pool_mask, pool_use_mask = fr["ctx"], fr["pool_mask"], True
        encs = [dict(vecs=pool_vecs, pad_doc=self.ue.pad_doc.view(-1), W1=at.att_fc1.weight, b1=at.att_fc1.bias,
                     w2=at.att_fc2.weight.view(-1), b2=at.att_fc2.bias, user=w["user"], a=w["a"], e=w["e"])]
        for i in range(M):
            if not adopted:
                T[i, :B * H].copy_(th_list[i].reshape(B * H, D))
                T[i, B * H:R].copy_(tc_list[i].reshape(B * K, D))
            t = self.teachers[i]
            tv = T[i, :B * H]
            if self.nrms:
                tv = nrms_self_attention(t.multi_head_self_attn, t.pad_doc, tv, mask, use_mask, B, H, nb[1 + i])["ctx"]
            encs.append(dict(vecs=tv, pad_doc=t.pad_doc.view(-1), W1=t.attn.att_fc1.weight, b1=t.attn.att_fc1.bias,
                             w2=t.attn.att_fc2.weight.view(-1), b2=t.attn.att_fc2.bias, user=T[i, R:], a=w["ta"][i], e=None))
        ops.user_encoder_fwd_multi(encs, pool_mask, pool_use_mask, B, H)
        if M:
            ws, bs = [lin.weight for lin in self.transform], [lin.bias for lin in self.transform]
            sw, sb = _const_stride(ws), _const_stride(bs)
            if sw is not None and sb is not None:
                ops.sgemm_nt(T, ws[0], bs[0], TP, R + B, D, D, M, (R + B) * D, sw, sb, (R + B) * D)
            else:
                for i in range(M):
                    ops.sgemm_nt(T[i], ws[i], bs[i], TP[i], R + B, D, D, 1, 0, 0, 0, 0)
        ops.kd_loss(news, w["user"], label, T if M else None, TP if M else None, M, B, H, K, D, temperature, coef,
                    want_grad, w["score"], w["losses"], w["d_news"], w["d_user"], G if M else None)
        if want_grad:
            self.stage.zero_()
            if self.ue_trainable:
                sv = self._stage_view
                dpad, dW1, db1, dw2, db2 = (sv(self.ue.pad_doc), sv(at.att_fc1.weight), sv(at.att_fc1.bias),
                                            sv(at.att_fc2.weight), sv(at.att_fc2.bias))
            else:
                scratch = torch.zeros(D + Q * D + 2 * Q + 1, device=dev, dtype=F32)
                dpad, dW1, db1 = scratch[:D], scratch[D:D + Q * D], scratch[D + Q * D:D + Q * D + Q]
                dw2, db2 = scratch[D + Q * D + Q:D + Q * D + 2 * Q], scratch[D + Q * D + 2 * Q:]
            if not self.nrms:
                ops.user_encoder_bwd(news[:B * H], mask, self.ue.pad_doc.view(-1), at.att_fc1.weight, at.att_fc2.weight.view(-1),
                                     use_mask, w["a"], w["e"], w["d_user"], w["d_news"], dpad, dW1, db1, dw2, db2, w["ue_scratch"],
                                     B, H)
            else:
                self._nrms_backward(w, mask, use_mask, dpad, dW1, db1, dw2, db2, B, H, D)
            if self.tm_trainable and M:
                gw = [self._stage_view(lin.weight) for lin in self.transform]
                gb = [self._stage_view(lin.bias) for lin in self.transform]
                sw, sb = _const_stride(gw), _const_stride(gb)
                if sw is not None and sb is not None:
                    ops.sgemm_tn_acc(G, T, gw[0], gb[0], R + B, D, D, M, (R + B) * D, (R + B) * D, sw, sb)
                else:
                    for i in range(M):
                        ops.sgemm_tn_acc(G[i], T[i], gw[i], gb[i], R + B, D, D, 1, 0, 0, 0, 0)
        self.last = w
        return w

    def _nrms_backward(self, w, mask, use_mask, dpad, dW1, db1, dw2, db2, B, H, D):
        """d_user -> pooling bwd -> self-attention bwd -> W_Q/K/V gradients, input gradient, pad_doc blend bwd."""
        fr, at, mh = w["fr"], self.ue.attn, self.ue.multi_head_self_attn
        Rh, Dh, dev = B * H, fr["ctx"].shape[1], mask.device
        nb = w["nrms"][0]
        for name, shape in (("d_ctx", (Rh, Dh)), ("dqkv", (3, Rh, Dh)), ("dxb", (Rh, D))):
            if name not in nb:
                nb[name] = torch.empty(*shape, device=dev, dtype=F32)
        d_ctx = nb["d_ctx"].zero_()
        ops.user_encoder_bwd(fr["ctx"], fr["pool_mask"], self.ue.pad_doc.view(-1), at.att_fc1.weight, at.att_fc2.weight.view(-1),
                             True, w["a"], w["e"], w["d_user"], d_ctx, dpad, dW1, db1, dw2, db2, w["ue_scratch"], B, H)
        ops.nrms_attn_bwd(fr["qkv"], mask if use_mask else None, d_ctx, nb["dqkv"], B, H)
        if self.ue_trainable:      # stage views keep the flat buffer's [W_Q | W_K | W_V] / [b_Q | b_K | b_V] layout
            o = self.flat.off(mh.W_Q.weight) - self.head_begin
            gW = self.stage[o:o + 3 * Dh * D]
            o = self.flat.off(mh.W_Q.bias) - self.head_begin
            gb = self.stage[o:o + 3 * Dh]
            if self.flat.off(mh.W_V.weight) - self.flat.off(mh.W_Q.weight) != 2 * Dh * D or \
                    self.flat.off(mh.W_V.bias) - self.flat.off(mh.W_Q.bias) != 2 * Dh:
                raise TinyRecError("NRMS: W_Q / W_K / W_V are not contiguous in the flat buffer")
            ops.sgemm_tn_acc(nb["dqkv"], fr["xb"], gW, gb, Rh, Dh, D, 3, Rh * Dh, 0, Dh * D, Dh)
        ops.sgemm_nn(nb["dqkv"], fr["Wc"], nb["dxb"], Rh, D, Dh, 3, Rh * Dh, fr["sw"])
        ops.nrms_blend_bwd(nb["dxb"], None if use_mask else mask.reshape(-1), w["d_news"][:Rh], dpad)

    def step_backward(self, g_total):
        """Upstream gradient of the total loss (a device scalar) -> encoder backward + staged head grads."""
        w = self.last
        flat = self.flat
        w["d_news"].mul_(g_total)
        if self.head_end > self.head_begin:
            self.stage.mul_(g_total)
            flat.grad[self.head_begin:self.head_end].add_(self.stage[:self.head_end - self.head_begin])
        if self.comm_hook is None:
            self.enc.backward(w["d_news"], flat)
            return
        # Bucketed exchange: the flat buffer is laid out [layer low | ... | layer top | pooling head | user
        # encoder | transform_matrix] and the backward finishes it from the END: once layer i is done,
        # everything from its first parameter up to the previous bucket start is final.  The LOWEST trainable layer
        # has no later backward work to overlap with, so it reports its four contiguous parameter ranges one by one
        # (on_grads_ready) and only its smallest range trails the backward.
        done_to = [flat.numel]
        sent = []                      # [lo, hi) ranges of the lowest layer already handed to the hook

        def layer_done(i):
            lo = flat.off(self.enc.layers[i].q.weight)
            if lo >= done_to[0]:
                return
            if sent:                   # the lowest layer went out range by range: send what is left around them
                cur = lo
                for a, b in sorted(sent):
                    if a > cur:
                        self.comm_hook(flat, cur, a)
                    cur = max(cur, b)
                if done_to[0] > cur:
                    self.comm_hook(flat, cur, done_to[0])
            else:
                self.comm_hook(flat, lo, done_to[0])
            done_to[0] = lo

        def grads_ready(first, last):
            if not sent:               # everything above this layer (a single trainable layer: the heads) is final
                lr_low = self.enc.layers[self.enc.lowest_trainable_layer()]
                top = _align8(flat.off(lr_low.ln2.bias) + lr_low.ln2.bias.numel())
                if done_to[0] > top:
                    self.comm_hook(flat, top, done_to[0])
                    done_to[0] = top
            lo, hi = flat.off(first), _align8(flat.off(last) + last.numel())
            hi = min(hi, done_to[0])
            if hi > lo:
                self.comm_hook(flat, lo, hi)
                sent.append((lo, hi))

        self.enc.backward(w["d_news"], flat, on_layer_done=layer_done,
                          on_grads_ready=grads_ready if getattr(self, "fine_grained_comm", True) else None)
        if done_to[0] > 0:
            self.comm_hook(flat, 0, done_to[0])


def _rows_of(history, candidate):
    """[history rows | candidate rows] as one int64 [B (H + K), 2L] matrix: the tensors themselves when the device
    loader produced them adjacent in one buffer (tinyrec.dataloader.TrainBatcher), else a concatenated copy."""
    B, H, W = history.shape
    K = candidate.shape[1]
    if (history.is_contiguous() and candidate.is_contiguous() and history.dtype == candidate.dtype
            and history.untyped_storage().data_ptr() == candidate.untyped_storage().data_ptr()
            and candidate.storage_offset() == history.storage_offset() + B * H * W):
        return torch.as_strided(history, (B * (H + K), W), (W, 1))
    return torch.cat([history.reshape(B * H, W), candidate.reshape(B * K, W)], 0)


def _const_stride(tensors):
    """Element stride between consecutive fp32 tensors of a list if it is constant and 16-byte
    aligned (the flat buffer keeps transform_matrix.{i} that way), else None."""
    if len(tensors) == 1:
        return 0
    base = tensors[0].data_ptr()
    d = tensors[1].data_ptr() - base
    if d <= 0 or d % 16:
        return None
    for i, t in enumerate(tensors):
        if t.data_ptr() - base != i * d or not t.is_contiguous():
            return None
    return d // 4


def _trainable_signature(module):
    return [p for p in module.parameters() if p.requires_grad]


class _StepFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, anchor, state, args):
        w = state.step_forward(*args)
        ctx.state = state
        losses = w["losses"]
        return losses[3].clone(), losses[0].clone(), losses[1].clone(), losses[2].clone(), w["score"].clone()

    @staticmethod
    def backward(ctx, g_total, g_distill, g_emb, g_target, g_score):
        ctx.state.step_backward(g_total)
        return None, None, None


def _get_state(module, build):
    st = getattr(module, "_tnr_state", None)
    if st is None or not st.valid(module):
        st = build()
        object.__setattr__(module, "_tnr_state", st)
    return st


class ModelBert(nn.Module):
    """model_bert.py:179-205: (score, history_vecs, candidate_vecs, user_vec).  Inference semantics
    (outputs carry no autograd graph); the training entry points are ``Model.forward`` and
    ``tinyrec.model_bert_2.ModelBert.forward``."""

    def __init__(self, args, is_teacher=False):
        super().__init__()
        self.args = args
        self.news_encoder = NewsEncoder(args, is_teacher)
        self.user_encoder = UserEncoder(args)

    def forward(self, history, history_mask, candidate):
        B, H, W = history.shape
        K = candidate.shape[1]
        x = torch.cat([history.reshape(B * H, W), candidate.reshape(B * K, W)], 0)
        vec = self.news_encoder(x)
        hist = vec[:B * H].view(B, H, -1)
        cand = vec[B * H:].view(B, K, -1)
        user = self.user_encoder(hist, history_mask)
        w = torch.zeros(4 + 4 * B + 1, device=vec.device, dtype=F32)
        score = torch.empty(B, K, device=vec.device, dtype=F32)
        label = torch.zeros(B, device=vec.device, dtype=torch.int64)
        ops.kd_loss(vec, user, label, None, None, 0, B, H, K, vec.shape[1], 1.0, 1.0, False, score, w, None, None, None)
        return score, hist, cand, user


def kd_ce_loss(logits_S, logits_T, temperature=1):
    """model_bert.py:208-219.  Kept for API completeness (tiny torch expression on the caller's
    tensors); the training path computes it inside tnr_kd_loss_fwdbwd."""
    p_T = torch.softmax(logits_T / temperature, dim=-1)
    return -(p_T * torch.log_softmax(logits_S / temperature, dim=-1)).sum(dim=-1).mean()


def hid_mse_loss(state_S, state_T, mask=None, reduce=True):
    """model_bert.py:222-244 (API completeness; see kd_ce_loss)."""
    se = (state_S - state_T) ** 2
    if mask is None:
        return se.mean() if reduce else se.mean(dim=-1)
    if not reduce:
        return (se * mask.unsqueeze(-1)).mean(dim=-1)
    return (se * mask.unsqueeze(-1)).sum() / (mask.sum() * state_S.size(-1))


class Model(nn.Module):
    """model_bert.py:247-306: multi-teacher KD wrapper.
    forward(...) -> (total_loss, distill_loss, emb_loss, target_loss, student_score); only
    ``total_loss`` carries gradient (that is all run.py:194 back-propagates)."""

    def __init__(self, args):
        super().__init__()
        self.args = args
        self.teachers = nn.ModuleList([UserEncoder(args) for _ in range(args.num_teachers)])
        self.student = ModelBert(args, is_teacher=False)
        self.target_loss_fn = nn.CrossEntropyLoss()
        self.transform_matrix = nn.ModuleList([nn.Linear(args.news_dim, args.news_dim) for _ in range(args.num_teachers)])
        for module in self.transform_matrix:
            nn.init.xavier_uniform_(module.weight, gain=1.0)
            nn.init.constant_(module.bias, 0.0)

    def train_state(self):
        dev = self.transform_matrix[0].weight.device if len(self.transform_matrix) else self.student.user_encoder.pad_doc.device
        if dev.type != "cuda":
            raise TinyRecError("tinyrec Model needs its parameters on a CUDA device (no CPU path)")
        return _get_state(self, lambda: TrainState(self.student.news_encoder, self.student.user_encoder,
                                                   list(self.teachers), list(self.transform_matrix), dev))

    def forward(self, history, history_mask, candidate, label, teacher_history_embs, teacher_candidate_embs):
        st = self.train_state()
        want_grad = torch.is_grad_enabled() and st.flat is not None
        keep = lambda t: t if isinstance(t, list) else list(t)  # noqa: E731  (TeacherViews carries the loader's buffer)
        args = (history, history_mask, candidate, label, keep(teacher_history_embs), keep(teacher_candidate_embs),
                float(self.args.temperature), float(self.args.coef), bool(self.args.user_log_mask), want_grad,
                bool(self.training))
        if want_grad:
            return _StepFn.apply(st.anchor, st, args)
        w = st.step_forward(*args)
        ls = w["losses"]
        return ls[3].clone(), ls[0].clone(), ls[1].clone(), ls[2].clone(), w["score"].clone()
