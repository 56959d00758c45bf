"""Orchestration of the CUDA path: flat parameter / gradient buffers, bf16 shadow weights,
activation workspaces and the forward / backward kernel sequences of the news encoder and
of the scoring + KD head.  Pure plumbing: every arithmetic op is a kernel behind the C ABI
(tinyrec.ops); torch supplies device memory, streams and views.

Reference call stacks this replaces: SURVEY.md section 3.1 (train step), 3.2 (table build).
"""
import math

import torch

from . import ops
from ._lib import TinyRecError

BF = torch.bfloat16
F32 = torch.float32
LN_EPS = 1e-12            # tnlrv3/configuration_tnlrv3.py:61

# dropout tensor ids ("sites", include/tinyrec.h tnr_dropout.site): one Philox stream per tensor
SITE_EMB = 0              # embeddings output, tnlrv3/modeling.py:177
KIND_ATTN, KIND_ATT_OUT, KIND_FFN_OUT = 0, 1, 2    # attention probs :223; BertSelfOutput / BertOutput dense


def drop_site(layer, kind):
    return 8 * (layer + 1) + kind


class DropState:
    """Training-mode dropout of the encoder: probabilities from the model config and a device-resident
    64-bit seed that advances once per forward (the backward of the same step regenerates the masks
    from it; a captured CUDA graph replays with a fresh seed)."""

    def __init__(self, device, p_hidden=0.1, p_attn=0.1, seed=None):
        self.p_hidden, self.p_attn = float(p_hidden), float(p_attn)
        if seed is None:
            seed = torch.initial_seed() & 0x7FFFFFFFFFFFFFFF
        self.seed = torch.tensor([seed], device=device, dtype=torch.int64)

    def advance(self):
        self.seed.add_(1)

    def make(self, site, p):
        return ops.make_drop(self.seed, site, p)

    def offset(self, site_base):
        """A view of this state whose tensor ids are shifted by ``site_base``: a second encoder pass of the same step
        (the title pass after the body pass of the post-training models) draws masks independent of the first's, as
        the reference's ``nn.Dropout`` does for every ``news_encoder`` call."""
        return _DropView(self, site_base)


class _DropView:
    def __init__(self, state, site_base):
        self.p_hidden, self.p_attn, self.seed, self.site_base = state.p_hidden, state.p_attn, state.seed, int(site_base)

    def make(self, site, p):
        return ops.make_drop(self.seed, site + self.site_base, p)


def _align8(n):
    return (n + 7) // 8 * 8


def rel_pos_bucket_table(L, num_buckets=32, max_distance=128):
    """int64 [L, L] bucket of (pos_j - pos_i); host-side restatement of
    tnlrv3/modeling.py:345-373 for position_ids = arange(L) (batch-invariant)."""
    pos = torch.arange(L)
    rel = pos[None, :] - pos[:, None]
    half = num_buckets // 2
    ret = (rel > 0).long() * half
    n = rel.abs()
    exact = half // 2
    big = exact + (torch.log(n.float() / exact) / math.log(max_distance / exact) * (half - exact)).to(torch.long)
    big = torch.min(big, torch.full_like(big, half - 1))
    return ret + torch.where(n < exact, n, big)


class LayerRefs:
    """Parameter handles of one BertLayer, by the reference's attribute names."""

    def __init__(self, layer):
        s, a = layer.attention.self, layer.attention.output
        self.q, self.k, self.v = s.query, s.key, s.value
        self.o, self.ln1 = a.dense, a.LayerNorm
        self.f1, self.f2, self.ln2 = layer.intermediate.dense, layer.output.dense, layer.output.LayerNorm

    def params(self):
        return [self.q.weight, self.k.weight, self.v.weight, self.q.bias, self.k.bias, self.v.bias,
                self.o.weight, self.o.bias, self.ln1.weight, self.ln1.bias,
                self.f1.weight, self.f1.bias, self.f2.weight, self.f2.bias, self.ln2.weight, self.ln2.bias]


class FlatParams:
    """Trainable parameters re-homed into one flat fp32 buffer (+ flat grad, + bf16 shadow).

    The order keeps [Wq, Wk, Wv] and [bq, bk, bv] of a layer contiguous so the fused QKV GEMM,
    its wgrad and the Adam kernel all address them as one [3E, E] / [3E] tensor, and keeps
    transform_matrix.{i}.{weight,bias} at a constant stride for the batched fp32 GEMMs."""

    def __init__(self, ordered_params, device):
        self.params = ordered_params
        self.offsets = []
        off = 0
        for p in ordered_params:
            self.offsets.append(off)
            off += p.numel()
            # keep every tensor 8-element aligned unless the next one must stay contiguous
            off = _align8(off)
        self.numel = off
        self.data = torch.zeros(off, device=device, dtype=F32)
        # Data-parallel runs keep the gradient buffer in symmetric (peer-mapped) memory so that the exchange can be one
        # kernel over NVLink peer memory (tinyrec.parallel.SymmetricGradBuffer / tnr_allreduce_p2p); any failure to set
        # that up leaves a plain buffer and the NCCL all-reduce.
        self.symm, self.symm_error = None, None
        from . import parallel as _par
        if _par.SymmetricGradBuffer.wanted() and torch.device(device).type == "cuda":
            try:
                self.symm = _par.SymmetricGradBuffer(off, torch.device(device))
            except Exception as exc:  # noqa: BLE001  (reported by bench.py / the tests, not hidden)
                self.symm, self.symm_error = None, f"{type(exc).__name__}: {exc}"
        self.grad = self.symm.grad if self.symm is not None else torch.zeros(off, device=device, dtype=F32)
        self.shadow = torch.zeros(off, device=device, dtype=BF)
        for p, o in zip(ordered_params, self.offsets):
            view = self.data[o:o + p.numel()].view(p.shape)
            view.copy_(p.data)
            p.data = view
            p.grad = self.grad[o:o + p.numel()].view(p.shape)
        self._index = {id(p): i for i, p in enumerate(ordered_params)}
        self.refresh_shadow()

    def refresh_shadow(self):
        ops.cast_f32_bf16(self.data, self.shadow)
        self.versions = [p._version for p in self.params]

    def stale(self):
        return any(p._version != v for p, v in zip(self.params, self.versions))

    def attached(self):
        """True while every parameter still lives in the flat buffers (a `.to()` / `.cuda()` or an
        optimizer that replaced `.data` / `.grad` breaks this and forces a rebuild)."""
        for p, o in zip(self.params, self.offsets):
            if p.data_ptr() != self.data.data_ptr() + 4 * o:
                return False
        return True

    def reattach_grads(self):
        for p, o in zip(self.params, self.offsets):
            g = p.grad
            if g is None or g.data_ptr() != self.grad.data_ptr() + 4 * o:
                view = self.grad[o:o + p.numel()].view(p.shape)
                if g is None:
                    view.zero_()
                else:
                    view.copy_(g)
                p.grad = view

    def has(self, p):
        return id(p) in self._index

    def off(self, p):
        return self.offsets[self._index[id(p)]]

    def w_shadow(self, p, rows=None):
        o = self.off(p)
        n = p.numel() if rows is None else rows * p.shape[1]
        return self.shadow[o:o + n].view(-1, p.shape[1])

    def g_view(self, p, numel=None, shape=None):
        o = self.off(p)
        n = p.numel() if numel is None else numel
        v = self.grad[o:o + n]
        return v.view(shape) if shape is not None else v.view(p.shape) if numel is None else v


class _Frozen:
    """bf16 / fp32 device copies of frozen tensors, refreshed when the source `_version` or
    storage changes (e.g. after load_state_dict), or when ``gen`` changes (callers pass
    ops.param_generation for copies of parameters the fused Adam may have rewritten)."""

    def __init__(self):
        self.cache = {}

    def get(self, key, tensors, build, gen=None):
        sig = tuple((t.data_ptr(), t._version) for t in tensors) + (gen,)
        hit = self.cache.get(key)
        if hit is not None and hit[0] == sig:
            return hit[1]
        val = build()
        self.cache[key] = (sig, val)
        return val


class Encoder:
    """News encoder (TNLRv3 layers + word pooling + dense) on the CUDA path."""

    def __init__(self, news_encoder_module):
        self.mod = news_encoder_module
        bert = news_encoder_module.bert_model.bert
        self.bert = bert
        self.layers = [LayerRefs(l) for l in bert.encoder.layer]
        self.E = bert.embeddings.word_embeddings.weight.shape[1]
        self.A = bert.rel_pos_bias.weight.shape[0]
        self.F = self.layers[0].f1.weight.shape[0] if self.layers else 4 * self.E
        self.Q = news_encoder_module.attn.att_fc1.weight.shape[0]
        self.D = news_encoder_module.dense.weight.shape[0]
        # numerics the reference reads from the bert config (tnlrv3/configuration_tnlrv3.py:61, modeling.py:458-461)
        cfg = getattr(news_encoder_module, "bert_config", None) or {}
        self.ln_eps = float(cfg.get("layer_norm_eps", LN_EPS))
        self.rel_bins = int(cfg.get("rel_pos_bins", 32))
        self.max_rel = int(cfg.get("max_rel_pos", 128))
        if bert.rel_pos_bias.weight.shape[1] != self.rel_bins:
            raise TinyRecError(f"rel_pos_bias has {bert.rel_pos_bias.weight.shape[1]} buckets, config says {self.rel_bins}")
        self.frozen = _Frozen()
        self.ws = {}
        self.scratch_ln = None

    # ---- parameter access ---------------------------------------------------------
    def bottom_params(self):
        """The tensors below the first BertLayer, in flat-buffer order: the embedding block and the rel-pos bias
        table every layer shares."""
        emb = self.bert.embeddings
        return [emb.word_embeddings.weight, emb.position_embeddings.weight, emb.token_type_embeddings.weight,
                emb.LayerNorm.weight, emb.LayerNorm.bias, self.bert.rel_pos_bias.weight]

    def bottom_trainable(self):
        return any(p.requires_grad for p in self.bottom_params())

    def trainable_order(self):
        """Trainable parameters of the encoder in flat-buffer order: the trainable bottom tensors first, then whole
        BertLayers from the lowest up, then the word pooling and the dense head."""
        ln = self.bert.embeddings.LayerNorm
        if ln.weight.requires_grad != ln.bias.requires_grad:
            raise TinyRecError("embeddings.LayerNorm weight and bias must be trainable or frozen together")
        out = [p for p in self.bottom_params() if p.requires_grad]
        for lr in self.layers:
            ps = lr.params()
            flags = [p.requires_grad for p in ps]
            if any(flags):
                if not all(flags):
                    raise TinyRecError("a BertLayer must be trainable or frozen as a whole (run.py:101-112 policy)")
                out += ps
        for p in (self.mod.attn.att_fc1.weight, self.mod.attn.att_fc1.bias, self.mod.attn.att_fc2.weight,
                  self.mod.attn.att_fc2.bias, self.mod.dense.weight, self.mod.dense.bias):
            if p.requires_grad:
                out.append(p)
        return out

    def lowest_trainable_layer(self):
        for i, lr in enumerate(self.layers):
            if lr.q.weight.requires_grad:
                return i
        return len(self.layers)

    def save_from(self):
        """Lowest layer whose activations a training forward keeps: layer 0 when a bottom tensor trains (its gradient
        needs the backward down to the embedding output), else the lowest trainable layer."""
        return 0 if self.bottom_trainable() else self.lowest_trainable_layer()

    def check_supported(self):
        self.trainable_order()

    def _w(self, flat, p):
        """bf16 GEMM operand of a weight matrix."""
        if flat is not None and flat.has(p):
            return flat.w_shadow(p)
        return self.frozen.get(("w", id(p)), [p], lambda: p.detach().to(BF).contiguous())

    def layer_weights(self, flat, i):
        lr = self.layers[i]
        if flat is not None and flat.has(lr.q.weight):
            E = self.E
            o = flat.off(lr.q.weight)
            wqkv = flat.shadow[o:o + 3 * E * E].view(3 * E, E)
            ob = flat.off(lr.q.bias)
            bqkv = flat.data[ob:ob + 3 * E]
        else:
            wqkv = self.frozen.get(("wqkv", i), [lr.q.weight, lr.k.weight, lr.v.weight],
                                   lambda: torch.cat([lr.q.weight, lr.k.weight, lr.v.weight], 0).detach().to(BF).contiguous())
            bqkv = self.frozen.get(("bqkv", i), [lr.q.bias, lr.k.bias, lr.v.bias],
                                   lambda: torch.cat([lr.q.bias, lr.k.bias, lr.v.bias], 0).detach().float().contiguous())
        return wqkv, bqkv, self._w(flat, lr.o.weight), self._w(flat, lr.f1.weight), self._w(flat, lr.f2.weight)

    def diag_buckets(self, L, device):
        """int32 [2L-1]: bucket of key j for query i at index (j - i) + L - 1 (the gather index of relpos)."""
        def build():
            tab = rel_pos_bucket_table(L, self.rel_bins, self.max_rel)                                 # [i, j] -> bucket(j - i)
            return torch.cat([tab[1:, 0].flip(0), tab[0, :]]).to(device=device, dtype=torch.int32)    # d = -(L-1) .. L-1
        return self.frozen.get(("diag_buckets", L, str(device)), [], build)

    def relpos(self, L, flat=None):
        """fp32 [A, 2L-1] rel-pos bias vector, entry (j - i) + L - 1 (position_ids are arange(L), so the
        reference's [n, A, L, L] bias, modeling.py:458-463, is batch-invariant and Toeplitz).  A trainable table is
        re-gathered on the device by every call: the fused Adam rewrites it without moving ``_version``, and a replayed
        CUDA graph runs no Python, so no cached copy could follow it."""
        w = self.bert.rel_pos_bias.weight
        if flat is not None and flat.has(w):
            idx = self.frozen.get(("diag_index", L), [], lambda: self.diag_buckets(L, w.device).long())
            buf = self.frozen.get(("relpos_live", L), [], lambda: torch.empty(self.A, 2 * L - 1, device=w.device, dtype=F32))
            return torch.index_select(w.detach(), 1, idx, out=buf)
        return self.frozen.get(("relpos", L), [w],
                               lambda: w.detach().float()[:, self.diag_buckets(L, w.device).long()].contiguous())

    def word_table(self, flat=None):
        """bf16 word table of the forward: the flat buffer's bf16 shadow when it trains (the fused Adam refreshes it)."""
        w = self.bert.embeddings.word_embeddings.weight
        if flat is not None and flat.has(w):
            return flat.w_shadow(w)
        return self.frozen.get(("word",), [w], lambda: w.detach().to(BF).contiguous())

    # ---- workspaces -----------------------------------------------------------------
    def workspace(self, n, L, n_saved_layers, dev, tag=None):
        key = (n, L, n_saved_layers, tag)
        ws = self.ws.get(key)
        if ws is not None:
            return ws
        T, E, Fd = n * L, self.E, self.F
        mk = lambda *s, dt=BF: torch.empty(*s, device=dev, dtype=dt)  # noqa: E731
        ws = dict(x0=mk(T, E), xa=mk(T, E), xb=mk(T, E), qkv=mk(T, 3 * E), ctx=mk(T, E), pre=mk(T, E), x1=mk(T, E),
                  h=mk(T, Fd), e=mk(T, self.Q), a=mk(n, L, dt=F32), pooled=mk(n, E), saved=[])
        for _ in range(n_saved_layers):
            ws["saved"].append(dict(xin=None, qkv=mk(T, 3 * E), ctx=mk(T, E), pre1=mk(T, E), x1=mk(T, E),
                                    z=mk(T, Fd), h=mk(T, Fd), pre2=mk(T, E), xout=mk(T, E)))
        if n_saved_layers:
            ws.update(dx=mk(T, E), dx2=mk(T, E), dpre=mk(T, E), dpre_drop=mk(T, E), dz=mk(T, Fd), dqkv=mk(T, 3 * E), dctx=mk(T, E),
                      du=mk(T, self.Q), dnews_bf=mk(n, self.D), dpooled=mk(n, E, dt=F32))
        if len(self.ws) > 8:
            self.ws.clear()
        self.ws[key] = ws
        return ws

    # ---- forward ----------------------------------------------------------------------
    def forward(self, x, flat=None, save=False, out=None, drop=None, tag=None):
        """x int64 [n, 2L] -> news vectors fp32 [n, D].  With ``save`` the activations the
        backward needs are kept in the workspace (layers >= lowest trainable layer).  ``drop`` is a
        DropState (training mode, reference semantics) or None (eval)."""
        if x.dtype != torch.int64 or x.dim() != 2 or x.shape[1] % 2:
            raise TinyRecError(f"news encoder input must be int64 [n, 2L], got {x.dtype} {tuple(x.shape)}")
        x = x.contiguous()
        n, L = x.shape[0], x.shape[1] // 2
        dev = x.device
        nl = len(self.layers)
        low = self.save_from() if save else nl
        ws = self.workspace(n, L, nl - low if save else 0, dev, tag)      # tag: several saved passes per step
        emb = self.bert.embeddings
        relpos = self.relpos(L, flat)
        cur = ws["x0"]
        dmk = (lambda site, p: drop.make(site, p)) if drop is not None else (lambda site, p: None)
        ph, pa = (drop.p_hidden, drop.p_attn) if drop is not None else (0.0, 0.0)
        ops.embed_ln(x, L, self.word_table(flat), emb.position_embeddings.weight, emb.token_type_embeddings.weight[0],
                     emb.LayerNorm.weight, emb.LayerNorm.bias, self.ln_eps, cur, drop=dmk(SITE_EMB, ph))
        for i, lr in enumerate(self.layers):
            wqkv, bqkv, wo, w1, w2 = self.layer_weights(flat, i)
            if i >= low:
                sv = ws["saved"][i - low]
                sv["xin"] = cur
                qkv, ctx, pre1, x1, h, pre2, xout, z = sv["qkv"], sv["ctx"], sv["pre1"], sv["x1"], sv["h"], sv["pre2"], sv["xout"], sv["z"]
            else:
                qkv, ctx, pre1, x1, h, pre2, z = ws["qkv"], ws["ctx"], ws["pre"], ws["x1"], ws["h"], ws["pre"], None
                xout = ws["xb"] if cur is ws["xa"] else ws["xa"]
            ops.gemm(cur, wqkv, qkv, bias=bqkv)
            ops.attn_fwd(qkv, x, L, relpos, ctx, self.A, drop=dmk(drop_site(i, KIND_ATTN), pa))
            ops.gemm(ctx, wo, pre1, bias=lr.o.bias, residual=cur, drop=dmk(drop_site(i, KIND_ATT_OUT), ph))
            ops.layernorm_fwd(pre1, lr.ln1.weight, lr.ln1.bias, self.ln_eps, x1)
            # trained layers keep gelu'(z) (not z) for the backward: its dgrad epilogue is then a single multiply
            ops.gemm(x1, w1, h, bias=lr.f1.bias, act=ops.ACT_GELU_DAUX if z is not None else ops.ACT_GELU, aux=z)
            ops.gemm(h, w2, pre2, bias=lr.f2.bias, residual=x1, drop=dmk(drop_site(i, KIND_FFN_OUT), ph))
            ops.layernorm_fwd(pre2, lr.ln2.weight, lr.ln2.bias, self.ln_eps, xout)
            cur = xout
        at = self.mod.attn
        ops.gemm(cur, self._w(flat, at.att_fc1.weight), ws["e"], bias=at.att_fc1.bias, act=ops.ACT_TANH)
        ops.attnpool_fwd(cur, ws["e"], self.Q, at.att_fc2.weight.view(-1), at.att_fc2.bias, None, ws["pooled"], ws["a"], n, L)
        if out is None:
            out = torch.empty(n, self.D, device=dev, dtype=F32)
        ops.gemm(ws["pooled"], self._w(flat, self.mod.dense.weight), out, bias=self.mod.dense.bias)
        if save:
            ws["xlast"], ws["x"], ws["n"], ws["L"], ws["low"], ws["drop"] = cur, x, n, L, low, drop
            ws["relpos"] = relpos
        self.last_ws = ws
        return out

    # ---- fp32 inference forward (NewsEncoder precision='fp32') ------------------------------
    def _split_w(self, key, tensors, build_f32):
        """bf16 [hi | hi | lo] image [N, 3K] of an fp32 weight [N, K], split from the fp32 masters (never the bf16
        shadow) and cached until a source tensor changes, by torch or by the fused Adam (ops.param_generation)."""
        def build():
            w = build_f32().contiguous()
            return ops.split_bf16x3(w, torch.empty(w.shape[0], 3 * w.shape[1], device=w.device, dtype=BF), weight=True)
        return self.frozen.get(("split",) + key, tensors, build, gen=ops.param_generation)

    def layer_weights_fp32(self, i):
        lr = self.layers[i]
        qkv_w, qkv_b = [lr.q.weight, lr.k.weight, lr.v.weight], [lr.q.bias, lr.k.bias, lr.v.bias]
        wqkv = self._split_w(("wqkv", i), qkv_w, lambda: torch.cat([t.detach() for t in qkv_w], 0))
        bqkv = self.frozen.get(("bqkv_f32", i), qkv_b, lambda: torch.cat([t.detach() for t in qkv_b], 0).float().contiguous(),
                               gen=ops.param_generation)
        wo, w1, w2 = (self._split_w(("w", id(p)), [p], p.detach) for p in (lr.o.weight, lr.f1.weight, lr.f2.weight))
        return wqkv, bqkv, wo, w1, w2

    def workspace_fp32(self, n, L, dev):
        key = (n, L, "fp32")
        ws = self.ws.get(key)
        if ws is not None:
            return ws
        T, E = n * L, self.E
        mk = lambda *s: torch.empty(*s, device=dev, dtype=F32)  # noqa: E731
        ws = dict(xa=mk(T, E), xb=mk(T, E), x1=mk(T, E), pre=mk(T, E), qkv=mk(T, 3 * E), ctx=mk(T, E), h=mk(T, self.F),
                  u=mk(T, self.Q), pooled=mk(n, E),
                  # the split operand of every GEMM in turn (largest: the FFN2 input, [T, 3F])
                  split=torch.empty(T * 3 * max(E, self.F), device=dev, dtype=BF))
        if len(self.ws) > 8:
            self.ws.clear()
        self.ws[key] = ws
        return ws

    def forward_fp32(self, x, out=None):
        """x int64 [n, 2L] -> news vectors fp32 [n, D] with fp32 activations end to end (inference only: no dropout,
        nothing saved for a backward).  Every linear layer is one bf16 GEMM over K' = 3K split operands
        (include/tinyrec.h, tnr_split_bf16x3) with an fp32 output; about 1e-5 relative to a float64 reference."""
        if x.dtype != torch.int64 or x.dim() != 2 or x.shape[1] % 2:
            raise TinyRecError(f"news encoder input must be int64 [n, 2L], got {x.dtype} {tuple(x.shape)}")
        x = x.contiguous()
        n, L = x.shape[0], x.shape[1] // 2
        dev = x.device
        ws = self.workspace_fp32(n, L, dev)
        sp = ws["split"]

        def split(a, gelu=False):
            return ops.split_bf16x3(a, sp[:a.shape[0] * 3 * a.shape[1]].view(a.shape[0], 3 * a.shape[1]), gelu=gelu)

        emb = self.bert.embeddings
        relpos = self.relpos(L)
        cur = ws["xa"]
        ops.embed_ln_f32(x, L, emb.word_embeddings.weight.detach(), emb.position_embeddings.weight.detach(),
                         emb.token_type_embeddings.weight.detach()[0], emb.LayerNorm.weight.detach(),
                         emb.LayerNorm.bias.detach(), self.ln_eps, cur)
        for i, lr in enumerate(self.layers):
            wqkv, bqkv, wo, w1, w2 = self.layer_weights_fp32(i)
            ops.gemm(split(cur), wqkv, ws["qkv"], bias=bqkv)
            ops.attn_fwd_f32(ws["qkv"], x, L, relpos, ws["ctx"], self.A)
            ops.gemm(split(ws["ctx"]), wo, ws["pre"], bias=lr.o.bias.detach())
            ops.add_layernorm_f32(ws["pre"], cur, lr.ln1.weight.detach(), lr.ln1.bias.detach(), self.ln_eps, ws["x1"])
            ops.gemm(split(ws["x1"]), w1, ws["h"], bias=lr.f1.bias.detach())
            ops.gemm(split(ws["h"], gelu=True), w2, ws["pre"], bias=lr.f2.bias.detach())
            nxt = ws["xb"] if cur is ws["xa"] else ws["xa"]
            ops.add_layernorm_f32(ws["pre"], ws["x1"], lr.ln2.weight.detach(), lr.ln2.bias.detach(), self.ln_eps, nxt)
            cur = nxt
        at, dense = self.mod.attn, self.mod.dense
        w_fc1 = self._split_w(("w", id(at.att_fc1.weight)), [at.att_fc1.weight], at.att_fc1.weight.detach)
        ops.gemm(split(cur), w_fc1, ws["u"], bias=at.att_fc1.bias.detach())
        ops.attnpool_fwd_f32(cur, ws["u"], self.Q, at.att_fc2.weight.detach().view(-1), at.att_fc2.bias.detach(),
                             ws["pooled"], n, L)
        if out is None:
            out = torch.empty(n, self.D, device=dev, dtype=F32)
        w_dense = self._split_w(("w", id(dense.weight)), [dense.weight], dense.weight.detach)
        ops.gemm(split(ws["pooled"]), w_dense, out, bias=dense.bias.detach())
        return out

    # ---- backward -----------------------------------------------------------------------
    def _splitk(self, M, N, K):
        tiles = ((M + 127) // 128) * ((N + (255 if N > 128 else 127)) // (256 if N > 128 else 128))
        sms = 148
        s = max(1, int(round(2.0 * sms / tiles)))
        return max(1, min(s, (K + 63) // 64 // 4 or 1))

    def _wgrad(self, flat, p, dy, xin, rows=None):
        """dW[out,in] += dy[T,out]^T @ x[T,in]; db += colsum(dy)."""
        M = dy.shape[1]
        g = flat.g_view(p) if rows is None else flat.grad[flat.off(p):flat.off(p) + rows * p.shape[1]].view(rows, p.shape[1])
        ops.gemm(dy, xin, g, a_t=True, b_t=True, split_k=self._splitk(M, xin.shape[1], dy.shape[0]), accumulate=True)

    def backward(self, d_news, flat, on_layer_done=None, ws=None, on_grads_ready=None):
        """d_news fp32 [n, D] -> parameter gradients accumulated into ``flat.grad``.
        ``on_layer_done(i)`` is called after the last gradient kernel of encoder layer ``i`` was
        enqueued (bucketed gradient all-reduce overlapping the rest of the backward).
        ``on_grads_ready(first_param, last_param)``: finer notifications for the LOWEST trainable layer, whose
        gradient exchange has no later backward work to hide behind: the contiguous flat-buffer range
        [first_param .. last_param] is final.  With it the layer's weight gradients are issued so that the smallest
        range (attention.output: 2.4 MB) is the one that finishes last."""
        ws = self.last_ws if ws is None else ws      # ws: the workspace of the forward pass this backward belongs to
        n, L, low, x = ws["n"], ws["L"], ws["low"], ws["x"]
        drop = ws.get("drop")
        dmk = (lambda site, p: drop.make(site, p)) if drop is not None else (lambda site, p: None)
        ph, pa = (drop.p_hidden, drop.p_attn) if drop is not None else (0.0, 0.0)
        T, E = n * L, self.E
        nl = len(self.layers)
        at, dense = self.mod.attn, self.mod.dense
        if self.scratch_ln is None or self.scratch_ln.device != d_news.device:
            self.scratch_ln = torch.zeros(2 * E, device=d_news.device, dtype=F32)
        ops.cast_f32_bf16(d_news, ws["dnews_bf"])
        dnb = ws["dnews_bf"]
        if flat.has(dense.weight):
            self._wgrad(flat, dense.weight, dnb, ws["pooled"])
            ops.colsum(dnb, flat.g_view(dense.bias))
        ops.gemm(dnb, self._w(flat, dense.weight), ws["dpooled"], b_t=True)
        xl = ws["xlast"]
        if flat.has(at.att_fc1.weight):
            dw2, db2 = flat.g_view(at.att_fc2.weight).view(-1), flat.g_view(at.att_fc2.bias)
        else:
            dw2, db2 = self.scratch_ln[:self.Q], self.scratch_ln[E:E + 1]
        ops.attnpool_bwd(xl, ws["e"], self.Q, at.att_fc2.weight.view(-1), ws["a"], ws["dpooled"], ws["dx2"], ws["du"],
                         dw2, db2, n, L)
        if flat.has(at.att_fc1.weight):
            self._wgrad(flat, at.att_fc1.weight, ws["du"], xl)
            ops.colsum(ws["du"], flat.g_view(at.att_fc1.bias))
        if low >= nl:
            return
        emb = self.bert.embeddings
        rel_w = self.bert.rel_pos_bias.weight
        bottom = any(flat.has(p) for p in self.bottom_params())
        emb_train = any(flat.has(p) for p in self.bottom_params()[:5])
        # with a trainable bottom block the backward goes on below the lowest trainable layer, so that layer's exchange
        # has later work to hide behind: it is reported whole (on_layer_done), like every other layer
        lowest = self.lowest_trainable_layer() if not bottom and on_grads_ready is not None else -1
        relpos = ws.get("relpos")
        if relpos is None:
            relpos = self.relpos(L, flat)
        dx = ws["dx"]
        ops.gemm(ws["du"], self._w(flat, at.att_fc1.weight), dx, b_t=True, residual=ws["dx2"])
        for i in range(nl - 1, low - 1, -1):
            lr, sv = self.layers[i], ws["saved"][i - low]
            train = flat.has(lr.q.weight)
            fine = train and i == lowest
            wqkv, bqkv, wo, w1, w2 = self.layer_weights(flat, i)
            dpre, dz, dqkv, dctx, dx2 = ws["dpre"], ws["dz"], ws["dqkv"], ws["dctx"], ws["dx2"]
            sg, sb = (flat.g_view(lr.ln2.weight), flat.g_view(lr.ln2.bias)) if train else (self.scratch_ln[:E], self.scratch_ln[E:])
            # dpre = grad at (dropout(dense) + residual); dd = grad at the dense output (mask re-applied)
            d2 = dmk(drop_site(i, KIND_FFN_OUT), ph)
            dd = ws["dpre_drop"] if d2 is not None else dpre
            ops.layernorm_bwd(dx, sv["pre2"], lr.ln2.weight, self.ln_eps, dpre, sg, sb,
                              dx_drop=dd if d2 is not None else None, drop=d2,
                              dsum=flat.g_view(lr.f2.bias) if train else None)       # + f2.bias gradient
            if train:
                self._wgrad(flat, lr.f2.weight, dd, sv["h"])
                if fine:
                    on_grads_ready(lr.f2.weight, lr.ln2.bias)
            # dz = (dd @ W2) * gelu'(z); its column sums (the intermediate.dense bias gradient) come out of the
            # same epilogue
            ops.gemm(dd, w2, dz, b_t=True, act=ops.ACT_MULAUX, aux=sv["z"],
                     colsum=flat.g_view(lr.f1.bias) if train else None)
            if train:
                self._wgrad(flat, lr.f1.weight, dz, sv["x1"])
                if fine:
                    on_grads_ready(lr.f1.weight, lr.f1.bias)
            ops.gemm(dz, w1, dx2, b_t=True, residual=dpre)                 # d x1
            sg, sb = (flat.g_view(lr.ln1.weight), flat.g_view(lr.ln1.bias)) if train else (self.scratch_ln[:E], self.scratch_ln[E:])
            d1 = dmk(drop_site(i, KIND_ATT_OUT), ph)
            dd = ws["dpre_drop"] if d1 is not None else dpre
            ops.layernorm_bwd(dx2, sv["pre1"], lr.ln1.weight, self.ln_eps, dpre, sg, sb,
                              dx_drop=dd if d1 is not None else None, drop=d1,
                              dsum=flat.g_view(lr.o.bias) if train else None)        # + attention.output.dense.bias gradient
            if train and not fine:
                self._wgrad(flat, lr.o.weight, dd, sv["ctx"])
            ops.gemm(dd, wo, dctx, b_t=True)
            dbq = None
            if train:
                ob = flat.off(lr.q.bias)
                dbq = flat.grad[ob:ob + 3 * E]                             # [bq | bk | bv] gradient, fused
            if flat.has(rel_w):          # the table is shared by every layer: each one adds its dS sums
                ops.attn_bwd_drel(sv["qkv"], x, L, relpos, dctx, dqkv, self.A, self.diag_buckets(L, x.device),
                                  flat.g_view(rel_w), drop=dmk(drop_site(i, KIND_ATTN), pa), dbias=dbq)
            else:
                ops.attn_bwd(sv["qkv"], x, L, relpos, dctx, dqkv, self.A, drop=dmk(drop_site(i, KIND_ATTN), pa),
                             dbias=dbq)
            if train:
                self._wgrad(flat, lr.q.weight, dqkv, sv["xin"], rows=3 * E)
            if fine:
                # lowest trainable layer: the QKV range (7 MB) goes out now; the attention.output weight gradient was
                # held back (dd / ctx stay valid: no layer below overwrites them) so that the last exchange of the
                # step is the smallest range
                on_grads_ready(lr.q.weight, lr.v.bias)
                self._wgrad(flat, lr.o.weight, dd, sv["ctx"])
                on_grads_ready(lr.o.weight, lr.ln1.bias)
            if i > low or emb_train:
                ops.gemm(dqkv, wqkv, dx, b_t=True, residual=dpre)
            if on_layer_done is not None and train:
                on_layer_done(i)
        if emb_train:
            # dx: gradient at the embedding output; only the trainable tensors get a buffer
            g = lambda p: flat.g_view(p) if flat.has(p) else None  # noqa: E731
            ops.embed_ln_bwd(x, L, self.word_table(flat), emb.position_embeddings.weight, emb.token_type_embeddings.weight[0],
                             emb.LayerNorm.weight, self.ln_eps, dx, dword=g(emb.word_embeddings.weight),
                             dpos=g(emb.position_embeddings.weight),
                             dtype0=flat.g_view(emb.token_type_embeddings.weight)[0] if flat.has(emb.token_type_embeddings.weight) else None,
                             dgamma=g(emb.LayerNorm.weight), dbeta=g(emb.LayerNorm.bias), drop=dmk(SITE_EMB, ph))
