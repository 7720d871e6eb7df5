"""Drop-in replacement of the reference's ``model/mem_transformer.py`` on the libtgan_b200 kernels.

Same module tree, parameter names / shapes (the checkpoint contract, SURVEY.md section 5) and public methods as
the reference -- ``MemTransformerLM(cfg, n_token, vec_len)`` with ``forward(data, target, reset_mems, mems)``
(mem_transformer.py:653), ``forward_generate`` (:578), ``forward_generate_gumbel`` (:602), ``reset_length``
(:432), ``init_mems`` (:436) -- but the sub-modules are parameter containers only: all arithmetic of ``_forward``
(:484-576) and its backward runs in the CUDA library through ``tgan_b200.engine.TxlEngine``.  There is no eager /
CPU fallback: calling the model on a CPU tensor raises.
"""
import contextlib
import heapq
import os
import weakref
from dataclasses import dataclass
from typing import Dict, List, NamedTuple, Optional, Tuple

import torch
import torch.nn as nn

from utils.proj_adaptive_softmax import ProjectedAdaptiveLogSoftmax
from tgan_b200 import lib as L
from tgan_b200.engine import RingMems, TxlDims, TxlEngine


class PositionalEmbedding(nn.Module):
    """mem_transformer.py:7-23 (the sinusoid itself is produced by tgan_pos_emb)."""

    def __init__(self, demb):
        super().__init__()
        self.demb = demb
        inv_freq = 1 / (10000 ** (torch.arange(0.0, demb, 2.0) / demb))
        self.register_buffer("inv_freq", inv_freq)


class PositionwiseFF(nn.Module):
    """mem_transformer.py:26-60: parameters of the position-wise FFN + its LayerNorm."""

    def __init__(self, d_model, d_inner, dropout, pre_lnorm=False):
        super().__init__()
        self.d_model, self.d_inner, self.dropout = d_model, d_inner, dropout
        self.CoreNet = nn.Sequential(nn.Linear(d_model, d_inner), nn.ReLU(inplace=True), nn.Dropout(dropout),
                                     nn.Linear(d_inner, d_model), nn.Dropout(dropout))
        self.layer_norm = nn.LayerNorm(d_model)
        self.pre_lnorm = pre_lnorm


class RelMultiHeadAttn(nn.Module):
    """mem_transformer.py:63-160: parameters of the relative multi-head attention."""

    def __init__(self, n_head, d_model, d_head, dropout, dropatt=0, tgt_len=None, mem_len=None, pre_lnorm=False):
        super().__init__()
        self.n_head, self.d_model, self.d_head, self.dropout = n_head, d_model, d_head, dropout
        self.qkv_net = nn.Linear(d_model, 3 * n_head * d_head, bias=False)
        self.drop = nn.Dropout(dropout)
        self.dropatt = nn.Dropout(dropatt)
        self.o_net = nn.Linear(n_head * d_head, d_model, bias=False)
        self.layer_norm = nn.LayerNorm(d_model)
        self.scale = 1 / (d_head ** 0.5)
        self.pre_lnorm = pre_lnorm


class RelPartialLearnableMultiHeadAttn(RelMultiHeadAttn):
    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.r_net = nn.Linear(self.d_model, self.n_head * self.d_head, bias=False)


class RelPartialLearnableDecoderLayer(nn.Module):
    def __init__(self, n_head, d_model, d_head, d_inner, dropout, **kwargs):
        super().__init__()
        self.dec_attn = RelPartialLearnableMultiHeadAttn(n_head, d_model, d_head, dropout, **kwargs)
        self.pos_ff = PositionwiseFF(d_model, d_inner, dropout, pre_lnorm=kwargs.get("pre_lnorm"))


class AdaptiveEmbedding(nn.Module):
    """mem_transformer.py:284-341 (div_val 1, cutoffs []): owns ``emb_layers.0.weight``."""

    def __init__(self, n_token, d_embed, d_proj, vec_len, append_note_status):
        super().__init__()
        if append_note_status:
            raise NotImplementedError("append_note_status is off in every shipped config and not accelerated")
        if d_proj != d_embed:
            raise NotImplementedError("d_proj != d_embed is not part of the accelerated path")
        self.n_token, self.d_embed, self.d_proj = n_token, d_embed, d_proj
        self.append_note_status = append_note_status
        self.cutoffs = [n_token]
        self.emb_scale = d_proj ** 0.5
        self.emb_layers = nn.ModuleList([nn.Embedding(n_token, d_embed, sparse=False)])
        self.emb_projs = nn.ParameterList()


def _param_dict(model):
    """name -> Parameter (the module tree walk costs ~0.3 ms, a decode step asks three times: cached; the Parameter
    objects survive .to() / load_state_dict / flat-buffer re-pointing, and Module._apply drops the cache anyway)"""
    sd = model.__dict__.get("_param_cache")
    if sd is None:
        sd = dict(model.named_parameters())
        sd.setdefault("crit.out_layers.0.weight", model.crit.out_layers[0].weight)
        model.__dict__["_param_cache"] = sd
    return sd


class _TxlFunction(torch.autograd.Function):
    """One autograd node for the whole generator stack (embedding .. NLL or Gumbel-ST output)."""

    @staticmethod
    def forward(ctx, model, mode, inp, target, reset, mems, temperature, noise, names, grad_enabled, *params):
        eng = model._get_engine()
        # grad mode is off inside Function.forward, and needs_input_grad does not see a caller's no_grad(): that comes
        # in as grad_enabled (a call under no_grad() records no graph, so nothing would ever read saved activations)
        need_grad = grad_enabled and any(ctx.needs_input_grad)
        ectx = eng.forward(inp.detach(), reset, mems, mem_len=model.mem_len, same_length=model.same_length,
                           training=model.training, target=target if mode == "mle" else None,
                           n_pred=target.size(0) if mode == "mle" else None, save_for_backward=need_grad)
        model._new_mems = ectx.new_mems
        ctx.ectx, ctx.model, ctx.mode, ctx.names = ectx, model, mode, names
        ctx.params = params
        ctx.soft_in = inp.is_floating_point()
        T, B, V = ectx.T, ectx.B, model.n_token
        if mode == "mle":
            return ectx.nll.view(T, B)
        logits = torch.empty(T * B, V, dtype=torch.float32, device=eng.device)
        if mode == "logits":
            L.convert(ectx.logits, ectx.logits.stride(0), logits, V, T * B, V, V)
            return logits.view(T, B, V)
        # gumbel straight-through (mem_transformer.py:609-628)
        y = torch.empty(T * B, V, dtype=torch.float32, device=eng.device)
        U = None if noise is None else noise.reshape(T * B, V).to(device=eng.device, dtype=torch.float32).contiguous()
        eng.calls += 1
        tau = temperature if isinstance(temperature, torch.Tensor) else float(temperature)  # tensor: read on the device
        L.gumbel_st_fwd(ectx.logits, U, tau, y, logits, None, T * B, V, seed=eng.seed, site=eng._site(eng.calls, 3))
        ctx.y, ctx.tau = y, tau
        return logits.view(T, B, V)

    @staticmethod
    def backward(ctx, gout):
        ectx, model, mode = ctx.ectx, ctx.model, ctx.mode
        eng = model._get_engine()
        if ectx.layers is None or len(ectx.layers) == 0:
            raise RuntimeError("backward through a generator call that did not save activations")
        T, B, V = ectx.T, ectx.B, model.n_token
        gout = gout.contiguous().float()
        # Parameter gradients are ACCUMULATED straight into ``p.grad`` by one unpack kernel (what autograd's
        # AccumulateGrad nodes would do with 72 separate adds); the Function therefore returns None for them.
        targets = {}
        for n, prm in zip(ctx.names, ctx.params):
            if prm.grad is None:
                prm.grad = torch.zeros_like(prm, memory_format=torch.contiguous_format)
            targets[n] = prm.grad
        if mode == "mle":
            grads = eng.backward(ectx, dnll=gout, need_dinput=ctx.soft_in, grad_targets=targets,
                                 reducer=model.grad_reducer)
        else:
            g = gout.view(T * B, V)
            if mode == "gumbel":
                dl = torch.empty_like(g)
                L.gumbel_st_bwd(ctx.y, g, ctx.tau, dl, T * B, V)
                g = dl
            grads = eng.backward(ectx, dlogits32=g, need_dinput=ctx.soft_in, grad_targets=targets)
        dinp = None
        if ctx.soft_in:
            d = grads["__dinput__"]
            dinp = torch.empty(ectx.Q * B, V, dtype=torch.float32, device=eng.device)
            L.convert(d, d.stride(0), dinp, V, ectx.Q * B, V, V)
            dinp = dinp.view(ectx.Q, B, V)
        return (None, None, dinp, None, None, None, None, None, None, None) + (None,) * len(ctx.names)


class _GraphEntry:
    """One captured MLE segment: forward graph, backward graph, their static inputs and outputs."""
    fwd = bwd = ectx = None
    n_fwd = n_bwd = 0
    staged = None


class _TxlGraphFunction(torch.autograd.Function):
    """MLE forward / backward as two CUDA-graph replays (``MemTransformerLM.use_cuda_graphs``).

    A training segment is ~180 kernel launches of fixed shape; at small per-GPU batches (data parallel at 4-8 GPUs) the
    host cannot enqueue them as fast as the GPU retires them.  The engine calls for one (ring phase, shape) key are
    captured once and replayed; inputs are copied into static buffers, parameter gradients are accumulated into the
    ``.grad`` tensors that existed at capture (re-captured if they move), and the dropout masks advance through the
    device step counter (tgan_set_step_counter) that the forward graph bumps as its first node."""

    @staticmethod
    def forward(ctx, model, entry, names, *params):
        entry.fwd.replay()
        model._get_engine().pack_epoch += 1  # the graph re-packed the parameters: cached K/V projections are stale
        L.note_graph_replay(entry.n_fwd)
        ctx.model, ctx.entry, ctx.names, ctx.params = model, entry, names, params
        e = entry.ectx
        return e.nll.view(e.T, e.B).clone()

    @staticmethod
    def backward(ctx, gout):
        model, entry = ctx.model, ctx.entry
        eng = model._get_engine()
        entry.dnll.copy_(gout.reshape(-1))
        if entry.bwd is None:
            # The graph writes the step's parameter gradients into engine-owned staging tensors (reference layout), so
            # it never depends on where the caller keeps .grad (zero_grad(set_to_none=True) moves it every step).
            if model._grad_staging is None:  # shared by every captured segment of this model (replayed one at a time)
                model._grad_staging = {n: torch.empty_like(prm, memory_format=torch.contiguous_format)
                                       for n, prm in zip(ctx.names, ctx.params)}
            entry.staged = model._grad_staging
            # descriptor table staged outside the capture; the entry keeps it alive for the graph's lifetime
            entry.staged_desc = eng._unpack_desc_for(entry.staged)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            n0 = L.launch_count()
            with torch.cuda.graph(g, pool=eng.graph_pool()):
                eng.backward(entry.ectx, dnll=entry.dnll, grad_targets=entry.staged, accumulate=False,
                             reducer=model.grad_reducer)
            entry.bwd, entry.n_bwd = g, L.launch_count() - n0
            # eng.backward dropped the activations: their pool blocks may now be reused by the next key's capture
            # (graphs that share the pool are replayed strictly one after the other).  The entry must not keep the
            # ring alive either: its lifetime is the caller's `mems` handle (see _drop_ring_graphs)
            entry.ectx.ring = entry.ectx.new_mems = entry.ectx.hid_t = None
        entry.bwd.replay()
        L.note_graph_replay(entry.n_bwd)
        grads, staged = [], []
        for n, prm in zip(ctx.names, ctx.params):
            if prm.grad is None:
                prm.grad = torch.zeros_like(prm, memory_format=torch.contiguous_format)
            grads.append(prm.grad)
            staged.append(entry.staged[n])
        torch._foreach_add_(grads, staged)  # one multi-tensor kernel: .grad += this segment's gradients
        model._graph_pending = None
        return (None, None, None) + (None,) * len(ctx.names)


# ---- generation from a request queue: host schedule --------------------------------------------------------
_TECHNIQUES = {"random": 0, "topk": 1, "nucleus": 2}


@dataclass
class GenRequest:
    """One prime to continue with ``MemTransformerLM.generate_requests``; the settings mirror ``generate_batched``'s
    keywords.  prompt: int64 [T], T >= 1 (the conditioning tokens); gen_len >= 1 tokens are generated."""
    prompt: torch.Tensor
    gen_len: int
    technique: str = "topk"
    topk: int = 32
    top_p: float = 0.0
    temperature: float = 0.95
    exclude_bos: bool = True
    empty_token: int = -1
    num_empty_tokens_to_ignore: int = 0


class PrefillPlan(NamedTuple):
    """The context passes of ``request_schedule(..., context_pass=True)``.  Requests are prefilled in groups of up to
    ``batch_size`` consecutive requests (list order); group g's pass runs over ``blocks[g]`` (int64 [max(T_r - 1), G]:
    column j holds prompt[:-1] of the group's j-th request, left-padded by ``pads[g][j]`` rows of token 0; None when
    every prompt of the group is one token) and is enqueued at step ``steps[g]``, the start step of the group's first
    request (None: no pass).  ``desc`` int32 [n, 4] lists, in request order, one (source column, first source position,
    destination column, rows) copy per request with n_r = min(T_r - 1, mem_len) > 0 rows: the last n_r rows of its
    pass.  ``slices[t]`` = [(group, first descriptor, count, max rows)] to apply at step t, in group order.
    ``run0`` int32 [R]: the run of empty_token at the end of prompt[:-1].  ``lead`` = P0 = min(mem_len,
    max_r(T_r - 1)): the queue ring's leading rows."""
    lead: int
    blocks: List[Optional[torch.Tensor]]
    pads: List[torch.Tensor]
    steps: List[Optional[int]]
    desc: torch.Tensor
    slices: Dict[int, List[Tuple[int, int, int, int]]]
    run0: torch.Tensor


class RequestSchedule(NamedTuple):
    """The step-by-column plan of ``generate_requests``.  ``tables`` int32 [4, S, B] holds, per step t and column b:
    forced   -- the input token of the step, or -1 for "the column's sample of step t - 1";
    req      -- the request served, or -1 for an idle column;
    out_off  -- where the step's sample goes in the flat output, or -1 when it is not kept;
    key_start -- the step at which the column's current request started (an idle column: t itself).
    The row written at step t has absolute position t, so key_start is also the request's key floor.
    ``out_base[r]``: offset of request r's first generated token in the flat output.
    With a context pass (``prefill`` is not None) the tables are [5, S, B]: the row written at step t has absolute
    position P0 + t, key_start is the key floor P0 + t0 - n_r of a request that starts at step t0 on its n_r prefilled
    rows (an idle column: P0 + t), and the fifth row, ``start``, is the step at which the column's request started."""
    tables: torch.Tensor
    out_base: List[int]
    prefill: Optional[PrefillPlan] = None

    @property
    def forced(self):
        return self.tables[0]

    @property
    def req(self):
        return self.tables[1]

    @property
    def out_off(self):
        return self.tables[2]

    @property
    def key_start(self):
        return self.tables[3]

    @property
    def start(self):
        return self.tables[4] if self.prefill is not None else self.tables[3]


def _trailing_run(seq, token):
    n = 0
    for x in reversed(seq):
        if x != token:
            break
        n += 1
    return n


def request_schedule(prompts, gen_lens, batch_size, *, context_pass=False, mem_len=None,
                     empty_tokens=None) -> RequestSchedule:
    """Plan ``len(prompts)`` requests on min(batch_size, len(prompts)) columns.  Request r occupies one column for
    T_r + gen_len_r - 1 consecutive steps: it feeds its T_r prompt tokens one per step, the step that feeds the last
    one samples its first token, and each later step feeds the previous sample.  Requests go in list order to the
    column that frees first, ties to the lowest column.  Idle columns (the tail of the queue) are fed token 0 and floored
    at their own row: they produce nothing.  prompts: 1-D int sequences (CPU); gen_lens: ints >= 1.

    context_pass=True: prompt[:-1] is consumed by context passes (``prefill``, see PrefillPlan) instead, so request r
    occupies its column for gen_len_r steps only; its first step feeds prompt[-1] on its n_r = min(T_r - 1, mem_len)
    prefilled rows.  Needs ``mem_len`` > 0; ``empty_tokens`` (one per request, default -1) sets ``run0``."""
    if context_pass and not (mem_len or 0) > 0:
        raise ValueError("a context pass needs mem_len > 0")
    B = min(batch_size, len(prompts))
    R = len(prompts)
    occupy = [g if context_pass else len(p) + g - 1 for p, g in zip(prompts, gen_lens)]
    free = [(0, c) for c in range(B)]  # (step at which the column frees, column): a heap
    place = []
    for n in occupy:
        t0, c = heapq.heappop(free)
        place.append((t0, c))
        heapq.heappush(free, (t0 + n, c))
    S = max(t for t, _ in free)
    tables = torch.empty(5 if context_pass else 4, S, B, dtype=torch.int32)
    forced, req, out_off, key_start = tables[:4]
    steps = torch.arange(S, dtype=torch.int32).view(S, 1).expand(S, B)
    forced.zero_()
    req.fill_(-1)
    out_off.fill_(-1)
    lead = min(mem_len, max(len(p) for p in prompts) - 1) if context_pass else 0
    key_start.copy_(steps + lead)
    if context_pass:
        tables[4].copy_(steps)
    out_base, base = [], 0
    for r, ((t0, c), prompt, g, n) in enumerate(zip(place, prompts, gen_lens, occupy)):
        T = len(prompt)
        req[t0:t0 + n, c] = r
        if context_pass:
            forced[t0, c] = int(prompt[-1])
            forced[t0 + 1:t0 + n, c] = -1
            out_off[t0:t0 + n, c] = torch.arange(base, base + g, dtype=torch.int32)
            key_start[t0:t0 + n, c] = lead + t0 - min(T - 1, mem_len)
            tables[4, t0:t0 + n, c] = t0
        else:
            forced[t0:t0 + T, c] = torch.as_tensor(prompt, dtype=torch.int32)
            forced[t0 + T:t0 + n, c] = -1
            out_off[t0 + T - 1:t0 + n, c] = torch.arange(base, base + g, dtype=torch.int32)
            key_start[t0:t0 + n, c] = t0
        out_base.append(base)
        base += g
    if not context_pass:
        return RequestSchedule(tables, out_base)
    blocks, pads, pass_steps, desc, slices = [], [], [], [], {}
    for gi, g0 in enumerate(range(0, R, B)):
        members = range(g0, min(g0 + B, R))
        Tm = max(len(prompts[r]) - 1 for r in members)
        pad = torch.tensor([Tm - (len(prompts[r]) - 1) for r in members], dtype=torch.int32)
        block = None
        if Tm > 0:
            block = torch.zeros(Tm, len(members), dtype=torch.int64)
            for j, r in enumerate(members):
                block[int(pad[j]):, j] = torch.as_tensor(prompts[r][:-1], dtype=torch.int64)
        blocks.append(block)
        pads.append(pad)
        pass_steps.append(place[g0][0] if Tm > 0 else None)
        for j, r in enumerate(members):
            n_r = min(len(prompts[r]) - 1, mem_len)
            if n_r == 0:
                continue
            t0, c = place[r]
            sl = slices.setdefault(t0, [])
            if sl and sl[-1][0] == gi:  # descriptors of one (group, step) are consecutive: request order
                _, lo, cnt, mx = sl[-1]
                sl[-1] = (gi, lo, cnt + 1, max(mx, n_r))
            else:
                sl.append((gi, len(desc), 1, n_r))
            desc.append([j, Tm - n_r, c, n_r])
    empty_tokens = [-1] * R if empty_tokens is None else list(empty_tokens)
    run0 = torch.tensor([_trailing_run(list(p)[:-1], e) for p, e in zip(prompts, empty_tokens)], dtype=torch.int32)
    plan = PrefillPlan(lead, blocks, pads, pass_steps, torch.tensor(desc, dtype=torch.int32).view(-1, 4), slices, run0)
    return RequestSchedule(tables, out_base, plan)


class MemTransformerLM(nn.Module):
    def __init__(self, cfg, n_token, vec_len):
        n_layer, n_head, d_model = cfg.MODEL.num_layers, cfg.MODEL.num_heads, cfg.MODEL.units
        d_head = d_model // n_head
        d_inner, dropout, dropatt = cfg.MODEL.inner_size, cfg.MODEL.dropout, cfg.MODEL.attention_dropout
        pre_lnorm = cfg.MODEL.pre_lnorm
        super().__init__()
        if pre_lnorm:
            raise NotImplementedError("pre_lnorm=True is off in every shipped config and not accelerated yet")
        self.cfg = cfg
        self.n_token = n_token
        self.d_embed = self.d_model = d_model
        self.n_head, self.d_head = n_head, d_head
        self.pad_type = cfg.TRAIN.pad_type
        self.replace_start_with_pad = cfg.TRAIN.replace_start_with_pad
        self.word_emb = AdaptiveEmbedding(n_token, d_model, d_model, vec_len, cfg.TRAIN.append_note_status)
        self.drop = nn.Dropout(dropout)
        self.n_layer = n_layer
        self.tgt_len, self.mem_len = cfg.TRAIN.tgt_length, cfg.TRAIN.mem_length
        self.max_klen = self.tgt_len + self.mem_len
        self.layers = nn.ModuleList([
            RelPartialLearnableDecoderLayer(n_head, d_model, d_head, d_inner, dropout, tgt_len=self.tgt_len,
                                            mem_len=self.mem_len, dropatt=dropatt, pre_lnorm=pre_lnorm)
            for _ in range(n_layer)])
        self.crit = ProjectedAdaptiveLogSoftmax(n_token, d_model, d_model)
        if cfg.MODEL.tie_embedding:
            self.crit.out_layers[0].weight = self.word_emb.emb_layers[0].weight
        else:
            raise NotImplementedError("tie_embedding=False is not part of the accelerated path")
        self.same_length = cfg.MODEL.same_length
        self.clamp_len = cfg.MODEL.clamp_len
        self.detach_mems_grad = True  # kept for the GAN loop; memory is always detached (mem_transformer.py:461-475)
        self.pos_emb = PositionalEmbedding(d_model)
        self.r_w_bias = nn.Parameter(torch.Tensor(n_head, d_head))
        self.r_r_bias = nn.Parameter(torch.Tensor(n_head, d_head))
        # fp32 mode (TGAN_B200_DTYPE=fp32) reproduces the reference's fp32 arithmetic to 1e-4; bf16 is the default
        self.compute_dtype = torch.float32 if os.environ.get("TGAN_B200_DTYPE", "bf16") == "fp32" else torch.bfloat16
        self.kernel_impl = L.IMPL_AUTO
        self._engine = None
        self._new_mems = None
        # replay each steady-state MLE segment (forward, backward) as CUDA graphs instead of ~180 launches; see
        # _TxlGraphFunction.  Off by default: it pins the input / gradient buffers of the captured shapes.
        self.use_cuda_graphs = False
        # data parallel: tgan_b200.dp.BucketReducer that all-reduces the MLE gradients bucket by bucket inside backward
        # (None: single process, or the caller reduces the flat gradient itself)
        self.grad_reducer = None
        self._graphs = {}
        self._graph_rings = {}
        self._graph_pending = None
        self._grad_staging = None

    def _apply(self, fn, *args, **kwargs):
        self.__dict__.pop("_param_cache", None)
        return super()._apply(fn, *args, **kwargs)

    # ---- reference API ---------------------------------------------------------------------------------
    def reset_length(self, tgt_len, mem_len):
        self.tgt_len, self.mem_len = tgt_len, mem_len

    def init_mems(self, n_layers):
        if self.mem_len > 0:
            param = next(self.parameters())
            return torch.empty(n_layers + 1, 0, dtype=param.dtype, device=param.device)
        return None

    def _get_engine(self) -> TxlEngine:
        dev = self.r_w_bias.device
        if dev.type != "cuda":
            raise RuntimeError("tgan_b200 MemTransformerLM runs on CUDA only (no CPU fallback): move the model to a GPU")
        drop, dropatt = self.drop.p, self.layers[0].dec_attn.dropatt.p
        e = self._engine
        if e is None or e.device != dev or e.dtype != self.compute_dtype or e.impl != self.kernel_impl:
            dims = TxlDims(self.n_layer, self.n_head, self.d_model, self.layers[0].pos_ff.d_inner, self.n_token,
                           drop, dropatt, self.clamp_len)
            e = TxlEngine(dims, dev, self.compute_dtype, seed=torch.initial_seed() & 0x7FFFFFFFFFFFFFFF,
                          impl=self.kernel_impl)
            self._engine = e
        e.d.dropout, e.d.dropatt, e.d.clamp_len = drop, dropatt, self.clamp_len
        e.bind_params(_param_dict(self))
        return e

    @contextlib.contextmanager
    def grad_window(self):
        """``with model.grad_window(): loss.backward()`` -- every backward call through the generator inside the block
        accumulates in the engine's padded gradient buffers; ``.grad`` is updated once when the block ends (see
        TxlEngine.begin_grad_window).  TransformerGAN wraps the backward of a sampled chunk (64 single-token calls)."""
        eng = self._get_engine()
        eng.begin_grad_window()
        try:
            yield
        finally:
            targets = {}
            pd = _param_dict(self)
            for n, *_ in eng.layout.reference_map():
                prm = pd[n]
                if prm.grad is None:
                    prm.grad = torch.zeros_like(prm, memory_format=torch.contiguous_format)
                targets[n] = prm.grad
            eng.end_grad_window(targets)

    def _graph_entry(self, eng, data, target, reset_mems, ring):
        """The captured forward for this (ring phase, shape) key; captured on first use."""
        B, Q, T = data.shape[1], data.shape[0], target.shape[0]
        # Keyed by the identity of the ring's storage object; a finalizer drops every entry of a ring when the ring
        # dies (each epoch's `mems=None` makes a new one), so a recycled address can never match a stale graph and old
        # entries do not pin their activations / pool blocks forever.
        rid = id(ring.slabs)
        key = (rid, ring.start, ring.length, Q, B, T, self.mem_len, self.same_length, self.training,
               eng.d.dropout, eng.d.dropatt, eng._param_key)
        entry = self._graphs.get(key)
        if entry is None:
            if rid not in self._graph_rings:
                self._graph_rings[rid] = weakref.finalize(ring.slabs, MemTransformerLM._drop_ring_graphs,
                                                          weakref.ref(self), rid)
            entry = _GraphEntry()
            entry.ids, entry.tgt = data.clone(), target.clone()
            entry.reset = torch.zeros(B, dtype=torch.uint8, device=data.device)
            entry.dnll = torch.zeros(T * B, dtype=torch.float32, device=data.device)
            ctr = L.step_counter(data.device)
            eng.invalidate()  # the parameter re-pack must be part of the graph
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            n0 = L.launch_count()
            with torch.cuda.graph(g, pool=eng.graph_pool()):
                ctr.add_(1)
                entry.ectx = eng.forward(entry.ids, entry.reset, ring, mem_len=self.mem_len, same_length=self.same_length,
                                         training=self.training, target=entry.tgt, n_pred=T, save_for_backward=True)
            eng.invalidate()
            entry.fwd, entry.n_fwd = g, L.launch_count() - n0
            nm = entry.ectx.new_mems
            entry.new_mems = None if nm is None else (nm.start, nm.length)
            self._graphs[key] = entry
        entry.ids.copy_(data)
        entry.tgt.copy_(target)
        if reset_mems is None:
            entry.reset.zero_()
        else:
            entry.reset.copy_(reset_mems)
        return entry

    @staticmethod
    def _drop_ring_graphs(self_ref, rid):
        self = self_ref()
        if self is None:
            return
        self._graph_rings.pop(rid, None)
        for k in [k for k in self._graphs if k[0] == rid]:
            del self._graphs[k]

    def _run(self, mode, data, target, reset_mems, mems, temperature=None, noise=None):
        eng = self._get_engine()
        if self.pad_type != "model":
            reset_mems = None  # the reset mask exists only for pad_type == 'model' (mem_transformer.py:495-528)
        names = [r for r, *_ in eng.layout.reference_map()]
        pd = _param_dict(self)
        if (self.use_cuda_graphs and mode == "mle" and isinstance(mems, RingMems) and self.mem_len > 0
                and mems.length == self.mem_len and mems.bsz == data.shape[1] and torch.is_grad_enabled()
                and self._graph_pending is None and data.dim() == 2):
            if mems.key_start is not None:
                raise L.TganError("a memory that carries a key floor (left-padded prompts) is for inference only: "
                                  "it cannot enter a captured training step")
            ring = eng._prepare_ring(mems, data.shape[1], data.shape[0], self.mem_len)
            if ring is mems:  # steady state: the ring is reused in place, only (start, length) move
                entry = self._graph_entry(eng, data, target, reset_mems, ring)
                self._graph_pending = entry
                out = _TxlGraphFunction.apply(self, entry, names, *[pd[n] for n in names])
                start, length = entry.new_mems
                ring.note_write((ring.start + ring.length) % ring.capacity, data.shape[0])  # the replay wrote the rows
                return out, RingMems(ring.slabs, start, length, self.d_model, kv=ring.kv, shared=ring.shared)
        out = _TxlFunction.apply(self, mode, data, target, reset_mems, mems, temperature, noise, names,
                                 torch.is_grad_enabled(), *[pd[n] for n in names])
        return out, self._new_mems

    def forward(self, data, target, reset_mems, mems, status_vec=None):
        """-> (nll [tgt_len, bsz], new_mems)   (mem_transformer.py:653-670)"""
        if status_vec is not None:
            raise NotImplementedError("status_vec / append_note_status is not accelerated")
        return self._run("mle", data, target, reset_mems, mems)

    def forward_generate(self, data, mems, status_vec=None):
        """-> (logits [T, bsz, n_token] fp32, new_mems)   (mem_transformer.py:578-600)"""
        if status_vec is not None:
            raise NotImplementedError("status_vec / append_note_status is not accelerated")
        return self._run("logits", data, None, None, mems)

    def forward_generate_gumbel(self, data, temperature, mems, status_vec=None, noise=None):
        """-> (straight-through one-hot [T, bsz, n_token], new_mems)   (mem_transformer.py:602-651).
        ``noise``: optional uniform [T, bsz, n_token] tensor replacing the reference's CPU ``torch.rand`` draw
        (parity tests); default is device-side Philox."""
        if status_vec is not None:
            raise NotImplementedError("status_vec / append_note_status is not accelerated")
        return self._run("gumbel", data, None, None, mems, temperature=temperature, noise=noise)

    # ---- batched generation (generate.py:207-304 for a whole batch, sampling on the device) ----------------
    @torch.no_grad()
    def generate_batched(self, start_ids, gen_len, *, technique="topk", topk=32, top_p=0.0, temperature=0.95,
                         exclude_bos=True, empty_token=-1, num_empty_tokens_to_ignore=0, mems=None, uniforms=None,
                         prompt_lengths=None):
        """The generation loop of generate.py:207-304 for ``B`` sequences at once with NO per-token host
        synchronisation: per step one single-token forward (projected-K/V cache, ``memory_length`` = ``self.mem_len``)
        and one ``tgan_sample_tokens`` launch (exclude-BOS, empty-bar suppression once the last
        ``num_empty_tokens_to_ignore`` tokens were all ``empty_token``, temperature, top-k / nucleus / random, one
        categorical draw per sequence); the sampled ids feed the next step on the device.

        start_ids: int64 [T0, B] -- the conditioning tokens (unconditional generation: one row of BOS ids, :180-186).
        uniforms:  optional [gen_len, B] uniforms in [0, 1) replacing the device RNG (parity tests).
        prompt_lengths: optional [B] ints -- prompts of different lengths: sequence b is primed with
                   ``start_ids[:prompt_lengths[b], b]`` (right-padded input; the rows below are ignored).  Each
                   sequence then generates exactly what it would generate alone.  The prompts are left-aligned on the
                   device, and the returned memory carries a per-sequence key floor that hides the pad rows from
                   every later call: ``generate_batched(ids[-1:], n, mems=mems)`` and ``forward_generate`` continue
                   correctly (``mems.materialize()`` returns the pad rows too).  Needs ``mems=None``.  Such a memory
                   is for inference only: it raises in any call that would train through it.
        Returns (ids int64 [gen_len, B], mems)."""
        eng = self._get_engine()
        dev = eng.device
        start_ids = start_ids.to(dev)
        T0, B = start_ids.shape
        mode = {"random": 0, "topk": 1, "nucleus": 2}[technique]
        real = None  # [T0, B] bool: which rows of the (aligned) block are prompt tokens; None = all of them
        if prompt_lengths is not None:
            start_ids, real, mems = self._ragged_prompts(eng, start_ids, prompt_lengths, mems)
            T0 = start_ids.shape[0]
        if T0 > 1:  # context pass over all but the last conditioning token (:190-199)
            _, mems = self._run("logits", start_ids[:-1], None, None, mems)
        cur = start_ids[-1:].contiguous()
        out = torch.empty(gen_len, B, dtype=torch.int64, device=dev)
        k = int(num_empty_tokens_to_ignore)
        run = suppress = None
        if k > 0:
            # length of the run of `empty_token` at the end of each sequence (conditioning tokens included, :235-238)
            run = torch.zeros(B, dtype=torch.int32, device=dev)
            for t in range(T0):  # (pad rows precede a sequence's prompt: they leave the run at 0)
                hit = start_ids[t] == empty_token if real is None else (start_ids[t] == empty_token) & real[t]
                run = torch.where(hit, run + 1, torch.zeros_like(run))
        V = self.n_token
        for t in range(gen_len):
            ectx = eng.forward(cur, None, mems, mem_len=self.mem_len, same_length=self.same_length, training=False,
                               save_for_backward=False)
            mems = ectx.new_mems
            if k > 0:
                suppress = (run >= k).to(torch.uint8)
            eng.calls += 1
            L.sample_tokens(ectx.logits, out[t], V, u=None if uniforms is None else uniforms[t].contiguous(),
                            suppress_empty=suppress, exclude_bos=exclude_bos, empty_token=empty_token, mode=mode,
                            topk=topk or 0, top_p=top_p, temperature=temperature, seed=eng.seed,
                            site=eng._site(eng.calls, 5))
            cur = out[t:t + 1]
            if k > 0:
                run = torch.where(out[t] == empty_token, run + 1, torch.zeros_like(run))
        return out, mems

    def _ragged_prompts(self, eng, start_ids, prompt_lengths, mems):
        """Right-padded prompts [T0, B] of lengths len_b -> (the prompts left-aligned into [max len_b, B], which rows
        of it are real, an empty ring whose key floor starts sequence b at its first real row)."""
        T0, B = start_ids.shape
        if mems is not None:
            raise ValueError("prompt_lengths needs mems=None: pad rows inside an existing memory cannot be masked")
        lens = torch.as_tensor(prompt_lengths).to("cpu", torch.int64).reshape(-1)
        if lens.numel() != B:
            raise ValueError(f"prompt_lengths has {lens.numel()} entries for a batch of {B}")
        if bool((lens < 1).any()) or bool((lens > T0).any()):
            raise ValueError(f"prompt_lengths must lie in [1, {T0}] (the rows of start_ids)")
        T = int(lens.max())
        pad = (T - lens).to(start_ids.device)
        rows = torch.arange(T, device=start_ids.device).view(T, 1)
        # row t of column b holds prompt token t - pad_b; the pad rows repeat token 0 (any valid id: they are masked)
        aligned = start_ids.gather(0, (rows - pad).clamp(min=0))
        ring = eng.new_ring(B, max(T - 1, 1), self.mem_len)
        ring.key_start = pad.to(torch.int32)
        return aligned, rows >= pad, ring

    @torch.no_grad()
    def generate_requests(self, requests, batch_size, *, uniforms=None, context_pass=False):
        """Continue every ``GenRequest`` of a queue, ``batch_size`` sequences at a time: a column that finishes a request
        takes the next one at the following step (``request_schedule``), so no column waits for the longest sequence
        of a fixed batch.  All columns share one ring memory; each column carries a per-sequence key floor raised to
        the first row of its current request, so a request never sees the rows of the requests before it and computes
        what it computes alone.  Per step: the single-token forward of ``generate_batched`` and one
        ``tgan_sample_step`` launch (per-request settings, empty-bar run, sampling, next input), with no host
        synchronisation: the schedule is uploaded once, up front.

        context_pass=False (the default): prompts are fed one token per step, so request r takes its column for
        T_r + gen_len_r - 1 steps.  Request r's tokens equal ``generate_batched(prompt[:, None], gen_len, <its
        settings>, uniforms=u[:, None])`` up to rounding; with ``same_length=False`` that holds for prompts of up to
        mem_len + 2 tokens only: a longer prompt row sees at most mem_len earlier rows here, as every single-token step
        does, while generate_batched's context pass lets it see the whole prompt.  The default keeps these semantics
        for existing callers.

        context_pass=True: prompt[:-1] of each group of ``batch_size`` consecutive requests goes through one ragged
        context pass (the forward of ``generate_batched(prompt_lengths=)``); where a request starts, the last
        min(T_r - 1, mem_len) rows of its pass (layer inputs and projected K/V) are copied into its column right below
        the step's write position (``tgan_ring_scatter``), and the request takes its column for gen_len_r steps only.
        Request r's tokens then equal ``generate_batched(prompt[:, None], gen_len, ...)`` alone up to rounding for every
        prompt length and both ``same_length`` settings.

        requests: list of GenRequest.  uniforms: optional list with one [gen_len_r] tensor of uniforms in [0, 1) per
        request, replacing the device RNG (parity tests).  Returns a list whose entry r is request r's generated ids,
        int64 [gen_len_r] on the model's device (views into one buffer)."""
        if not isinstance(context_pass, bool):
            raise ValueError(f"context_pass must be a bool, got {context_pass!r}")
        reqs = list(requests)
        if not reqs:
            raise ValueError("generate_requests needs at least one request")
        if int(batch_size) < 1:
            raise ValueError(f"batch_size must be >= 1, got {batch_size}")
        if self.mem_len <= 0:
            raise ValueError("generate_requests needs mem_len > 0: the requests of a column share its ring memory")
        V = self.n_token
        prompts, gen_lens, rows_i, rows_f = [], [], [], []
        for r, q in enumerate(reqs):
            p = torch.as_tensor(q.prompt).cpu()
            if p.dim() != 1 or p.numel() < 1 or p.dtype.is_floating_point or p.dtype == torch.bool:
                raise ValueError(f"request {r}: prompt must be a non-empty 1-D integer tensor")
            if int(p.min()) < 0 or int(p.max()) >= V:
                raise ValueError(f"request {r}: prompt tokens must lie in [0, {V})")
            if int(q.gen_len) < 1:
                raise ValueError(f"request {r}: gen_len must be >= 1, got {q.gen_len}")
            if q.technique not in _TECHNIQUES:
                raise ValueError(f"request {r}: unknown technique {q.technique!r} (one of {sorted(_TECHNIQUES)})")
            if q.temperature < 0:
                raise ValueError(f"request {r}: temperature must be >= 0")
            prompts.append(p.tolist())
            gen_lens.append(int(q.gen_len))
            rows_i.append([_TECHNIQUES[q.technique], int(q.topk or 0), int(bool(q.exclude_bos)), int(q.empty_token),
                           int(q.num_empty_tokens_to_ignore)])
            rows_f.append([float(q.temperature), float(q.top_p)])
        if uniforms is not None:
            uniforms = list(uniforms)
            if len(uniforms) != len(reqs):
                raise ValueError(f"uniforms has {len(uniforms)} entries for {len(reqs)} requests")
            for r, (u, g) in enumerate(zip(uniforms, gen_lens)):
                if tuple(u.shape) != (g,):
                    raise ValueError(f"uniforms[{r}] has shape {tuple(u.shape)}, expected ({g},)")
        eng = self._get_engine()
        dev = eng.device
        sch = request_schedule(prompts, gen_lens, int(batch_size), context_pass=context_pass, mem_len=self.mem_len,
                               empty_tokens=[row[3] for row in rows_i])
        S, B = sch.tables.shape[1:]

        def upload(t):  # pinned staging, one cudaMemcpyAsync: no synchronisation
            return t.pin_memory().to(dev, non_blocking=True)

        tables = upload(sch.tables)
        forced, req, out_off, key_start = tables[:4]
        start = tables[4] if context_pass else key_start
        req_i = upload(torch.tensor(rows_i, dtype=torch.int32))
        req_f = upload(torch.tensor(rows_f, dtype=torch.float32))
        u = None
        if uniforms is not None:
            us = [x.reshape(-1).float() for x in uniforms]
            u = upload(torch.cat(us)) if all(x.device.type == "cpu" for x in us) else torch.cat([x.to(dev) for x in us])
        out = torch.empty(sum(gen_lens), dtype=torch.int64, device=dev)
        run = torch.zeros(B, dtype=torch.int32, device=dev)
        cur = forced[0].to(torch.int64).view(1, B)  # the input tokens; tgan_sample_step writes the next ones in place
        run0 = upload(sch.prefill.run0) if context_pass else None
        for t, ectx in self._queue_forwards(eng, sch, key_start, cur, upload):
            eng.calls += 1
            L.sample_step(ectx.logits, req[t], start[t], out_off[t], forced[t + 1] if t + 1 < S else None, req_i,
                          req_f, run, cur, out, V, t, u=u, run0=run0, seed=eng.seed, site=eng._site(eng.calls, 5))
        return [out[b:b + g] for b, g in zip(sch.out_base, gen_lens)]

    def _queue_forwards(self, eng, sch, key_start, cur, upload):
        """The forwards of a request queue, one per step: yields (t, ctx of step t's single-token forward over ``cur``
        [1, B]), the caller writing the next step's inputs into ``cur`` in between.  With a context pass, the prefill
        passes and the copies of their rows run at their steps, before that step's forward.  key_start: the
        schedule's key floors on the device; upload: host tensor -> device without synchronisation."""
        S, B = sch.tables.shape[1:]
        plan, events = sch.prefill, {}
        if plan is not None:
            desc = upload(plan.desc) if plan.desc.numel() else None
            blocks = [b for b in plan.blocks if b is not None]
            flat = upload(torch.cat([b.reshape(-1) for b in blocks])) if blocks else None
            pads = upload(torch.cat(plan.pads))
            passes, bo, po = [], 0, 0  # group g: (prompt block, pad) views into the uploads, or None
            for b, pd in zip(plan.blocks, plan.pads):
                passes.append(None if b is None else (flat[bo:bo + b.numel()].view(b.shape), pads[po:po + pd.numel()]))
                bo += 0 if b is None else b.numel()
                po += pd.numel()
            # per step: the passes enqueued there and the copies applied there, a group's pass before its copies and
            # the copies of an earlier group before a later group's pass (which releases the earlier prefill ring)
            for g, t in enumerate(plan.steps):
                if t is not None:
                    events.setdefault(t, []).append((g, -1, 0, 0))
            for t, sl in plan.slices.items():
                events.setdefault(t, []).extend(sl)
            for ev in events.values():
                ev.sort()
            last = {}  # group -> the step of its last copies, after which its prefill ring is released
            for t, sl in plan.slices.items():
                for g, *_ in sl:
                    last[g] = max(last.get(g, t), t)
            mems = eng.new_queue_ring(B, plan.lead, self.mem_len)  # the row written at step t has position P0 + t
        else:
            mems = eng.new_ring(B, 1, self.mem_len)  # empty, pos0 = 0: the row written at step t has position t
        pre = None  # the ctx of the current group's prefill pass: the only reference to its ring
        for t in range(S):
            for g, lo, n, max_rows in events.get(t, ()):
                if lo < 0:
                    pre = self._prefill_pass(eng, *passes[g])
                else:
                    mems = eng.scatter_prefill(mems, pre, desc, lo, n, max_rows, self.mem_len)
                    if last[g] == t:
                        pre = None  # every request of the group has its rows: release its prefill ring
            mems.key_start = key_start[t]  # a contiguous int32 row of the uploaded table: no copy
            ectx = eng.forward(cur, None, mems, mem_len=self.mem_len, same_length=self.same_length, training=False,
                               save_for_backward=False)
            mems = ectx.new_mems
            yield t, ectx

    def _prefill_pass(self, eng, blk, pad):
        """One group's context pass over its prompt block blk (int64 [Tm, G], column j left-padded by pad[j] rows, pad
        int32 [G]) into a ring of its own -> the forward's ctx (keep_kv=True), which scatter_prefill reads.  The pass
        has no memory, so mem_len enters it only through the same_length shift, and that is the same for every
        mem_len >= Tm: the ring is sized for min(mem_len, Tm) instead of the model's mem_len."""
        ml = min(self.mem_len, blk.shape[0])
        ring = eng.new_ring(blk.shape[1], blk.shape[0], ml)
        ring.key_start = pad
        return eng.forward(blk, None, ring, mem_len=ml, same_length=self.same_length, training=False,
                           save_for_backward=False, keep_kv=True)
