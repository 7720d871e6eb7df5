"""Drop-in replacement of the reference's ``model/mem_transformer.py`` on the libtgan_b200 kernels.

Same module tree, parameter names / shapes (the checkpoint contract, SURVEY.md section 5) and public methods as
the reference -- ``MemTransformerLM(cfg, n_token, vec_len)`` with ``forward(data, target, reset_mems, mems)``
(mem_transformer.py:653), ``forward_generate`` (:578), ``forward_generate_gumbel`` (:602), ``reset_length``
(:432), ``init_mems`` (:436) -- but the sub-modules are parameter containers only: all arithmetic of ``_forward``
(:484-576) and its backward runs in the CUDA library through ``tgan_b200.engine.TxlEngine``.  There is no eager /
CPU fallback: calling the model on a CPU tensor raises.
"""
import contextlib
import os
import weakref

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
