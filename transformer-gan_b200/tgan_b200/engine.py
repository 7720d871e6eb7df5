"""Host-side orchestration of the Transformer-XL generator on the libtgan_b200 kernels.

This file owns *plumbing only*: device buffers (torch tensors used as raw memory), the padded parameter layout,
the recurrence-memory ring buffer and the order in which the C-ABI kernels are enqueued.  All arithmetic happens
in libtgan_b200.so; nothing here calls a torch math op on the hot path.

Reference behaviour implemented (file:line relative to /root/reference/model):
  * MemTransformerLM._forward            mem_transformer.py:484-576
  * RelPartialLearnableMultiHeadAttn     mem_transformer.py:162-257   (post-LN)
  * PositionwiseFF                       mem_transformer.py:46-60     (post-LN)
  * _update_mems                         mem_transformer.py:445-482   (ring buffer: zero-copy)
  * ProjectedAdaptiveLogSoftmax          utils/proj_adaptive_softmax.py:64-84 (cutoffs == [])
and the closed-form backward of all of them (SURVEY.md section 9).
"""
from __future__ import annotations

import contextlib
import math
from dataclasses import dataclass
from typing import Dict, List, Optional, Tuple

import torch

from . import lib as L


def _ceil(x: int, m: int) -> int:
    return (x + m - 1) // m * m


@dataclass
class TxlDims:
    n_layer: int
    n_head: int
    d_model: int
    d_inner: int
    n_token: int
    dropout: float = 0.0
    dropatt: float = 0.0
    clamp_len: int = -1

    @property
    def d_head(self) -> int:
        return self.d_model // self.n_head

    @property
    def DP(self) -> int:
        return _ceil(self.d_model, 64)

    @property
    def NH(self) -> int:
        return self.n_head * L.HS

    @property
    def DIP(self) -> int:
        return _ceil(self.d_inner, 64)

    @property
    def VP(self) -> int:
        return _ceil(self.n_token, 64)


# ---------------------------------------------------------------------------------------------------------
# recurrence memory: ring buffer of the layer inputs (mem_transformer.py:445-482 without the copy)
# ---------------------------------------------------------------------------------------------------------
class RingMems:
    """Per-layer-input memory [n_layer+1 slabs] x [capacity positions] x [B] x [DP] in the compute dtype.

    ``start`` is the ring position of logical memory row 0, ``length`` the number of valid memory rows.
    The reference returns a fresh ``[n_layer+1, M, B, d_model]`` fp32 tensor per call; ``materialize()``
    produces exactly that tensor (for tests, checkpoints and the generate.py self-check).

    A ring that holds left-padded prompts of different lengths (``generate_batched(prompt_lengths=...)``) carries a
    per-sequence key floor: ``key_start`` (device int32 [B]) is the absolute position of the first real row of each
    sequence and ``pos0`` the absolute position of logical memory row 0; every forward over the ring masks the keys
    below the floor (tgan_relattn_fwd_ragged).  ``key_start`` is None for every other ring.  Such a ring is for
    inference only: a forward that saves activations for a backward raises."""

    def __init__(self, slabs: torch.Tensor, start: int, length: int, d_model: int, kv: Optional[dict] = None,
                 shared: Optional[dict] = None, key_start: Optional[torch.Tensor] = None, pos0: int = 0):
        self.slabs = slabs
        self.start = start
        self.length = length
        self.d_model = d_model
        self.key_start = key_start  # shared by every window over the same slabs, like ``kv``
        self.pos0 = pos0
        # State shared by every window (handle) over the same slabs: ``gen`` counts the writes into the ring and
        # ``writes`` logs the most recent ones as (gen, position, count).  A handle remembers the generation it was
        # produced at; it stays valid until a LATER write lands inside its window (the reference returns fresh
        # tensors, so an old ``mems`` may legally be passed again -- here that works as long as its rows are intact,
        # and raises instead of silently attending over overwritten rows otherwise).
        self.shared = shared if shared is not None else {"gen": 0, "writes": []}
        self.gen = self.shared["gen"]
        # projected-K/V cache of the ring rows (decode-sized calls only, see TxlEngine.forward): shared by every
        # RingMems window over the same slabs.  {"buf": [n_layer, capacity, B, 2*N*64], "lo", "hi": cached physical
        # rows, "tag": parameter-pack epoch the rows were projected with}
        self.kv = kv if kv is not None else {"buf": None, "lo": 0, "hi": 0, "tag": -1}

    @property
    def capacity(self) -> int:
        return self.slabs.shape[1]

    @property
    def bsz(self) -> int:
        return self.slabs.shape[2]

    def check_fresh(self):
        """Raise if a write issued after this handle was produced overwrote one of its rows."""
        if self.length == 0:
            return
        C = self.capacity
        log = self.shared["writes"]
        if log and log[0][0] > self.gen + 1 and self.shared["gen"] - self.gen > len(log):
            raise L.TganError("stale memory handle: older than the ring's write log (pass the most recent `new_mems`)")
        for g, pos, cnt in log:
            if g <= self.gen:
                continue
            # overlap of the circular ranges [pos, pos+cnt) and [start, start+length)
            d = (pos - self.start) % C
            if d < self.length or d + cnt > C:
                raise L.TganError(
                    "stale memory handle: rows of this `mems` were overwritten by a later forward on the same ring "
                    "(the ring-buffer memory aliases storage; pass the most recent `new_mems`, or "
                    "`mems.materialize()` a copy if an old memory must be kept)")

    def note_write(self, pos: int, count: int) -> int:
        sh = self.shared
        sh["gen"] += 1
        sh["writes"] = [w for w in sh["writes"][-63:]] + [(sh["gen"], pos, count)]
        return sh["gen"]

    def segments(self, first: int, count: int) -> List[Tuple[int, int]]:
        """physical (position, count) runs covering logical rows [first, first+count)."""
        out, C = [], self.capacity
        pos = (self.start + first) % C
        while count > 0:
            n = min(count, C - pos)
            out.append((pos, n))
            pos = (pos + n) % C
            count -= n
        return out

    def materialize(self) -> torch.Tensor:
        """-> fp32 [n_layer+1, length, B, d_model] (logical order), via tgan_convert.  Every row, the pad rows below
        a ``key_start`` floor included: row m of sequence b is real iff pos0 + m >= key_start[b]."""
        S, C, B, DP = self.slabs.shape
        out = torch.empty(S, self.length, B, self.d_model, dtype=torch.float32, device=self.slabs.device)
        for s in range(S):
            row = 0
            for pos, n in self.segments(0, self.length):
                L.convert(self.slabs, DP, out, self.d_model, n * B, self.d_model, self.d_model,
                          src_off=(s * C + pos) * B * DP, dst_off=(s * self.length + row) * B * self.d_model)
                row += n
        return out

    # tensor-ish conveniences used by callers that treat mems as opaque
    def size(self, dim=None):
        shp = (self.slabs.shape[0], self.length, self.bsz, self.d_model)
        return shp if dim is None else shp[dim]

    @property
    def shape(self):
        return self.size()

    def __len__(self):
        return self.slabs.shape[0]

    def __iter__(self):
        return iter(self.materialize())

    def detach(self):
        return self

    def numel(self):
        s = self.size()
        return s[0] * s[1] * s[2] * s[3]


# ---------------------------------------------------------------------------------------------------------
# parameter layout
# ---------------------------------------------------------------------------------------------------------
class ParamLayout:
    """Offsets of the padded (kernel-private) parameter copies and of the padded fp32 gradient buffers."""

    def __init__(self, d: TxlDims):
        self.d = d
        DP, NH, DIP, VP = d.DP, d.NH, d.DIP, d.VP
        self.mat: Dict[str, Tuple[int, int, int]] = {}  # name -> (offset, rows, ld)
        self.gmat: Dict[str, Tuple[int, int, int]] = {}
        self.vec: Dict[str, Tuple[int, int]] = {}  # name -> (offset, n)
        mo = go = vo = 0

        def add_mat(name, rows, ld, grad=True, transposed=True):
            nonlocal mo, go
            self.mat[name] = (mo, rows, ld)
            mo += rows * ld
            if transposed:
                self.mat[name + ".T"] = (mo, ld, rows)
                mo += rows * ld
            if grad:
                self.gmat[name] = (go, rows, ld)
                go += rows * ld

        def add_vec(name, n):
            nonlocal vo
            self.vec[name] = (vo, n)
            vo += n

        add_mat("E", VP, DP)
        # the r_net weights of all layers sit back to back: r = r_net(pos_emb) of every layer is ONE GEMM per forward
        # ([K, n_layer * N*64]), and their gradients one GEMM per backward
        for l in range(d.n_layer):
            add_mat(f"l{l}.Wr", NH, DP, transposed=False)
        add_vec("u", NH)
        add_vec("vb", NH)
        add_vec("bias_out", VP)
        for l in range(d.n_layer):
            p = f"l{l}."
            add_mat(p + "Wqkv", 3 * NH, DP)
            add_mat(p + "Wo", DP, NH)
            add_mat(p + "W1", DIP, DP)
            add_mat(p + "W2", DP, DIP)
            for v, n in (("b1", DIP), ("b2", DP), ("ln1_g", DP), ("ln1_b", DP), ("ln2_g", DP), ("ln2_b", DP)):
                add_vec(p + v, n)
        self.mat_elems, self.gmat_elems, self.vec_elems = mo, go, vo

    def reference_map(self):
        """(reference state_dict name, packed name, kind, row_group, row_pad, col_group, col_pad)."""
        d = self.d
        dh = d.d_head
        out = [("word_emb.emb_layers.0.weight", "E", "mat", 1, 1, 1, 1),
               ("r_w_bias", "u", "vec", 1, 1, dh, L.HS),
               ("r_r_bias", "vb", "vec", 1, 1, dh, L.HS),
               ("crit.out_layers.0.bias", "bias_out", "vec", 1, 1, 1, 1)]
        for l in range(d.n_layer):
            r, p = f"layers.{l}.", f"l{l}."
            out += [
                (r + "dec_attn.qkv_net.weight", p + "Wqkv", "mat", dh, L.HS, 1, 1),
                (r + "dec_attn.r_net.weight", p + "Wr", "mat", dh, L.HS, 1, 1),
                (r + "dec_attn.o_net.weight", p + "Wo", "mat", 1, 1, dh, L.HS),
                (r + "pos_ff.CoreNet.0.weight", p + "W1", "mat", 1, 1, 1, 1),
                (r + "pos_ff.CoreNet.3.weight", p + "W2", "mat", 1, 1, 1, 1),
                (r + "pos_ff.CoreNet.0.bias", p + "b1", "vec", 1, 1, 1, 1),
                (r + "pos_ff.CoreNet.3.bias", p + "b2", "vec", 1, 1, 1, 1),
                (r + "dec_attn.layer_norm.weight", p + "ln1_g", "vec", 1, 1, 1, 1),
                (r + "dec_attn.layer_norm.bias", p + "ln1_b", "vec", 1, 1, 1, 1),
                (r + "pos_ff.layer_norm.weight", p + "ln2_g", "vec", 1, 1, 1, 1),
                (r + "pos_ff.layer_norm.bias", p + "ln2_b", "vec", 1, 1, 1, 1),
            ]
        return out


class _Ctx:
    """Everything one forward saved for its backward."""
    pass


# bumped by notify_params_updated(): optimizers that write the parameter storage directly (tgan_b200.dp.FusedClipAdam
# on a FlatParams buffer) tell every engine to re-pack at its next forward
_PARAM_EPOCH = [0]


def notify_params_updated() -> None:
    _PARAM_EPOCH[0] += 1


class TxlEngine:
    """Forward / backward of the generator stack on libtgan_b200."""

    def __init__(self, dims: TxlDims, device, dtype=torch.bfloat16, seed: int = 1111, impl: int = L.IMPL_AUTO):
        if dims.d_head > L.HS:
            raise NotImplementedError(f"d_head {dims.d_head} > {L.HS} is not supported by the attention kernels")
        if dims.d_model % 2:
            raise NotImplementedError("odd d_model")
        self.d = dims
        self.device = torch.device(device)
        self.dtype = dtype
        self.impl = impl
        self.seed = seed
        self.calls = 0
        self.layout = ParamLayout(dims)
        lay = self.layout
        self.pmat = torch.zeros(lay.mat_elems, dtype=dtype, device=self.device)
        self.pvec = torch.zeros(lay.vec_elems, dtype=torch.float32, device=self.device)
        self.gmat = torch.zeros(lay.gmat_elems, dtype=torch.float32, device=self.device)
        self.gvec = torch.zeros(lay.vec_elems, dtype=torch.float32, device=self.device)
        self.inv_freq = (1 / (10000 ** (torch.arange(0.0, dims.d_model, 2.0) / dims.d_model))).to(self.device)
        self._params: Optional[Dict[str, torch.Tensor]] = None
        self._param_key = None
        self._packed_version = None
        self._dirty = False        # a backward ran since the last pack (an optimizer step may have followed)
        self._pack_desc = None
        self._unpack_cache: Dict[tuple, torch.Tensor] = {}
        self._es = 2 if dtype == torch.bfloat16 else 4
        self.pack_epoch = 0        # bumped whenever the packed parameter copies are rewritten
        self.kv_cache_max_q = 8    # calls with at most this many new rows keep / reuse the projected-K/V cache
        # Calls with at most this many query rows (the single-token steps of the sampling chain: R = batch) are a
        # string of launch-latency-bound kernels on a fraction of the SMs: their weight-gradient GEMMs (off the
        # backward's critical path) and the K/V projection of the forward run on a side stream, concurrently with the
        # dgrad chain.  Captured in a CUDA graph the fork / join events become plain dependency edges.
        self.side_stream_max_rows = 8192
        self._side = None
        self._window = None        # open gradient window: number of backward calls accumulated so far
        self._late = None          # (side event, side2 event, buffers) of the previous single-token backward in the window

    # -- parameters ---------------------------------------------------------------------------------------
    def bind_params(self, params: Dict[str, torch.Tensor]):
        """params: reference-layout fp32 CUDA tensors keyed by generator state_dict names."""
        key = tuple((n, params[n].data_ptr()) for n, *_ in self.layout.reference_map())
        if key == self._param_key:
            self._params = params
            return
        d, lay = self.d, self.layout
        rows_pack, rows_unpack, max_elems = [], [], 1
        self._grad_shapes = {}
        for ref, name, kind, rg, rgp, cg, cgp in lay.reference_map():
            t = params[ref]
            if t.dtype != torch.float32 or not t.is_cuda or not t.is_contiguous():
                raise L.TganError(f"parameter {ref} must be a contiguous fp32 CUDA tensor")
            if t.dim() == 2:
                r, c = t.shape
            else:
                r, c = 1, t.numel()
            if name in ("u", "vb"):
                r, c = 1, t.numel()  # [N, dh] flattened: column groups of dh -> 64
            max_elems = max(max_elems, r * c)
            self._grad_shapes[ref] = tuple(t.shape)
            if kind == "mat":
                off, _, ld = lay.mat[name]
                rows_pack.append([t.data_ptr(), off, r, c, ld, rg, rgp, cg, cgp, 0, 0, 0])
                if name + ".T" in lay.mat:
                    offt, _, ldt = lay.mat[name + ".T"]
                    rows_pack.append([t.data_ptr(), offt, r, c, ldt, rg, rgp, cg, cgp, 1, 0, 0])
                goff, _, gld = lay.gmat[name]
                rows_unpack.append([0, goff, r, c, gld, rg, rgp, cg, cgp, 0, 0, 0])
            else:
                off, _ = lay.vec[name]
                rows_pack.append([t.data_ptr(), off, r, c, c, rg, rgp, cg, cgp, 0, 1, 0])
                if name.endswith(".b1") and d.DP > d.d_model:
                    # db1 is column d_model of the padded dW1 (ones column in LayerNorm-1's pad lane, see forward):
                    # read it as a [d_inner, 1] matrix with row pitch DP out of the matrix-gradient buffer
                    goff, _, gld = lay.gmat[name[:-2] + "W1"]
                    rows_unpack.append([0, goff + d.d_model, c, 1, gld, 1, 1, 1, 1, 0, 0, 0])
                else:
                    rows_unpack.append([0, off, r, c, c, rg, rgp, cg, cgp, 0, 1, 0])
        self._pack_desc = torch.tensor(rows_pack, dtype=torch.int64, device=self.device)
        self._unpack_rows = rows_unpack
        self._max_elems = max_elems
        self._params = params
        self._param_key = key
        self._packed_version = None
        self.pmat.zero_()
        self.pvec.zero_()

    def invalidate(self):
        """The parameters changed behind autograd's back (``p.data.add_``, a flat-buffer optimizer, a raw copy into the
        storage): re-pack the kernel-private copies at the next forward.  ``tgan_b200.dp`` optimizers call
        ``notify_params_updated()``; for third-party optimizers the engine re-packs on the first forward after any
        backward on its own (an optimizer step is always preceded by one), see ``pack``."""
        self._packed_version = None

    def pack(self):
        """Refresh the padded bf16 / fp32 parameter copies when the parameters may have changed: a version-counter
        change (in-place autograd-visible updates, load_state_dict), an explicit invalidate(), a
        notify_params_updated() from a flat-buffer optimizer, or any backward since the last pack (covers optimizers
        that update through ``p.data``, e.g. the reference's lamb.py:116, which bumps no version counter)."""
        ver = (tuple(p._version for p in self._params.values()), _PARAM_EPOCH[0])
        if ver == self._packed_version and not self._dirty:
            return
        L.pack_params(self.pmat, self.pvec, self._pack_desc, self._pack_desc.shape[0], self._max_elems)
        self._packed_version = ver
        self._dirty = False
        self.pack_epoch += 1

    def _m(self, name):  # (tensor, element offset, ld)
        off, rows, ld = self.layout.mat[name]
        return off, ld

    def _v(self, name) -> int:  # pointer (int) into pvec
        return self.pvec.data_ptr() + 4 * self.layout.vec[name][0]

    def _gv(self, name) -> int:
        return self.gvec.data_ptr() + 4 * self.layout.vec[name][0]

    # -- helpers ------------------------------------------------------------------------------------------
    def graph_pool(self):
        """One private memory pool shared by every captured segment (they are replayed strictly one after another)."""
        if getattr(self, "_graph_pool", None) is None:
            self._graph_pool = torch.cuda.graph_pool_handle()
        return self._graph_pool

    # -- gradient window -----------------------------------------------------------------------------------
    def begin_grad_window(self):
        """Until end_grad_window(), backward() calls ACCUMULATE into the padded gradient buffers without zeroing them
        first and without unpacking at the end: the 123 single-token backward calls of a sampling chain share one
        60 MB zero-fill and one unpack into the reference-layout gradients instead of paying both per token
        (every gradient kernel of the stack accumulates: TMA reduce-add / atomics)."""
        if self._window is not None:
            raise L.TganError("gradient window already open")
        self.gvec.zero_()
        self.gmat.zero_()
        self._window = 0

    def end_grad_window(self, grad_targets: Dict[str, torch.Tensor], accumulate: bool = True) -> int:
        """Unpack what the window accumulated into ``grad_targets`` (+= when ``accumulate``); returns the number of
        backward calls it covered (0: nothing to unpack)."""
        n, self._window = self._window, None
        if self._late is not None:  # join the side streams of the window's last backward call
            main = torch.cuda.current_stream()
            main.wait_event(self._late[0])
            main.wait_event(self._late[1])
            self._late[2].clear()
            self._late = None
        if n:
            desc = self._unpack_desc_for(grad_targets)
            L.unpack_grads(self.gmat, self.gvec, desc, desc.shape[0], self._max_elems, accumulate=accumulate)
        return n or 0

    def _use_side_streams(self, rows: int) -> bool:
        """Small calls inside a CUDA-graph capture only: launched from the host these calls are enqueue-bound (the GPU
        idles between kernels anyway) and every stream switch costs host time -- a generation step went from 1.6 to
        3.2 ms of host work with the forks enabled."""
        return rows <= self.side_stream_max_rows and torch.cuda.is_current_stream_capturing()

    def _side_stream(self, i: int = 0):
        if self._side is None:
            self._side = [torch.cuda.Stream(device=self.device) for _ in range(2)]
        return self._side[i]

    def _site(self, call_id: int, local: int) -> int:
        return call_id * 256 + local

    def _buf(self, *shape, dtype=None):
        return torch.empty(*shape, dtype=dtype or self.dtype, device=self.device)

    def new_ring(self, B: int, Q: int, mem_len: int) -> RingMems:
        # decode-sized segments get a longer ring: the window then slides mem_len steps before a re-layout is due
        cap = mem_len + Q if Q > self.kv_cache_max_q else 2 * mem_len + Q
        slabs = torch.zeros(self.d.n_layer + 1, cap, B, self.d.DP, dtype=self.dtype, device=self.device)
        return RingMems(slabs, 0, 0, self.d.d_model)

    def import_mems(self, mems: torch.Tensor, Q: int, mem_len: int) -> RingMems:
        """reference-layout fp32 mems [n_layer+1, M, B, d_model] -> ring (tgan_convert pads and casts)."""
        S, M, B, D = mems.shape
        ring = self.new_ring(B, Q, max(mem_len, M))
        mems = mems.contiguous().float()
        C, DP = ring.capacity, self.d.DP
        for s in range(S):
            L.convert(mems, D, ring.slabs, DP, M * B, D, DP, src_off=s * M * B * D, dst_off=s * C * B * DP)
        ring.length = M
        return ring

    def _prepare_ring(self, mems, B: int, Q: int, mem_len: int) -> RingMems:
        if mems is None or (isinstance(mems, torch.Tensor) and mems.numel() == 0):
            return self.new_ring(B, Q, mem_len)
        if isinstance(mems, torch.Tensor):
            return self.import_mems(mems, Q, mem_len)
        ring: RingMems = mems
        if ring.bsz != B:
            raise L.TganError(f"memory batch size {ring.bsz} != input batch size {B}")
        ring.check_fresh()
        # An incoming memory longer than mem_len (reset_length shrank it between calls) is attended over in full and
        # truncated afterwards, as the reference does (mem_transformer.py:556-575, 463-470).
        n = ring.length
        w = (ring.start + n) % ring.capacity
        # decode-sized calls keep [memory; new rows] physically contiguous (the projected-K/V cache and the attention
        # kernels' single K / V base pointer need it): compact just before the window would wrap
        wraps = Q <= self.kv_cache_max_q and ring.start + n + Q > ring.capacity
        if ring.capacity < n + Q or w + Q > ring.capacity or ring.capacity < mem_len + Q or wraps:
            # re-layout: the write position reached the end of the buffer (every capacity - mem_len decode steps) or
            # tgt_len / mem_len changed between calls
            return self._relayout(ring, Q, mem_len)
        return ring

    def _relayout(self, ring: RingMems, Q: int, mem_len: int) -> RingMems:
        """Compact the live window to position 0 of a fresh ring in the compute dtype (plain row copies), carrying the
        projected-K/V cache rows along so that a long decode never re-projects its memory."""
        new = self.new_ring(ring.bsz, Q, max(mem_len, ring.length))
        n = ring.length
        keep_kv = (ring.kv["buf"] is not None and ring.kv["tag"] == self.pack_epoch and n > 0 and
                   len(ring.segments(0, n)) == 1 and ring.kv["lo"] <= ring.start and ring.kv["hi"] == ring.start + n)
        row = 0
        for pos, cnt in ring.segments(0, n):
            new.slabs[:, row:row + cnt].copy_(ring.slabs[:, pos:pos + cnt])
            row += cnt
        if keep_kv:
            buf = ring.kv["buf"]
            nb = torch.empty(buf.shape[0], new.capacity, buf.shape[2], buf.shape[3], dtype=buf.dtype, device=buf.device)
            nb[:, :n].copy_(buf[:, ring.start:ring.start + n])
            new.kv.update(buf=nb, lo=0, hi=n, tag=self.pack_epoch)
        new.length = n
        new.gen = new.shared["gen"]
        new.key_start, new.pos0 = ring.key_start, ring.pos0  # logical row 0 stays row 0
        return new

    def new_queue_ring(self, B: int, lead: int, mem_len: int) -> RingMems:
        """The ring of a request queue whose prompts are prefilled by context passes (scatter_prefill): ``lead``
        leading rows, zero and meant to be floored, then the decode steps' rows (pos0 = 0: the row of step t has
        absolute position lead + t).  Its projected-K/V cache exists from the start, tagged with the current parameter
        pack and covering the leading rows, so the first step projects only its new row and the K/V rows that
        scatter_prefill writes count as cached."""
        self.pack()
        ring = self.new_ring(B, 1, mem_len)
        ring.length = lead
        buf = torch.empty(self.d.n_layer, ring.capacity, B, 2 * self.d.NH, dtype=self.dtype, device=self.device)
        buf[:, :lead].zero_()
        ring.kv.update(buf=buf, lo=0, hi=lead, tag=self.pack_epoch)
        return ring

    def scatter_prefill(self, ring: RingMems, src: _Ctx, desc: torch.Tensor, lo: int, n: int, max_rows: int,
                        mem_len: int) -> RingMems:
        """Copy prefilled rows into a request queue's ring right below the next single-token step's write position
        (tgan_ring_scatter): descriptors desc[lo:lo+n] (device int32 [*, 4]: source column, first source position,
        destination column, rows <= max_rows) read the ring and the K/V rows of ``src``, the ctx of a
        ``forward(keep_kv=True)`` over the prompts.  The ring is prepared for that step first, so a re-layout that is
        due happens before the copy and the rows land in the window the step reads.  Returns that ring."""
        ring = self._prepare_ring(ring, ring.bsz, 1, mem_len)
        w = ring.start + ring.length  # a decode ring keeps [memory; next row] contiguous: no wrap
        if max_rows > ring.length:
            raise L.TganError(f"internal: {max_rows} prefilled rows do not fit a window of {ring.length}")
        st = ring.kv
        kv_ok = st["buf"] is not None and st["tag"] == self.pack_epoch and st["lo"] <= ring.start and st["hi"] == w
        kv, kv_stride = src.kv_rows
        C, B = ring.capacity, ring.bsz
        # a stale K/V cache is re-projected from the slabs by the next forward: then only the slabs are copied
        L.ring_scatter(desc, n, max_rows, w, src.ring.slabs, ring.slabs, kv if kv_ok else None,
                       st["buf"] if kv_ok else None, src_kv_stride=kv_stride, dst_kv_stride=C * B * 2 * self.d.NH,
                       desc_off=lo)
        return ring

    # -- forward ------------------------------------------------------------------------------------------
    def forward(self, inp: torch.Tensor, reset: Optional[torch.Tensor], mems, *, mem_len: int, same_length: bool,
                training: bool, target: Optional[torch.Tensor] = None, n_pred: Optional[int] = None,
                save_for_backward: bool = True, keep_kv: bool = False) -> _Ctx:
        """inp: int64 [Q,B] token ids or float [Q,B,V] soft one-hot rows.  Returns a ctx with
        ``nll`` (fp32 [T*B], when target is given), ``logits`` (fp32 [T*B, VP]) and ``new_mems``.
        keep_kv: the ctx also exposes the projected K/V rows of every layer as ``kv_rows`` = (tensor, layer stride in
        elements), row (position p, sequence b) of layer l at element l * stride + (p * B + b) * 2 * NH, p a physical
        ring position (scatter_prefill reads them).  Calls with Q <= kv_cache_max_q find them in the ring's K/V cache;
        longer ones keep their per-layer K/V rows in one [n_layer, K*B, 2*NH] buffer, which needs [memory; segment]
        to start at ring position 0 (a fresh ring)."""
        d, lay, dt = self.d, self.layout, self.dtype
        DP, NH, DIP, VP, D = d.DP, d.NH, d.DIP, d.VP, d.d_model
        if save_for_backward and getattr(mems, "key_start", None) is not None:
            # no backward kernel honours the key floor: the gradients would include the pad rows
            raise L.TganError("a memory that carries a key floor (left-padded prompts) is for inference only: "
                              "it cannot be used in a forward that saves activations for a backward")
        self.pack()
        Q, B = inp.shape[0], inp.shape[1]
        ring = self._prepare_ring(mems, B, Q, mem_len) if mem_len > 0 else self.new_ring(B, Q, 0)
        M = ring.length
        K = M + Q
        R, KR = Q * B, K * B
        C = ring.capacity
        w = (ring.start + M) % C  # write position of this segment
        if w + Q > C:
            raise L.TganError("internal: ring write would wrap")
        if mem_len > 0:
            ring.note_write(w, Q)
        self.calls += 1
        cid = self.calls
        p_drop = d.dropout if training else 0.0
        p_att = d.dropatt if training else 0.0
        seed = self.seed
        ctx = _Ctx()
        ctx.Q, ctx.B, ctx.M, ctx.K, ctx.cid, ctx.p_drop, ctx.p_att = Q, B, M, K, cid, p_drop, p_att
        ctx.ring, ctx.w, ctx.same_length, ctx.training = ring, w, same_length, training
        slab_elems = C * B * DP
        cur_off = [s * slab_elems + w * B * DP for s in range(d.n_layer + 1)]
        ctx.cur_off = cur_off
        ctx.mem_segs = ring.segments(0, M)
        # contiguous runs of [memory rows; current rows] in logical order
        segs = list(ctx.mem_segs) + [(w, Q)]
        merged = []
        for pos, n in segs:
            if merged and merged[-1][0] + merged[-1][1] == pos:
                merged[-1] = (merged[-1][0], merged[-1][1] + n)
            else:
                merged.append((pos, n))
        ctx.x_segs = merged
        if keep_kv and not (Q <= self.kv_cache_max_q and mem_len > 0 and len(merged) == 1) and \
                (len(merged) != 1 or merged[0][0] != 0):
            raise L.TganError("keep_kv: a segment longer than kv_cache_max_q keeps its K/V rows only on a fresh ring")
        # same_length mask shift (mem_transformer.py:496-503)
        msl = Q
        if same_length:
            mask_len = K - mem_len
            msl = Q - mask_len if mask_len > 0 else Q
        ctx.msl = msl
        reset_u8 = None
        if reset is not None and M > 0:
            reset_u8 = reset.to(device=self.device, dtype=torch.uint8).contiguous()
        ctx.reset = reset_u8
        slabs = ring.slabs
        es = self._es

        # 1. embedding (-> ring slab 0, current rows)
        if inp.dim() == 2:
            ids = inp.to(self.device).contiguous()
            ctx.ids, ctx.soft = ids, None
            eoff, eld = self._m("E")
            L.embed_fwd(ids, self.pmat[eoff:], slabs, R, D, DP, math.sqrt(D), p_drop, seed, self._site(cid, 0),
                        out_off=cur_off[0])
        else:
            V = d.n_token
            soft = self._buf(R, VP)
            L.convert(inp.contiguous().float(), V, soft, VP, R, V, VP)
            ctx.ids, ctx.soft = None, soft
            etoff, etld = self._m("E.T")
            L.gemm(soft, self.pmat, slabs, transB=True, M=R, N=D, K=VP, lda=VP, ldb=etld, ldc=DP, b_off=etoff,
                   c_off=cur_off[0], alpha=math.sqrt(D), flags=L.EPI_DROPOUT if p_drop > 0 else 0, drop_p=p_drop,
                   seed=seed, site=self._site(cid, 0), impl=self.impl)
        # 2. positional embedding
        pe = self._buf(K, DP)
        L.pos_emb(self.inv_freq, pe, K, D, DP, d.clamp_len, p_drop, seed, self._site(cid, 1))
        ctx.pe = pe
        scale = 1.0 / math.sqrt(d.d_head)
        ctx.layers = []
        r_all = self._buf(K, d.n_layer * NH)
        L.gemm(pe, self.pmat, r_all, M=K, N=d.n_layer * NH, K=DP, ldb=DP, b_off=self._m("l0.Wr")[0], impl=self.impl)
        # Projected-K/V cache (SURVEY section 10: the reference re-projects every memory row at each of the 123 sampling
        # steps / every generated token, mem_transformer.py:166-170).  For decode-sized calls the K/V rows live in a
        # buffer that mirrors the ring; rows projected by an earlier call with the same packed parameters are reused
        # and only the new rows go through the GEMM.  Same values up to nothing: the rows are bit-identical.
        use_cache = Q <= self.kv_cache_max_q and mem_len > 0 and len(ctx.x_segs) == 1
        kv_from = 0
        kv_all = None
        if keep_kv and not use_cache:
            kv_all = self._buf(d.n_layer, KR, 2 * NH)
        if use_cache:
            st, s0 = ring.kv, ctx.x_segs[0][0]
            if st["buf"] is None or st["buf"].shape[1:3] != (C, B) or st["buf"].dtype != dt:
                st["buf"] = torch.empty(d.n_layer, C, B, 2 * NH, dtype=dt, device=self.device)
                st["tag"] = -1
            cached = M > 0 and st["tag"] == self.pack_epoch and st["lo"] <= s0 and st["hi"] == w
            kv_from = w if cached else s0  # first physical row that still has to be projected
        for l in range(d.n_layer):
            p = f"l{l}."
            sv = _Ctx()
            woff, wld = self._m(p + "Wqkv")
            # single-token calls: q (and, in the backward, dq) are the first third of [R, 3 * NH] rows -- the backward then
            # has dq | dk | dv of the current position side by side and needs ONE dgrad / wgrad GEMM for them
            q = self._buf(R, 3 * NH)[:, :NH] if Q == 1 else self._buf(R, NH)
            r = r_all[:, l * NH:(l + 1) * NH]  # view: row pitch n_layer * NH
            x_base = l * slab_elems
            if use_cache:
                kv, kv_off = ring.kv["buf"], (l * C + ctx.x_segs[0][0]) * B * 2 * NH
                side = self._side_stream() if self._use_side_streams(R) else None
                main = torch.cuda.current_stream()
                if side is not None:  # the K/V projection of the new rows runs beside the Q projection
                    side.wait_stream(main)
                with (torch.cuda.stream(side) if side is not None else contextlib.nullcontext()):
                    L.gemm(slabs, self.pmat, kv, M=(w + Q - kv_from) * B, N=2 * NH, K=DP, lda=DP, ldb=wld, ldc=2 * NH,
                           a_off=x_base + kv_from * B * DP, b_off=woff + NH * wld, c_off=(l * C + kv_from) * B * 2 * NH,
                           impl=self.impl)
            L.gemm(slabs, self.pmat, q, M=R, N=NH, K=DP, lda=DP, ldb=wld, a_off=cur_off[l], b_off=woff, impl=self.impl)
            if use_cache:
                if side is not None:
                    main.wait_stream(side)
            else:
                kv, kv_off = (self._buf(KR, 2 * NH) if kv_all is None else kv_all[l]), 0
                row = 0
                for pos, n in ctx.x_segs:
                    L.gemm(slabs, self.pmat, kv, M=n * B, N=2 * NH, K=DP, lda=DP, ldb=wld, a_off=x_base + pos * B * DP,
                           b_off=woff + NH * wld, c_off=row * B * 2 * NH, impl=self.impl)
                    row += n
            att = self._buf(R, NH)
            lse = self._buf(B * d.n_head * Q, dtype=torch.float32)
            L.relattn_fwd(q, kv, kv, 2 * NH, r, self._v("u"), self._v("vb"), reset_u8, att, lse, B, d.n_head, Q, M, msl,
                          same_length, scale, p_att, seed, self._site(cid, 8 + 4 * l), impl=self.impl, k_off=kv_off,
                          v_off=kv_off + NH, key_start=ring.key_start, key_base=ring.pos0)
            # O projection + dropout + residual (fp32) -> LN
            ooff, old = self._m(p + "Wo")
            z1 = self._buf(R, DP, dtype=torch.float32)
            L.gemm(att, self.pmat, z1, M=R, N=DP, K=NH, ldb=old, b_off=ooff, aux=slabs, aux_off=cur_off[l], ldaux=DP,
                   flags=L.EPI_ADD_AUX | (L.EPI_DROPOUT if p_drop > 0 else 0), drop_p=p_drop, seed=seed,
                   site=self._site(cid, 9 + 4 * l), impl=self.impl)
            a = self._buf(R, DP)
            mean1, rstd1 = self._buf(R, dtype=torch.float32), self._buf(R, dtype=torch.float32)
            # lane D of `a` is a ones column when the padding leaves room: dW1 = dh^T a then carries db1 in column D
            L.ln_fwd(z1, a, self._v(p + "ln1_g"), self._v(p + "ln1_b"), mean1, rstd1, R, D, DP, pad_one=DP > D)
            # FFN
            w1off, w1ld = self._m(p + "W1")
            h = self._buf(R, DIP)
            L.gemm(a, self.pmat, h, M=R, N=DIP, K=DP, ldb=w1ld, b_off=w1off, bias=self._v(p + "b1"),
                   flags=L.EPI_BIAS | L.EPI_RELU | (L.EPI_DROPOUT if p_drop > 0 else 0), drop_p=p_drop, seed=seed,
                   site=self._site(cid, 10 + 4 * l), impl=self.impl)
            w2off, w2ld = self._m(p + "W2")
            z2 = self._buf(R, DP, dtype=torch.float32)
            L.gemm(h, self.pmat, z2, M=R, N=DP, K=DIP, ldb=w2ld, b_off=w2off, bias=self._v(p + "b2"), aux=a, ldaux=DP,
                   flags=L.EPI_BIAS | L.EPI_ADD_AUX | (L.EPI_DROPOUT if p_drop > 0 else 0), drop_p=p_drop, seed=seed,
                   site=self._site(cid, 11 + 4 * l), impl=self.impl)
            mean2, rstd2 = self._buf(R, dtype=torch.float32), self._buf(R, dtype=torch.float32)
            L.ln_fwd(z2, slabs, self._v(p + "ln2_g"), self._v(p + "ln2_b"), mean2, rstd2, R, D, DP,
                     y_off=cur_off[l + 1])
            if save_for_backward:
                sv.q, sv.kv, sv.kv_off, sv.r, sv.att, sv.lse = q, kv, kv_off, r, att, lse
                sv.z1, sv.a, sv.mean1, sv.rstd1 = z1, a, mean1, rstd1
                sv.h, sv.z2, sv.mean2, sv.rstd2 = h, z2, mean2, rstd2
                ctx.layers.append(sv)
        if use_cache:
            st = ring.kv
            st["lo"] = st["lo"] if kv_from == w and M > 0 else ctx.x_segs[0][0]
            st["hi"], st["tag"] = w + Q, self.pack_epoch
        if keep_kv:
            ctx.kv_rows = (ring.kv["buf"], C * B * 2 * NH) if use_cache else (kv_all, KR * 2 * NH)
        # 3. final dropout, logits, NLL
        T = Q if n_pred is None else n_pred
        ctx.T = T
        RT = T * B
        hid_off = cur_off[d.n_layer] + (Q - T) * B * DP
        if p_drop > 0:
            hidden = self._buf(RT, DP)
            L.dropout(slabs, hidden, RT, DP, DP, DP, p_drop, seed, self._site(cid, 2), src_off=hid_off)
            hid_t, hid_o = hidden, 0
        else:
            hid_t, hid_o = slabs, hid_off
        ctx.hid_t, ctx.hid_o = hid_t, hid_o
        eoff, eld = self._m("E")
        logits = self._buf(RT, VP, dtype=torch.float32)
        L.gemm(hid_t, self.pmat, logits, M=RT, N=d.n_token, K=DP, lda=DP, ldb=eld, a_off=hid_o, b_off=eoff,
               bias=self._v("bias_out"), flags=L.EPI_BIAS, impl=self.impl)
        ctx.logits = logits
        ctx.nll = None
        if target is not None:
            tgt = target.to(self.device).contiguous().view(-1)
            nll = self._buf(RT, dtype=torch.float32)
            lse_ce = self._buf(RT, dtype=torch.float32)
            L.ce_fwd(logits, tgt, nll, lse_ce, RT, d.n_token)
            ctx.target, ctx.nll, ctx.lse_ce = tgt, nll, lse_ce
        # 4. memory update: the layer inputs already sit in the ring; only the window moves
        if mem_len > 0:
            new_len = min(M + Q, mem_len)
            new_start = (ring.start + M + Q - new_len) % C
            ctx.new_mems = RingMems(ring.slabs, new_start, new_len, D, kv=ring.kv, shared=ring.shared,
                                    key_start=ring.key_start, pos0=ring.pos0 + M + Q - new_len)
        else:
            ctx.new_mems = None
        return ctx

    # -- backward -----------------------------------------------------------------------------------------
    def backward(self, ctx: _Ctx, dnll: Optional[torch.Tensor] = None, dlogits32: Optional[torch.Tensor] = None,
                 need_dinput: bool = False, grad_targets: Optional[Dict[str, torch.Tensor]] = None,
                 accumulate: bool = True, reducer=None) -> Dict[str, torch.Tensor]:
        """Gradients (reference layout, fp32) of sum(nll * dnll) [+ sum(logits * dlogits32)] w.r.t. every
        generator parameter.  With ``grad_targets`` ({state_dict name: fp32 tensor}, e.g. the parameters' ``.grad``)
        the gradients are ACCUMULATED into (``accumulate=False``: written to) those tensors by one kernel (no per-tensor
        allocation, no autograd accumulate nodes); otherwise fresh tensors are returned.  With need_dinput the gradient w.r.t. the soft
        one-hot input rows is returned under the key '__dinput__' (fp32 [Q*B, VP]).
        ``reducer`` (tgan_b200.dp.BucketReducer): data-parallel runs all-reduce each layer's padded gradient block on a
        side stream as soon as that layer's backward has been enqueued (last layer first), overlapping the exchange with
        the layers below; the shared tensors (embedding, r_net, biases) follow at the end, before the unpack."""
        d, lay, dt = self.d, self.layout, self.dtype
        DP, NH, DIP, VP, D = d.DP, d.NH, d.DIP, d.VP, d.d_model
        Q, B, M, K, cid = ctx.Q, ctx.B, ctx.M, ctx.K, ctx.cid
        R, KR, T = Q * B, K * B, ctx.T
        RT = T * B
        seed, p_drop, p_att = self.seed, ctx.p_drop, ctx.p_att
        slabs = ctx.ring.slabs
        slab_elems = ctx.ring.capacity * B * DP
        cur_off = ctx.cur_off
        impl = self.impl
        gm, gv = self.gmat, self.gvec
        # every weight-gradient GEMM accumulates (TMA reduce-add / split-K partial sums) into buffers zeroed ONCE here:
        # one 60 MB memset instead of a memset node in front of each of the ~37 split-K launches
        if self._window is None:
            gv.zero_()
            gm.zero_()
        else:
            self._window += 1

        # small calls: weight-gradient GEMMs on the side stream (see side_stream_max_rows); their operands are kept
        # alive in `keep` until the join at the end -- the caching allocator would otherwise hand a freed block to the
        # next allocation on the main stream while the side stream still reads it
        side = self._side_stream() if (reducer is None and self._use_side_streams(R)) else None
        main = torch.cuda.current_stream()
        keep = []

        side2 = self._side_stream(1) if side is not None else None

        def wgrad(name, dY, X, rows, n_out, k_in, *, dy_off=0, x_off=0, ldy=None, ldx=None, row_off=0, stream=None):
            """gmat[name][row_off : row_off+n_out, :k_in] (+)= dY^T X"""
            goff, _, gld = lay.gmat[name]
            st = stream if stream is not None else side
            if st is not None:
                st.wait_stream(main)  # everything enqueued so far (the producers of dY, the zeroing of gm)
                keep.append((dY, X))
            with (torch.cuda.stream(st) if st is not None else contextlib.nullcontext()):
                L.gemm(dY, X, gm, transA=True, transB=False, M=n_out, N=k_in, K=rows, lda=ldy, ldb=ldx, ldc=gld,
                       a_off=dy_off, b_off=x_off, c_off=goff + row_off * gld, flags=L.EPI_ACCUM, impl=impl)

        # ---- loss head
        dl = self._buf(RT, VP)
        if dnll is not None:
            L.ce_bwd(ctx.logits, ctx.target, ctx.lse_ce, dnll.contiguous().view(-1).float(), dl, RT, d.n_token, VP)
            if dlogits32 is not None:
                raise L.TganError("either dnll or dlogits32")
        else:
            L.convert(dlogits32, dlogits32.stride(0), dl, VP, RT, d.n_token, VP)
        L.colsum(dl, gv, RT, d.n_token, ld=VP, out_off=lay.vec["bias_out"][0])
        wgrad("E", dl, ctx.hid_t, RT, VP, DP, ldy=VP, ldx=DP, x_off=ctx.hid_o)
        etoff, etld = self._m("E.T")
        dx = self._buf(R, DP)
        if T < Q:
            dx.zero_()
        dxo = (Q - T) * B * DP
        L.gemm(dl, self.pmat, dx, M=RT, N=DP, K=VP, lda=VP, ldb=etld, b_off=etoff, c_off=dxo, impl=impl)
        if p_drop > 0:
            L.dropout(dx, dx, RT, DP, DP, DP, p_drop, seed, self._site(cid, 2), src_off=dxo, dst_off=dxo)
        scale = 1.0 / math.sqrt(d.d_head)
        dr_all32 = self._buf(K, d.n_layer * NH, dtype=torch.float32)
        for l in reversed(range(d.n_layer)):
            p = f"l{l}."
            sv = ctx.layers[l]
            x_base = l * slab_elems
            # LN2 backward
            dz2, dz2d = self._buf(R, DP), (self._buf(R, DP) if p_drop > 0 else None)
            L.ln_bwd(dx, sv.z2, self._v(p + "ln2_g"), sv.mean2, sv.rstd2, dz2, dz2d, self._gv(p + "ln2_g"),
                     self._gv(p + "ln2_b"), R, D, DP, p_drop, seed, self._site(cid, 11 + 4 * l),
                     dsum=self._gv(p + "b2"))  # db2 = column sums of the gradient entering W2's output dropout
            g2 = dz2d if dz2d is not None else dz2
            wgrad(p + "W2", g2, sv.h, R, DP, DIP, ldy=DP, ldx=DIP)
            w2toff, w2tld = self._m(p + "W2.T")
            dh = self._buf(R, DIP)
            L.gemm(g2, self.pmat, dh, M=R, N=DIP, K=DP, ldb=w2tld, b_off=w2toff, aux=sv.h, ldaux=DIP,
                   flags=L.EPI_MASK_POS, alpha=1.0 / (1.0 - p_drop) if p_drop > 0 else 1.0, impl=impl)
            if DP == D:  # no pad lane for the ones column: separate pass for db1
                L.colsum(dh, gv, R, d.d_inner, ld=DIP, out_off=lay.vec[p + "b1"][0])
            wgrad(p + "W1", dh, sv.a, R, DIP, DP, ldy=DIP, ldx=DP)
            w1toff, w1tld = self._m(p + "W1.T")
            da = self._buf(R, DP)
            L.gemm(dh, self.pmat, da, M=R, N=DP, K=DIP, ldb=w1tld, b_off=w1toff, aux=dz2, ldaux=DP,
                   flags=L.EPI_ADD_AUX, impl=impl)
            # LN1 backward
            dz1, dz1d = self._buf(R, DP), (self._buf(R, DP) if p_drop > 0 else None)
            L.ln_bwd(da, sv.z1, self._v(p + "ln1_g"), sv.mean1, sv.rstd1, dz1, dz1d, self._gv(p + "ln1_g"),
                     self._gv(p + "ln1_b"), R, D, DP, p_drop, seed, self._site(cid, 9 + 4 * l))
            g1 = dz1d if dz1d is not None else dz1
            wgrad(p + "Wo", g1, sv.att, R, DP, NH, ldy=DP, ldx=NH)
            wotoff, wotld = self._m(p + "Wo.T")
            datt = self._buf(R, NH)
            L.gemm(g1, self.pmat, datt, M=R, N=NH, K=DP, ldb=wotld, b_off=wotoff, impl=impl)
            # attention core backward
            qp = sv.q.stride(0)  # the kernels address dq with q's row pitch (3 * NH for single-token calls)
            dq3 = self._buf(R, qp)
            dq = dq3[:, :NH]
            dkv = self._buf(KR, 2 * NH)
            dr32 = dr_all32[:, l * NH:(l + 1) * NH]  # view: this layer's column block
            split = side is not None and Q == 1  # single-token step: memory-side half on the second side stream
            # Q == 1: dS scratch [B, N, K]; split: + P~ [B, N, K] + the per-sequence r_w_bias / r_r_bias parts [2][B, NH]
            delta = self._buf(B * d.n_head * (Q if Q > 1 else (2 * K if split else K)) + (2 * B * NH if split else 0),
                              dtype=torch.float32)
            if split:
                head = (sv.q, sv.kv, sv.kv, 2 * NH, sv.r, self._v("u"), self._v("vb"), ctx.reset, sv.att, datt, sv.lse,
                        delta, dq)
                tail = (dr32, self._gv("u"), self._gv("vb"), B, d.n_head, M, ctx.msl, ctx.same_length, scale, p_att, seed,
                        self._site(cid, 8 + 4 * l))
                # query side: dk / dv of the current position (key row M) land in dq3[:, NH:3NH] -- the kernel addresses
                # key row j at dk + (j * B + b) * lddkv, so the base is shifted back by M rows of the 3 * NH pitch
                back = M * B * 3 * NH
                L.relattn_bwd_step(1, *head, dq3, dq3, 3 * NH, *tail, k_off=sv.kv_off, v_off=sv.kv_off + NH,
                                   dk_off=NH - back, dv_off=2 * NH - back)
                side2.wait_stream(main)
                with torch.cuda.stream(side2):  # memory side: rows j < M of dkv, dR, bias sums
                    L.relattn_bwd_step(2, *head, dkv, dkv, 2 * NH, *tail, k_off=sv.kv_off, v_off=sv.kv_off + NH, dv_off=NH)
                keep.append((delta, dq3, dkv, datt))
            else:
                L.relattn_bwd(sv.q, sv.kv, sv.kv, 2 * NH, sv.r, self._v("u"), self._v("vb"), ctx.reset, sv.att, datt,
                              sv.lse, delta, dq, dkv, dkv, 2 * NH, dr32, self._gv("u"), self._gv("vb"), B, d.n_head, Q, M,
                              ctx.msl, ctx.same_length, scale, p_att, seed, self._site(cid, 8 + 4 * l), impl=impl,
                              k_off=sv.kv_off, v_off=sv.kv_off + NH, dv_off=NH)
            wtoff, wtld = self._m(p + "Wqkv.T")
            if split:
                # [dq | dk | dv] of the current position: one weight-gradient GEMM for all of Wqkv ...
                wgrad(p + "Wqkv", dq3, slabs, R, 3 * NH, DP, ldy=3 * NH, ldx=DP, x_off=cur_off[l])
                row, left = 0, M  # ... the memory rows (behind the memory-side kernels on their stream) ...
                for pos, n in ctx.x_segs:
                    n = min(n, left)
                    if n > 0:
                        wgrad(p + "Wqkv", dkv, slabs, n * B, 2 * NH, DP, ldy=2 * NH, ldx=DP, dy_off=row * B * 2 * NH,
                              x_off=x_base + pos * B * DP, row_off=NH, stream=side2)
                    row, left = row + n, left - n
                # ... and one dgrad GEMM: dx_l = dz1 + [dq | dk | dv] Wqkv
                dx = self._buf(R, DP)
                L.gemm(dq3, self.pmat, dx, M=R, N=DP, K=3 * NH, ldb=wtld, b_off=wtoff, aux=dz1, ldaux=DP,
                       flags=L.EPI_ADD_AUX, impl=impl)
            else:
                wgrad(p + "Wqkv", dq3, slabs, R, NH, DP, ldy=qp, ldx=DP, x_off=cur_off[l])
                row = 0
                for pos, n in ctx.x_segs:
                    wgrad(p + "Wqkv", dkv, slabs, n * B, 2 * NH, DP, ldy=2 * NH, ldx=DP, dy_off=row * B * 2 * NH,
                          x_off=x_base + pos * B * DP, row_off=NH)
                    row += n
                # dx_l = dz1 + dq Wq + dkv[current rows] Wkv
                t = self._buf(R, DP)
                L.gemm(dq, self.pmat, t, M=R, N=DP, K=NH, ldb=wtld, b_off=wtoff, aux=dz1, ldaux=DP, flags=L.EPI_ADD_AUX,
                       impl=impl)
                dx = self._buf(R, DP)
                L.gemm(dkv, self.pmat, dx, M=R, N=DP, K=2 * NH, lda=2 * NH, ldb=wtld, a_off=M * B * 2 * NH,
                       b_off=wtoff + NH, aux=t, ldaux=DP, flags=L.EPI_ADD_AUX, impl=impl)
            if reducer is not None:  # this layer's weight / bias / LayerNorm gradients are final: exchange them now
                m0, m1 = lay.gmat[p + "Wqkv"][0], lay.gmat[p + "W2"][0] + lay.gmat[p + "W2"][1] * lay.gmat[p + "W2"][2]
                v0, v1 = lay.vec[p + "b1"][0], lay.vec[p + "ln2_b"][0] + lay.vec[p + "ln2_b"][1]
                reducer.reduce(gm, m0, m1 - m0)
                reducer.reduce(gv, v0, v1 - v0)
        # Late join (inside a gradient window, single-token calls): nothing the main stream does from here to the end of
        # the window needs the side streams' results -- the r_net weight gradient below moves to the memory-side stream,
        # where dR is produced -- so the join with THIS call's side work is deferred by one call (its buffers are kept
        # alive until then): the last layer's memory-side tail (~90 us) overlaps the head of the next token's backward
        # instead of idling the main stream.  end_grad_window() joins the last one.
        late = side is not None and self._window is not None and Q == 1
        if side is not None and not late:
            main.wait_stream(side)
            if Q == 1:  # (a stream that never forked from a capturing stream must not be joined into the capture)
                main.wait_stream(side2)
            keep.clear()
        # ---- r_net weight gradients of all layers: dWr_all = dR_all^T pos_emb
        NL = d.n_layer * NH
        if late:
            side2.wait_stream(main)
        with (torch.cuda.stream(side2) if late else contextlib.nullcontext()):
            if dt == torch.float32:
                dr_all = dr_all32
            else:
                dr_all = self._buf(K, NL)
                L.convert(dr_all32, NL, dr_all, NL, K, NL, NL)
            L.gemm(dr_all, ctx.pe, gm, transA=True, transB=False, M=NL, N=DP, K=K, lda=NL, ldb=DP, ldc=DP,
                   c_off=lay.gmat["l0.Wr"][0], flags=L.EPI_ACCUM, impl=impl)
        if late:
            keep.append((dr_all, dr_all32, ctx.pe, ctx.layers, ctx.soft))
            prev, self._late = self._late, (side.record_event(), side2.record_event(), keep)
            if prev is not None:
                main.wait_event(prev[0])
                main.wait_event(prev[1])
                prev[2].clear()
        # ---- embedding
        out: Dict[str, torch.Tensor] = {}
        goff, _, gld = lay.gmat["E"]
        if ctx.ids is not None:
            L.embed_bwd(ctx.ids, dx, gm[goff:], R, d.n_token, D, DP, math.sqrt(D), p_drop, seed, self._site(cid, 0))
        else:
            if p_drop > 0:
                L.dropout(dx, dx, R, DP, DP, DP, p_drop, seed, self._site(cid, 0))
            # dE[v, :] += sqrt(D) * soft^T dx ;  dsoft = sqrt(D) * dx E^T
            L.gemm(ctx.soft, dx, gm, transA=True, transB=False, M=VP, N=DP, K=R, lda=VP, ldb=DP, ldc=gld, c_off=goff,
                   alpha=math.sqrt(D), flags=L.EPI_ACCUM, impl=impl)
            if need_dinput:
                eoff, eld = self._m("E")
                dsoft = self._buf(R, VP, dtype=torch.float32)
                L.gemm(dx, self.pmat, dsoft, M=R, N=d.n_token, K=DP, ldb=eld, b_off=eoff, alpha=math.sqrt(D), impl=impl)
                out["__dinput__"] = dsoft
        if reducer is not None:  # shared tensors: embedding, r_net of every layer, r_w_bias / r_r_bias, output bias
            reducer.reduce(gm, 0, lay.gmat["l0.Wqkv"][0])
            reducer.reduce(gv, 0, lay.vec["l0.b1"][0])
            reducer.join()
        # ---- unpack to reference-layout gradients
        if self._window is not None:
            grads = {}  # end_grad_window() unpacks once for all the calls of the window
        elif grad_targets is not None:
            desc = self._unpack_desc_for(grad_targets)
            L.unpack_grads(gm, gv, desc, desc.shape[0], self._max_elems, accumulate=accumulate)
            grads = {}
        else:
            grads = {}
            rows = []
            for (ref, name, kind, *_), urow in zip(lay.reference_map(), self._unpack_rows):
                g = torch.empty(self._grad_shapes[ref], dtype=torch.float32, device=self.device)
                grads[ref] = g
                rows.append([g.data_ptr()] + urow[1:])
            desc = self._stage_desc(rows)
            L.unpack_grads(gm, gv, desc, len(rows), self._max_elems)
            out["__desc__"] = desc  # keep the descriptor table alive until the kernel ran
        ctx.layers = None  # release activations
        self._dirty = True  # an optimizer step may follow: the next forward re-packs (see pack)
        out.update(grads)
        return out

    def _stage_desc(self, rows) -> torch.Tensor:
        """Descriptor table -> device through pinned memory (an asynchronous copy: no host synchronisation).  The
        returned device tensor carries its pinned source (``_host``) so that whoever keeps the table alive -- the
        cache below, a captured graph's entry -- also keeps the copy's source alive."""
        host = torch.tensor(rows, dtype=torch.int64).pin_memory()
        dev = torch.empty_like(host, device=self.device)
        dev.copy_(host, non_blocking=True)
        dev._host = host
        self._desc_keepalive = getattr(self, "_desc_keepalive", [])[-7:] + [dev]
        return dev

    def _unpack_desc_for(self, targets: Dict[str, torch.Tensor]) -> torch.Tensor:
        """Cached unpack table whose destinations are the given gradient tensors, keyed by their addresses.  Captured
        graphs must additionally hold the returned tensor themselves (their kernels read it at every replay): the
        cache is bounded and evicts the oldest tables."""
        key = tuple(targets[ref].data_ptr() for ref, *_ in self.layout.reference_map())
        dev = self._unpack_cache.get(key)
        if dev is not None:
            return dev
        rows = []
        for (ref, name, kind, *_), urow in zip(self.layout.reference_map(), self._unpack_rows):
            t = targets[ref]
            if t.dtype != torch.float32 or not t.is_contiguous() or tuple(t.shape) != self._grad_shapes[ref]:
                raise L.TganError(f"gradient target for {ref} must be a contiguous fp32 tensor of the parameter's shape")
            rows.append([t.data_ptr()] + urow[1:])
        dev = self._stage_desc(rows)
        while len(self._unpack_cache) >= 16:
            self._unpack_cache.pop(next(iter(self._unpack_cache)))
        self._unpack_cache[key] = dev
        return dev
