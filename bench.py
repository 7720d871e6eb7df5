#!/usr/bin/env python
"""bench.py -- train tokens/sec of the Transformer-XL + GAN training cycle (experiment_spanbert.yml shapes) on N B200s.

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA kernels through the C-ABI)
    python bench.py --impl reference --gpus N --steps K ...  # reference arm: the CPU implementation of the same cycle
    python bench.py ... --dump-outputs DIR                   # also write one iteration's outputs (dump_outputs)

BASELINE.json's metric is "train tokens/sec (GAN step)".  A "step" is one iteration of the reference's train loop
(train.py:859-1090) on synthetic MAESTRO-vocab tokens: an MLE optimizer step of MemTransformerLM over the global batch
(512 sequences x 128 tokens, memory 1024; forward + backward + gradient clip + Adam) and, on every 5th iteration
(DISCRIMINATOR.dis_loss_freq = gen_loss_freq = 5), one discriminator update (TransformerGAN.forward(..., "dis_loss"):
123 Gumbel-softmax sampling steps, BERT 5x768 discriminator on real / fake, WGAN-GP) and one generator update
("gen_loss": the same sampling chain with gradient, discriminator forward / backward to the samples).  Tokens counted
= the MLE target tokens, exactly what train.py logs (train.py:906, 1158-1163).  K should be a multiple of 5 (whole
cycles); the timed region starts on a cycle boundary.  `extras` (N = 1, own process): `mle_only` keeps round 1's headline
(the MLE step of experiment_baseline.yml alone), `gan_phases` the ms per adversarial update, `generate` BASELINE config 5
(batched generation against a full 4146-position memory with on-device sampling), `eager_gpu_bar` the reference's
algorithm run eagerly on the same GPU.

One process per GPU.  N > 1 is data parallel over sequences: every rank runs the configuration's batch (512 sequences
per GPU: WEAK scaling, global batch 512 x N; `--scaling strong` keeps the global batch at 512 and divides it as
train.py:226-227 does) on its own token stream (seed + 1000 x rank, train.py:224).  The only exchange is the gradient
all-reduce: the MLE gradients go bucket by bucket (one per layer, last layer first) through tgan_allreduce_bucket on a
side stream inside the backward (captured in its CUDA graph), the two adversarial updates all-reduce their flat
gradient buffer once.  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "transformer-gan_b200"))

import torch  # noqa: E402

# experiment_spanbert.yml / experiment_baseline.yml (model/training_config/*.yml): same generator and MLE shapes
WORK = dict(n_layer=6, n_head=10, d_model=500, d_inner=1000, n_token=310, tgt_len=128, mem_len=1024,
            global_batch=512, dropout=0.1, dropatt=0.1, clip=1.0, lr=0.002,
            dis_tgt_len=128, dis_mem_len=128, context_len=5, sample_chunks_mem=2, gan_freq=5)
BERT_CFG = dict(vocab_size=311, hidden_size=768, num_hidden_layers=5, num_attention_heads=12, intermediate_size=3072,
                max_position_embeddings=512, type_vocab_size=2, hidden_act="gelu", hidden_dropout_prob=0.1,
                attention_probs_dropout_prob=0.1, layer_norm_eps=1e-12, model_type="bert")
# where the "largest share of the timed cycle" claim of `roofline` comes from
ROOFLINE_NOTE = "profiles/r2_launch_summary_cycle.txt"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="gan", choices=["gan", "mle"],
                    help="gan: experiment_spanbert.yml cycle (the BASELINE metric); mle: experiment_baseline.yml MLE step only")
    ap.add_argument("--batch-chunk", type=int, default=1, help="micro-batches per step (reference yml: 16; native: 1)")
    ap.add_argument("--global-batch", type=int, default=WORK["global_batch"],
                    help="sequences per optimizer step: per GPU under weak scaling, in total under strong scaling")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--no-buckets", action="store_true", help="N > 1: one flat all-reduce after the backward instead of "
                    "per-layer buckets overlapped with it")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--kernel-impl", type=int, default=0, help="0 auto, 1 force SIMT, 2 force tcgen05")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the side measurements (phases, eager GPU bar)")
    ap.add_argument("--extras-only", action="store_true", help="(internal) run only the side measurements and print their JSON")
    ap.add_argument("--no-graphs", action="store_true", help="enqueue every kernel from the host instead of replaying "
                    "the captured CUDA graphs (MLE forward / backward per ring phase, one graph per adversarial phase)")
    ap.add_argument("--cpu-batch", type=int, default=4)
    ap.add_argument("--warm-segments", type=int, default=None,
                    help="untimed MLE steps before timing (default: enough to fill the recurrence memory + capture graphs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="one GPU: after the timed steps, run each phase of the iteration from a fixed state and "
                    "write what it computed (see dump_outputs) as DIR/<name>.npy")
    return ap.parse_args()


class Vocab:
    vec_len = 0

    def __len__(self):
        return WORK["n_token"]


def make_cfg(bert_dir, dis_batch_chunk=1):
    ns = types.SimpleNamespace
    return ns(MODEL=ns(num_layers=WORK["n_layer"], num_heads=WORK["n_head"], units=WORK["d_model"],
                       inner_size=WORK["d_inner"], dropout=WORK["dropout"], attention_dropout=WORK["dropatt"],
                       tie_embedding=True, tie_proj=False, pre_lnorm=False, same_length=False, clamp_len=-1),
              TRAIN=ns(tgt_length=WORK["tgt_len"], mem_length=WORK["mem_len"], pad_type="model",
                       replace_start_with_pad=False, append_note_status=False),
              DISCRIMINATOR=ns(type="bert" if bert_dir else "Null", tgt_len=WORK["dis_tgt_len"], mem_len=WORK["dis_mem_len"],
                               context_len=WORK["context_len"], sample_chunks_mem=WORK["sample_chunks_mem"],
                               truncate_backprop=False, backprop_outside=True, gen_loss_factor=1.0, dis_loss_factor=1.0,
                               batch_chunk=dis_batch_chunk,
                               BERT=ns(model_path=bert_dir, loss_type="wgan-gp", model_type="bert_lm", random_weights=False,
                                       freeze_layers=["0", "1", "2", "3", "4"]),
                               CNN=ns(embed_dim=64, hidden_dim=64, num_rep=64, init="uniform", loss_type="rsgan")),
              PPO=ns(dis_D_type="bert", dis_D_num_rep=1, clip_param=0.4))


def synth_bert_checkpoint(seed=0):
    """experiment_spanbert.yml points at ../BERT/checkpoint-1969000, which the reference does not ship: synthesize a
    seed-initialised BertForMaskedLM checkpoint of the same architecture so that the SHIPPED code path runs
    (random_weights False -> embeddings + all 5 layers frozen, pooler + classifier train; SURVEY 8c)."""
    from transformers import BertConfig, BertForMaskedLM
    d = tempfile.mkdtemp(prefix="tgan_bert_")
    torch.manual_seed(seed)
    cfg = BertConfig(**{k: v for k, v in BERT_CFG.items() if k != "model_type"})
    BertForMaskedLM(cfg).save_pretrained(d)
    return d


def init_like_train_py(model, seed):
    """train.py:291-371 with INITIALIZER base/embed 'normal' 0.01: weights N(0, .01), LN weight N(1, .01), biases 0."""
    g = torch.Generator().manual_seed(seed)
    for name, p in model.named_parameters():
        if name.endswith("layer_norm.weight"):
            p.data.copy_(1.0 + 0.01 * torch.randn(p.shape, generator=g))
        elif name.endswith("bias") and "r_" not in name:
            p.data.zero_()
        else:
            p.data.copy_(0.01 * torch.randn(p.shape, generator=g))


class ClockSampler:
    """SM clock / throttle reasons sampled every 50 ms DURING the timed region through NVML (in-process thread; an
    external ``nvidia-smi -lms`` loop was measured to slow the timed steps by 10-20 %)."""

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.sm, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[gpu_index]) if vis and vis.split(",")[gpu_index].isdigit() else gpu_index
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # noqa: BLE001
            self.nv, self.err = None, repr(e)

    def _loop(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001  (older NVML name)
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.05)

    def start(self):
        if self.nv is None:
            return
        self._thread = threading.Thread(target=self._loop, daemon=True)
        self._thread.start()

    def stop(self):
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + self.err]}
        self._stop.set()
        self._thread.join(timeout=2)
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return None


def workload_config(args, world):
    gan = args.workload == "gan"
    name = ("experiment_spanbert.yml Transformer-XL + GAN training cycle: every iteration an MLE optimizer step, every 5th "
            "iteration one discriminator update + one generator update (123 Gumbel-softmax sampling steps, BERT 5x768 "
            "discriminator, WGAN-GP)") if gan else "experiment_baseline.yml Transformer-XL MLE training step"
    per_gpu = args.global_batch if args.scaling == "weak" else args.global_batch // world
    return {"workload": name + " (6 layers, 10 heads, d_model 500, d_inner 1000, vocab 310, tgt_len 128, mem_len 1024, "
                        "dropout 0.1), synthetic MAESTRO-vocab tokens",
            "global_batch": per_gpu * world, "per_gpu_batch": per_gpu, "seq_len": WORK["tgt_len"], "mem_len": WORK["mem_len"],
            "all_reduce": None if world == 1 else ("one flat NCCL all-reduce per optimizer step" if args.no_buckets else
                          "MLE: 7 buckets (6 layers + shared tensors) via tgan_allreduce_bucket on a side stream inside "
                          "backward; dis / gen updates: one flat NCCL all-reduce each"),
            "batch_chunk": args.batch_chunk, "parallelism": f"dp{world}",
            "gan": {"dis_tgt_len": 128, "dis_mem_len": 128, "context_len": 5, "sample_chunks_mem": 2, "freq": 5,
                    "discriminator": "BERT 5x768, shipped trainable set (pooler + classifier), wgan-gp",
                    "dis_batch": per_gpu * world} if gan else None,
            "launch": "host launches" if args.no_graphs else
                      "CUDA graphs (MLE: one forward + one backward graph per ring phase; one graph per adversarial phase)",
            "l2": "per-step working set (activations + recurrence memory, several GB) is far larger than the 126 MB L2"}


# ---------------------------------------------------------------------------------------------------------
# CPU implementation of the same cycle: the oracle port of the reference path, all host threads
# ---------------------------------------------------------------------------------------------------------
def cpu_cycle_setup(batch, gan=True):
    """-> step(i): runs iteration i of the cycle on the CPU (fp32) at `batch` sequences, returns tokens consumed."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import txl_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    shape = O.TxlShape(n_layer=WORK["n_layer"], n_head=WORK["n_head"], d_model=WORK["d_model"],
                       d_inner=WORK["d_inner"], n_token=WORK["n_token"], mem_len=WORK["mem_len"])
    shape_gan = O.TxlShape(n_layer=WORK["n_layer"], n_head=WORK["n_head"], d_model=WORK["d_model"],
                           d_inner=WORK["d_inner"], n_token=WORK["n_token"], mem_len=WORK["dis_mem_len"])
    p = O.init_params(shape, 1111)
    for t in p.values():
        t.requires_grad_(True)
    g = torch.Generator().manual_seed(1111)
    Q, V = WORK["tgt_len"], WORK["n_token"]
    # steady-state shapes only need a full-size memory: start from a random one instead of running 8 segments
    state = {"mems": 0.1 * torch.randn(shape.n_layer + 1, WORK["mem_len"], batch, shape.d_model, generator=g)}
    disc = None
    if gan:
        from transformers import BertConfig, BertForSequenceClassification
        torch.manual_seed(0)
        cfg = BertConfig(**{k: v for k, v in BERT_CFG.items() if k != "model_type"})
        cfg._attn_implementation = "eager"
        bert = BertForSequenceClassification(cfg).train()
        for name, prm in bert.named_parameters():  # shipped trainable set (transformer_gan.py:568-585)
            prm.requires_grad_(not (name.startswith("bert.embeddings") or name.startswith("bert.encoder.layer")))
        E = bert.bert.embeddings.word_embeddings.weight
        on_emb = lambda e: bert(inputs_embeds=e)[0][:, 0]
        disc = (lambda x: on_emb(x @ E)), (lambda x: x @ E), on_emb

    def clear():
        for t in p.values():
            t.grad = None

    def step(i):
        data = torch.randint(2, V, (Q, batch), generator=g)
        target = torch.randint(2, V, (Q, batch), generator=g)
        loss, state["mems"] = O.mle_forward(data, target, torch.zeros(batch, dtype=torch.bool), state["mems"], p, shape)
        loss.mean().backward()
        clear()
        if gan and i % WORK["gan_freq"] == 0:
            T, ctx, ch = WORK["dis_tgt_len"], WORK["context_len"], WORK["sample_chunks_mem"]
            for mode in ("dis_loss", "gen_loss"):
                dis_data = torch.randint(2, V, (T, batch), generator=g)
                U = [torch.rand(1, batch, V, generator=g) for _ in range(T - ctx)]
                al = [torch.rand(batch, generator=g) for _ in range(ch)]
                O.gan_step(mode, dis_data, p, shape_gan, disc[0], 1, "wgan-gp", 1.0, U, al, T, ctx, ch,
                           embed=disc[1], disc_on_embeds=disc[2])
                clear()
        return Q * batch

    return step


def cpu_baseline(batch, gan, budget_s=25.0):
    step = cpu_cycle_setup(batch, gan)
    t0 = time.perf_counter()
    toks, n = 0, 0
    # whole cycles only (iteration 0 of each carries the GAN updates); stop after the first cycle past the budget
    while True:
        toks += step(n)
        n += 1
        if n % WORK["gan_freq"] == 0 and (time.perf_counter() - t0 >= budget_s or n >= 4 * WORK["gan_freq"]):
            break
    dt = time.perf_counter() - t0
    return {"value": toks / dt, "unit": "tokens/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"oracle/txl_oracle.py fp32 on the host: {n} iterations ({n // WORK['gan_freq']} whole cycle(s): "
                      f"MLE fwd+bwd each iteration, dis + gen update every 5th) at B={batch} sequences x Q=128 tokens, "
                      f"M=1024 (same model / shapes as the GPU workload, reduced batch)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    gan = args.workload == "gan"
    step = cpu_cycle_setup(args.cpu_batch, gan)
    for w in range(args.warmup):  # warm-up: MLE iterations (the GAN updates run inside the timed region from iteration 0)
        step(1)
    t0 = time.perf_counter()
    toks = 0
    for i in range(args.steps):
        toks += step(i)
    dt = time.perf_counter() - t0
    v = toks / dt
    cores = torch.get_num_threads()
    sample = (f"each step = one iteration of the cycle on the oracle port (fp32, {cores} threads) at B={args.cpu_batch} x "
              f"Q=128 tokens, M=1024; iterations 0, 5, ... carry the dis + gen updates (123 sampling steps, HF BERT 5x768, "
              f"WGAN-GP): a bounded sample of the 512-sequence step")
    print(json.dumps({
        "impl": "reference", "metric": "train tokens/sec (GAN step)" if gan else "train tokens/sec", "value": v,
        "unit": "tokens/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, max(1, int(os.environ.get("WORLD_SIZE", "1")))),
        "cpu_baseline": {"value": v, "unit": "tokens/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# ---------------------------------------------------------------------------------------------------------
# the GPU workload
# ---------------------------------------------------------------------------------------------------------
class Cycle:
    """The train.py iteration on this rank's shard: MLE step every call, dis + gen update every 5th."""

    def __init__(self, args, dev, world, rank):
        import transformer_gan as TG
        from tgan_b200 import dp
        from tgan_b200 import lib as L
        self.L, self.dp, self.args, self.dev, self.world = L, dp, args, dev, world
        self.gan = args.workload == "gan"
        Q, V = WORK["tgt_len"], WORK["n_token"]
        self.B = args.global_batch if args.scaling == "weak" else args.global_batch // world   # sequences on this rank
        self.n_chunks = args.batch_chunk
        self.Bc = self.B // self.n_chunks
        bert_dir = synth_bert_checkpoint() if self.gan else None
        torch.manual_seed(0)
        model = TG.TransformerGAN(make_cfg(bert_dir), Vocab())
        init_like_train_py(model.generator, 1111)
        model = model.to(dev).train()
        gen = model.generator
        gen.compute_dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float32
        gen.kernel_impl = args.kernel_impl
        gen.use_cuda_graphs = not args.no_graphs
        model.use_cuda_graphs = not args.no_graphs
        model.temperature = 1.0
        self.model, self.generator = model, gen
        # one flat parameter / gradient buffer per optimizer group: all-reduce, clip and Adam are one call each
        self.fp = dp.FlatParams(gen.parameters())
        lr = WORK["lr"] / world  # train.py:392 divides lr by the GPU count
        self.reducer = None
        if world > 1 and not args.no_buckets:
            self.reducer = gen.grad_reducer = dp.BucketReducer(world, rank, dev)
        self.opt = dp.FusedClipAdam(self.fp, lr, clip=WORK["clip"], world=world,       # `optimizer` (MLE)
                                    reduce=self.reducer is None)
        self.gen_opt = dp.FusedClipAdam(self.fp, lr, clip=WORK["clip"], world=world)   # `gen_optimizer` (train.py:1085-1090)
        self.dis_opt = self.dfp = None
        if self.gan:
            d = model.discriminator
            trainable = []
            for i, prm in enumerate(d.parameters()):  # train.py:944-947 toggles exactly these
                prm.requires_grad_(i in d.unfreeze_idx)
                if i in d.unfreeze_idx:
                    trainable.append(prm)
            self.dfp = dp.FlatParams(trainable)
            self.dis_opt = dp.FusedClipAdam(self.dfp, lr, clip=WORK["clip"], world=world)
        # --dump-outputs: the seeded initial parameters, the state dump_outputs() starts from
        self.initial = None
        if args.dump_outputs:
            self.initial = [fp.flat.clone() for fp in (self.fp, self.dfp) if fp is not None]
        g = torch.Generator().manual_seed(dp.rank_seed(1111, rank))  # train.py:224
        pin = lambda t: t.pin_memory()
        nbuf = 4 * self.n_chunks
        self.host_data = [pin(torch.randint(2, V, (Q, self.Bc), generator=g)) for _ in range(nbuf)]
        self.host_tgt = [pin(torch.randint(2, V, (Q, self.Bc), generator=g)) for _ in range(nbuf)]
        self.host_dis = [pin(torch.randint(2, V, (WORK["dis_tgt_len"], self.B), generator=g)) for _ in range(4)]
        self.dev_data = [t.to(dev) for t in self.host_data]
        self.dev_tgt = [t.to(dev) for t in self.host_tgt]
        self.dev_dis = [t.to(dev) for t in self.host_dis]
        self.reset = torch.zeros(self.Bc, dtype=torch.bool, device=dev)
        self.mems = [None] * self.n_chunks
        self.loss_host = torch.zeros(3).pin_memory()
        self.it = 0
        self.h2d = self.d2h = 0

    def mle_step(self, e2e):
        model, nck = self.model, self.n_chunks
        total = None
        for c in range(nck):
            i = (self.it * nck + c) % len(self.host_data)
            if e2e:
                data = self.host_data[i].to(self.dev, non_blocking=True)
                tgt = self.host_tgt[i].to(self.dev, non_blocking=True)
                self.h2d += 2 * data.numel() * 8
            else:
                data, tgt = self.dev_data[i], self.dev_tgt[i]
            ret = model(data, tgt, self.reset, "mle", self.mems[c])
            loss, self.mems[c] = ret["mle"], ret["mems"]
            l = loss.mean() / nck  # train.py:891-892 (no pad tokens in the synthetic stream)
            l.backward()
            total = l.detach() if total is None else total + l.detach()
        self.opt.step()  # one NCCL all-reduce of the flat gradient per optimizer step, then fused clip + Adam
        if e2e:
            self.loss_host[0:1].copy_(total.view(1), non_blocking=True)
            self.d2h += 4
        return total

    def gan_updates(self, e2e):
        model = self.model
        k = (self.it // WORK["gan_freq"]) % 2
        for j, (phase, opt) in enumerate((("dis_loss", self.dis_opt), ("gen_loss", self.gen_opt))):
            if e2e:
                dis_data = self.host_dis[2 * k + j].to(self.dev, non_blocking=True)
                self.h2d += dis_data.numel() * 8
            else:
                dis_data = self.dev_dis[2 * k + j]
            ret = model(dis_data, None, None, phase)  # backward runs inside (backprop_outside, transformer_gan.py:487-502)
            opt.step()
            # neither phase may leave gradients in the other model's buffers (train.py zero_grads both optimizers)
            self.fp.zero_grad()
            self.dfp.zero_grad()
            if e2e:
                self.loss_host[1 + j:2 + j].copy_(ret[phase].detach().float().view(1), non_blocking=True)
                self.d2h += 4

    def iteration(self, e2e=False):
        self.mle_step(e2e)
        if self.gan and self.it % WORK["gan_freq"] == 0:
            self.gan_updates(e2e)
        self.it += 1


def dump_outputs(cyc, out_dir, max_elems=1 << 20):
    """Each phase of the timed iteration -- MLE step, discriminator update, generator update: forward + backward
    through the same captured CUDA graphs, then the phase's fused clip + Adam step -- run from a state that is the same
    in every run, written as float32 ``out_dir/<name>.npy``: ``mle_loss`` (per-token NLL [tgt_len, B]), ``mems`` (the
    recurrence memory [n_layer+1, mem_len, B, d_model] it returns, flattened, batch chunks one after another),
    ``dis_loss``, ``gp_loss``, ``gen_loss``, and per phase ``<mle|dis|gen>_grad`` (the gradient of the parameters the
    phase's optimizer updates) and ``<mle|dis|gen>_update`` (parameters after the optimizer step minus before).  An
    array of more than max_elems entries is written as a sample of its flat entries drawn from a fixed seed; at the
    default workload the files come to about 27 MB.

    The state: the seeded initial parameters, zero gradients, fresh optimizer moments, and a recurrence memory of
    seeded N(0, 1) rows in the ring the timed steps left (same ring phase, so the captured graphs replay); it is
    restored before every phase.  Not the state the timed steps leave: the fp32 gradient reductions are atomics, so
    every step differs between runs in the last bits, and the ~50 optimizer steps and Gumbel sampling before the dump
    grow that into a different trajectory.  From the fixed state only the phase's own reductions differ between runs.
    The first Adam step moves a parameter by about lr * sign(gradient), so an entry whose gradient is at rounding level
    can move by +-lr in one run and -+lr in the other.  profiles/dump_outputs_repeatability.txt compares two runs."""
    import numpy as np
    from tgan_b200.engine import notify_params_updated
    inits = list(zip((cyc.fp, cyc.dfp), cyc.initial))

    def restore():
        for fp, init in inits:
            fp.flat.copy_(init)
            fp.zero_grad()
        notify_params_updated()

    arrays = {}

    def optimizer_step(name, opt, init):
        arrays[name + "_grad"] = opt.fp.grad.clone()
        opt.m.zero_()
        opt.v.zero_()
        opt.steps = 0
        opt.step()
        arrays[name + "_update"] = opt.fp.flat - init
        restore()

    restore()
    rng = torch.Generator(device=cyc.dev).manual_seed(1111)
    d = WORK["d_model"]
    for m in cyc.mems:
        m.slabs[..., :d].normal_(0.0, 1.0, generator=rng)
        m.slabs[..., d:].zero_()
    losses = []
    for c in range(cyc.n_chunks):  # Cycle.mle_step at iteration 0
        ret = cyc.model(cyc.dev_data[c], cyc.dev_tgt[c], cyc.reset, "mle", cyc.mems[c])
        losses.append(ret["mle"].detach())
        cyc.mems[c] = ret["mems"]
        (ret["mle"].mean() / cyc.n_chunks).backward()
    arrays["mle_loss"] = torch.cat(losses, 1)
    optimizer_step("mle", cyc.opt, cyc.initial[0])
    if cyc.gan:  # Cycle.gan_updates at iteration 0
        for j, (phase, opt, init) in enumerate((("dis_loss", cyc.dis_opt, cyc.initial[1]),
                                                ("gen_loss", cyc.gen_opt, cyc.initial[0]))):
            ret = cyc.model(cyc.dev_dis[j], None, None, phase)
            arrays.update((k, v) for k, v in ret.items() if k in (phase, "gp_loss") and v is not None)
            optimizer_step(phase[:3], opt, init)
    torch.cuda.synchronize()
    g = torch.Generator().manual_seed(0)

    def sample(t, n=max_elems):
        if t.numel() <= n:
            return t
        idx = torch.randint(0, t.numel(), (n,), generator=g).sort().values
        return t.reshape(-1)[idx.to(t.device)]

    # the memory materializes as fp32 (7.3 GB per chunk at the default workload): sample it chunk by chunk
    arrays["mems"] = torch.cat([sample(m.materialize(), max_elems // len(cyc.mems)).reshape(-1) for m in cyc.mems])
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), sample(t.detach()).float().cpu().numpy())


def attention_roofline(dev, B, pk):
    """Live CUDA-event timing of the kernel with the largest share of the timed cycle -- the fused relative-position
    attention BACKWARD at the MLE step's shape (B sequences x 10 heads, Q = 128, K = 1152, dropout 0.1) -- and of the
    forward; algorithmic FLOPs = SURVEY 8d's 3 * 2 * B * N * Q * K * d_head per pass, backward = 2x forward."""
    from tgan_b200 import lib as L
    N, Q, M, dh, HS = WORK["n_head"], WORK["tgt_len"], WORK["mem_len"], WORK["d_model"] // WORK["n_head"], 64
    K, NH = Q + M, N * HS
    g = torch.Generator().manual_seed(0)

    def mk(rows):
        x = torch.zeros(rows, N, HS)
        x[..., :dh] = torch.randn(rows, N, dh, generator=g)
        return x.reshape(rows, NH).to(dev).bfloat16()
    q, do, r = mk(Q * B), mk(Q * B), mk(K)
    kv = torch.cat([mk(K * B), mk(K * B)], 1).contiguous()
    u, vb = torch.zeros(NH, device=dev), torch.zeros(NH, device=dev)
    out = torch.empty(Q * B, NH, device=dev, dtype=torch.bfloat16)
    lse = torch.empty(B * N * Q, device=dev)
    dq, dkv = torch.empty_like(q), torch.empty_like(kv)
    dr = torch.empty(K, NH, device=dev)
    du, dvb = torch.zeros(NH, device=dev), torch.zeros(NH, device=dev)
    delta = torch.empty(B * N * Q, device=dev)
    scale = 1 / math.sqrt(dh)

    def fwd():
        L.relattn_fwd(q, kv, kv, 2 * NH, r, u, vb, None, out, lse, B, N, Q, M, Q, False, scale, 0.1, 1, 2, impl=2, v_off=NH)

    def bwd():
        L.relattn_bwd(q, kv, kv, 2 * NH, r, u, vb, None, out, do, lse, delta, dq, dkv, dkv, 2 * NH, dr, du, dvb, B, N, Q,
                      M, Q, False, scale, 0.1, 1, 2, impl=2, v_off=NH, dv_off=NH)
    res = {}
    for name, fn, mult in (("fwd", fwd, 1.0), ("bwd", bwd, 2.0)):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        t = e0.elapsed_time(e1) / reps / 1e3
        flops = mult * 3 * 2.0 * B * N * Q * K * dh
        res[name] = (t, flops)
    peak = (pk or {}).get("bf16_tflops", 1590.0)
    src = "MEASURED_PEAKS.json bf16_tflops (burst, kernel timed alone)" if pk else "fallback 1.59 PFLOP/s"

    def entry(name, kernel, traffic_key):
        t, flops = res[name]
        traffic = None
        try:
            for e in json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_full_summary.json"))):
                if traffic_key in e["kernel"]:
                    traffic = e["dram_bytes_total"] * B / float(e.get("batch", 512))
        except Exception:  # noqa: BLE001
            pass
        return {"bound": "tensor", "kernel": kernel, "achieved": flops / t / 1e12, "peak": peak, "unit": "TFLOP/s",
                "frac": flops / t / 1e12 / peak, "traffic": traffic, "algorithmic_flops_per_launch": flops,
                "us_per_launch": t * 1e6, "peak_source": src, "share_source": ROOFLINE_NOTE,
                "shape": f"B={B} N=10 Q=128 K=1152 d_head=50 (padded 64), attention dropout 0.1; L2-cold (K/V of one "
                         f"launch = {2 * K * B * NH * 2 / 1e6:.0f} MB)"}
    return entry("bwd", "relattn_bwd_tc_kernel", "relattn_bwd"), entry("fwd", "relattn_fwd_tc_kernel", "relattn_fwd")


def time_calls(fn, reps):
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return sorted(ts)[len(ts) // 2]


def eager_gpu_bar(dev):
    """BASELINE.md 4.6 / SURVEY 2a: the same modules run EAGER on the B200 (library kernels: ATen / cuBLAS) -- the
    oracle port executes unchanged on CUDA tensors.  MLE fwd+bwd at B = 32 (the oracle materialises the [B, N, Q, K]
    score tensors in fp32 like the reference does), TF32 matmuls and bf16 autocast."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import txl_oracle as O
    shape = O.TxlShape(n_layer=WORK["n_layer"], n_head=WORK["n_head"], d_model=WORK["d_model"],
                       d_inner=WORK["d_inner"], n_token=WORK["n_token"], mem_len=WORK["mem_len"])
    B, Q, V = 32, WORK["tgt_len"], WORK["n_token"]
    p = {k: v.to(dev).requires_grad_(True) for k, v in O.init_params(shape, 1111).items()}
    g = torch.Generator().manual_seed(1)
    mems = (0.1 * torch.randn(shape.n_layer + 1, WORK["mem_len"], B, shape.d_model, generator=g)).to(dev)
    data = torch.randint(2, V, (Q, B), generator=g).to(dev)
    target = torch.randint(2, V, (Q, B), generator=g).to(dev)
    reset = torch.zeros(B, dtype=torch.bool, device=dev)
    out = {"batch": B, "what": "oracle/txl_oracle.py (the reference's algorithm, eager torch) on cuda: MLE fwd+bwd, M=1024"}
    prev = torch.backends.cuda.matmul.allow_tf32

    def step():
        loss, _ = O.mle_forward(data, target, reset, mems, p, shape)
        loss.mean().backward()
        for t in p.values():
            t.grad = None
    try:
        torch.backends.cuda.matmul.allow_tf32 = True
        step()
        out["tf32_tokens_per_s"] = Q * B / (time_calls(step, 3) / 1e3)

        def step_bf16():
            with torch.autocast("cuda", dtype=torch.bfloat16):
                loss, _ = O.mle_forward(data, target, reset, mems, p, shape)
            loss.float().mean().backward()
            for t in p.values():
                t.grad = None
        step_bf16()
        out["bf16_autocast_tokens_per_s"] = Q * B / (time_calls(step_bf16, 3) / 1e3)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    return out


def generate_bar(dev, B=128, mem_len=4146, steps=48):
    """BASELINE config 5 (inference_unconditional.yml: memory_length = 4146, top-k 32, temperature 0.95) for B sequences
    at once through MemTransformerLM.generate_batched: single-token forward against the FULL memory (projected-K/V
    cache) + on-device sampling per step, no host synchronisation inside the loop.  The memory is filled by running the
    loop itself over mem_len positions' worth of context first (fed as 128-token segments)."""
    import mem_transformer as MT
    ns = types.SimpleNamespace
    cfg = ns(MODEL=ns(num_layers=WORK["n_layer"], num_heads=WORK["n_head"], units=WORK["d_model"],
                      inner_size=WORK["d_inner"], dropout=0.1, attention_dropout=0.1, tie_embedding=True, tie_proj=False,
                      pre_lnorm=False, same_length=True, clamp_len=-1),
             TRAIN=ns(tgt_length=128, mem_length=mem_len, pad_type="model", replace_start_with_pad=False,
                      append_note_status=False))
    torch.manual_seed(0)
    model = MT.MemTransformerLM(cfg, WORK["n_token"], 0)
    init_like_train_py(model, 1111)
    model = model.to(dev).eval()
    model.compute_dtype = torch.bfloat16
    model.reset_length(1, mem_len)
    g = torch.Generator().manual_seed(3)
    mems = None
    with torch.no_grad():
        for _ in range((mem_len + 127) // 128):  # context: fills the memory
            _, mems = model.forward_generate(torch.randint(2, WORK["n_token"], (128, B), generator=g).to(dev), mems)
        start = torch.randint(2, WORK["n_token"], (1, B), generator=g).to(dev)
        ids, mems = model.generate_batched(start, 8, mems=mems)  # warm-up (ring re-layout for single-token calls)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        ids, mems = model.generate_batched(ids[-1:], steps, mems=mems)
        e1.record()
        host_ms = (time.perf_counter() - t0) * 1e3 / steps
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    K = mem_len + 1
    kv_bytes = 2.0 * K * B * WORK["n_head"] * 64 * 2 * WORK["n_layer"]
    hbm = (peaks() or {}).get("hbm_gbs", 6555.2)
    return {"what": "inference_unconditional.yml: batched generation, top-k 32, temperature 0.95, on-device sampling",
            "batch": B, "memory_length": mem_len, "ms_per_token_step": ms, "host_enqueue_ms_per_step": host_ms,
            "tokens_per_s": B / (ms / 1e3), "kv_stream_bytes_per_step": kv_bytes,
            "hbm_frac_of_kv_stream": kv_bytes / (ms / 1e3) / 1e9 / hbm,
            "distinct_ids_in_last_step": int(ids[-1].unique().numel())}


def run_extras_only(args):
    """Side measurements in their own process: a failure there can never take the headline line with it."""
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    extras = {}
    cyc = Cycle(args, dev, 1, 0)
    fill = WORK["mem_len"] // WORK["tgt_len"]
    phases = 0 if args.no_graphs else (WORK["mem_len"] + WORK["tgt_len"]) // WORK["tgt_len"]
    try:
        for _ in range(fill + phases + 2):
            cyc.mle_step(False)
        ms = time_calls(lambda: [cyc.mle_step(False) for _ in range(5)], 3) / 5
        toks = WORK["tgt_len"] * args.global_batch
        extras["mle_only"] = {"ms_per_step": ms, "tokens_per_s": toks / (ms / 1e3),
                              "step_tensor_frac_of_sustained_peak": 231.8e6 * toks / (ms / 1e3) /
                              ((peaks() or {}).get("bf16_tflops_sustained", 1400.0) * 1e12),
                              "what": "experiment_baseline.yml MLE step alone (round 1's headline), 231.8 MFLOP/token fwd+bwd"}
        if cyc.gan:
            res = {}
            L = cyc.L
            for phase, opt in (("dis_loss", cyc.dis_opt), ("gen_loss", cyc.gen_opt)):
                def call():
                    cyc.model(cyc.dev_dis[0], None, None, phase)
                    opt.step()
                    cyc.fp.zero_grad()
                    cyc.dfp.zero_grad()
                for _ in range(3):
                    call()
                n0 = L.launch_count()
                res[phase + "_ms"] = time_calls(call, 3)
                res[phase + "_launches"] = (L.launch_count() - n0) // 3
            extras["gan_phases"] = res
    except Exception as e:  # noqa: BLE001
        extras["phases_error"] = repr(e)[:300]
    del cyc
    torch.cuda.empty_cache()
    for name, fn in (("generate", lambda: generate_bar(dev)), ("eager_gpu_bar", lambda: eager_gpu_bar(dev))):
        try:
            extras[name] = fn()
        except Exception as e:  # noqa: BLE001
            extras[name] = {"error": repr(e)[:300]}
    print(json.dumps(extras))


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    if args.extras_only:
        return run_extras_only(args)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        # the dumped phases replay the captured MLE backward, whose bucket all-reduces no other rank would join
        raise SystemExit("--dump-outputs runs on one GPU only (WORLD_SIZE=1)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from tgan_b200 import lib as L

    if (args.global_batch if args.scaling == "weak" else args.global_batch // world) % args.batch_chunk or \
            (args.scaling == "strong" and args.global_batch % world):
        raise SystemExit("batch must divide by gpus (strong scaling) and batch_chunk")
    Q = WORK["tgt_len"]
    cyc = Cycle(args, dev, world, rank)
    freq = WORK["gan_freq"]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(k, e2e):
        cyc.it = 0  # the timed region starts on a cycle boundary: iterations 0, 5, ... carry the GAN updates
        cyc.h2d = cyc.d2h = 0
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = L.launch_count()
        e0.record()
        for _ in range(k):
            cyc.iteration(e2e)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), L.launch_count() - l0

    # Untimed: what the workload needs before it is in steady state -- 8 MLE segments to fill the 1024-position
    # recurrence memory, one pass over the 9 ring phases so that every phase's CUDA graphs exist, the eager +
    # capturing calls of both adversarial phases -- then the --warmup W iterations the contract asks for.
    fill = WORK["mem_len"] // Q
    phases = 0 if args.no_graphs else (WORK["mem_len"] + Q) // Q
    warm_segments = args.warm_segments if args.warm_segments is not None else fill + phases + 1
    for _ in range(warm_segments):
        cyc.mle_step(False)
    if cyc.gan:
        for _ in range(3):
            cyc.gan_updates(False)
    cyc.it = 0
    for _ in range(args.warmup):
        cyc.iteration(False)
    untimed = warm_segments + args.warmup
    sampler = ClockSampler(local)
    sampler.start()
    ms_dev, launches = timed(args.steps, False)
    clocks = sampler.stop()
    ms_e2e, _ = timed(args.steps, True)
    h2d, d2h = cyc.h2d / args.steps, cyc.d2h / args.steps
    torch.cuda.synchronize()
    final_loss = [float(x) for x in cyc.loss_host]
    if args.dump_outputs:
        dump_outputs(cyc, args.dump_outputs)
    global_batch = args.global_batch * world if args.scaling == "weak" else args.global_batch
    tokens = Q * global_batch * args.steps
    value = tokens / (ms_dev / 1e3)
    e2e_value = tokens / (ms_e2e / 1e3)
    gan_updates = len([i for i in range(args.steps) if i % freq == 0]) if cyc.gan else 0
    B_rank = cyc.B
    del cyc
    torch.cuda.empty_cache()

    roof = roof2 = None
    if rank == 0:
        try:
            roof, roof2 = attention_roofline(dev, B_rank, peaks())
        except Exception as e:  # noqa: BLE001
            roof = {"error": repr(e)[:200]}
    extras = None
    if rank == 0 and world == 1 and not args.no_extras and args.dtype == "bf16":
        cmd = [sys.executable, os.path.abspath(__file__), "--extras-only", "--global-batch", str(args.global_batch),
               "--workload", args.workload] + (["--no-graphs"] if args.no_graphs else [])
        env = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", str(local)))
        for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
            env.pop(k, None)
        try:
            out = subprocess.run(cmd, capture_output=True, text=True, timeout=420, env=env)
            extras = json.loads(out.stdout.strip().splitlines()[-1])
        except Exception as e:  # noqa: BLE001  (side measurement: never lose the headline line)
            extras = {"error": repr(e)[:200]}
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(args.cpu_batch, args.workload == "gan")
    if rank == 0:
        print(json.dumps({
            "metric": "train tokens/sec (GAN step)" if args.workload == "gan" else "train tokens/sec",
            "value": value, "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "untimed_steps": untimed, "ms_per_step": ms_dev / args.steps,
            "gan_updates_in_timed_region": {"dis": gan_updates, "gen": gan_updates},
            "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
            "config": workload_config(args, world), "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "tokens/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "final_losses_mle_dis_gen": final_loss},
            "gpu_launches": launches,
            "roofline": roof, "roofline_secondary": roof2, "cpu_baseline": cpu, "extras": extras}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
