"""Batched conditional generation from prompts of different lengths (generate_batched(prompt_lengths=...)) against the
two ways of running that workload without the key floor.

Real model (6 layers, 10 heads, d_model 500, d_inner 1000, vocab 310) in bf16, inference_unconditional.yml's
memory_length 4146, same_length, top-k 32, temperature 0.95; B = 128 prompts whose lengths are drawn (seeded) from
[1, 2048] and whose tokens are windows of a seeded token stream; 256 generated tokens.  Reports
  ragged:  the context pass (left-align + one forward over the longest prompt, pad rows masked by the key floor), the
           first token step (projects the K/V rows of the whole prompt block into the cache) and the steady token step;
  padded:  the same block padded to the longest prompt WITHOUT a floor (every sequence attends over the pad rows: the
           cost of an equal-length batch at the longest prompt, not a correct result);
  single:  8 of the prompts one at a time at B = 1 (the reference's speed class), ms per token step.
Times are CUDA events around host-enqueued work that ends in a synchronise, median of --reps repeats (each repeat
starts from a fresh context pass).  The card's name and power limit are read in the same run.

Usage: python tools/ragged_generate_bench.py [--reps 3] [--out FILE]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "transformer-gan_b200"))
import torch  # noqa: E402

import bench as BN  # noqa: E402

B, MEM_LEN, MAX_PROMPT, GEN, N_SINGLE = 128, 4146, 2048, 256, 8


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = (s.strip() for s in out[0].split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "torch_device": torch.cuda.get_device_name(0)}


def build(dev):
    import mem_transformer as MT
    ns = types.SimpleNamespace
    W = BN.WORK
    cfg = ns(MODEL=ns(num_layers=W["n_layer"], num_heads=W["n_head"], units=W["d_model"], inner_size=W["d_inner"],
                      dropout=0.1, attention_dropout=0.1, tie_embedding=True, tie_proj=False, pre_lnorm=False,
                      same_length=True, clamp_len=-1),
             TRAIN=ns(tgt_length=128, mem_length=MEM_LEN, pad_type="model", replace_start_with_pad=False,
                      append_note_status=False))
    torch.manual_seed(0)
    model = MT.MemTransformerLM(cfg, W["n_token"], 0)
    BN.init_like_train_py(model, 1111)
    model = model.to(dev).eval()
    model.compute_dtype = torch.bfloat16
    return model


def prompts(dev):
    """lengths in [1, MAX_PROMPT] and right-padded [MAX_PROMPT, B] prompts cut from one seeded token stream"""
    g = torch.Generator().manual_seed(2024)
    stream = torch.randint(2, BN.WORK["n_token"], (200_000,), generator=g)
    lens = torch.randint(1, MAX_PROMPT + 1, (B,), generator=g)
    lens[0] = MAX_PROMPT  # the block is as long as the longest prompt allows
    offs = torch.randint(0, stream.numel() - MAX_PROMPT, (B,), generator=g)
    start = torch.stack([stream[o:o + MAX_PROMPT] for o in offs.tolist()], 1)
    return start.to(dev), lens


class Timer:
    def __init__(self):
        self.e0, self.e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def __enter__(self):
        torch.cuda.synchronize()
        self.e0.record()
        return self

    def __exit__(self, *exc):
        self.e1.record()
        torch.cuda.synchronize()
        self.ms = self.e0.elapsed_time(self.e1)


def generate(model, start, lens, gen):
    """-> (context-pass ms, first-step ms, steady ms per step); lens None: no prompt_lengths (no floor)"""
    last = start[-1:] if lens is None else torch.stack([start[n - 1, b] for b, n in enumerate(lens.tolist())]).view(1, -1)
    with Timer() as t_ctx:
        _, mems = model.generate_batched(start, 0, prompt_lengths=lens)
    with Timer() as t_first:
        ids, mems = model.generate_batched(last, 1, mems=mems)
    with Timer() as t_steps:
        ids, mems = model.generate_batched(ids[-1:], gen - 1, mems=mems)
    del mems
    return t_ctx.ms, t_first.ms, t_steps.ms / (gen - 1)


def summary(runs):
    cols = list(zip(*runs))
    keys = ("context_pass_ms", "first_token_step_ms", "ms_per_token_step")
    return {k: {"median": statistics.median(c), "min": min(c), "max": max(c)} for k, c in zip(keys, cols)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--gen", type=int, default=GEN)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    model = build(dev)
    start, lens = prompts(dev)
    T = int(lens.max())
    # the same block left-aligned by hand: pad rows repeat each prompt's first token, as generate_batched does
    pad = (T - lens).to(dev)
    rows = torch.arange(T, device=dev).view(T, 1)
    padded = start.gather(0, (rows - pad).clamp(min=0))
    res = {"what": "generate_batched from prompts of different lengths (key floor) vs the same batch padded to the "
                   "longest prompt without a floor vs one prompt at a time",
           "card": card(), "batch": B, "memory_length": MEM_LEN, "generated_tokens": args.gen, "same_length": True,
           "prompt_lengths": {"min": int(lens.min()), "max": T, "mean": float(lens.float().mean()),
                              "real_tokens": int(lens.sum()), "block_tokens": T * B}}
    with torch.no_grad():
        generate(model, start, lens, 8)  # warm-up: every kernel, ring layout and allocation the timed runs use
        generate(model, padded, None, 8)
        generate(model, start[:int(lens[1]), 1:2].contiguous(), None, 8)
        ragged = [generate(model, start, lens, args.gen) for _ in range(args.reps)]
        flat = [generate(model, padded, None, args.gen) for _ in range(args.reps)]
        single = []
        for b in range(N_SINGLE):
            n = int(lens[b])
            _, _, ms = generate(model, start[:n, b:b + 1].contiguous(), None, args.gen)
            single.append({"prompt_length": n, "ms_per_token_step": ms})
    res["ragged"] = summary(ragged)
    res["padded_no_floor"] = summary(flat)
    res["single_prompt_b1"] = {"runs": single,
                               "ms_per_token_step_mean": statistics.mean(s["ms_per_token_step"] for s in single)}
    r, f = res["ragged"]["ms_per_token_step"]["median"], res["padded_no_floor"]["ms_per_token_step"]["median"]
    res["ragged_over_padded_token_step"] = r / f
    res["tokens_per_s"] = {"ragged": B / (r / 1e3),
                           "single_prompt_b1": 1.0 / (res["single_prompt_b1"]["ms_per_token_step_mean"] / 1e3)}
    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
