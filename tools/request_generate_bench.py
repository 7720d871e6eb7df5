"""Generation from a request queue (generate_requests: a finished column takes the next request at the following step),
with prompts fed one token per step and with one context pass per group of B prompts (context_pass=True), against
fixed batches of the same queue (generate_batched(prompt_lengths=...) over consecutive groups of B requests, each
group run to its longest gen_len).

Real model (6 layers, 10 heads, d_model 500, d_inner 1000, vocab 310) in bf16, inference_unconditional.yml's
memory_length 4146, same_length, top-k 32, temperature 0.95; B = 128 columns; 512 requests from a fixed seed with
prompt lengths uniform in [1, 256] (windows of a seeded token stream) and gen_len uniform in [128, 1024].
The three paths alternate in one process.  Reports per path: generated (kept) tokens per second over the whole run (CUDA
events around it, synchronise at the end, median of --reps), token steps, the share of column-steps that produced a
kept token, host time per step (the call's enqueue time before the closing synchronise) and the peak of
torch.cuda.max_memory_allocated over its runs.  For the context-pass path also: the size of one group's prefill ring and
K/V rows, and the device time of one group's prefill pass and of one group's row copies (tgan_ring_scatter) by
themselves (CUDA events, median of 5).  The card's name and power limit are read in the same run.

Usage: python tools/request_generate_bench.py [--reps 2] [--out FILE]"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402

from ragged_generate_bench import build, card  # noqa: E402

B, N_REQ, MAX_PROMPT, GEN_LO, GEN_HI = 128, 512, 256, 128, 1024


def queue():
    g = torch.Generator().manual_seed(2025)
    stream = torch.randint(2, 310, (200_000,), generator=g)
    lens = torch.randint(1, MAX_PROMPT + 1, (N_REQ,), generator=g).tolist()
    gens = torch.randint(GEN_LO, GEN_HI + 1, (N_REQ,), generator=g).tolist()
    offs = torch.randint(0, stream.numel() - MAX_PROMPT, (N_REQ,), generator=g).tolist()
    return [stream[o:o + n].clone() for o, n in zip(offs, lens)], gens


def timed(fn):
    """-> (device ms, host ms until the call returned)"""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    h0 = time.perf_counter()
    fn()
    h1 = time.perf_counter()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), (h1 - h0) * 1e3


def prefill_parts(model, sch):
    """Group 0's prefill pass and its row copies into a fresh queue ring, each timed by itself."""
    eng = model._get_engine()
    dev = eng.device
    pl = sch.prefill
    blk, pad = pl.blocks[0].to(dev), pl.pads[0].to(dev)
    desc = pl.desc.to(dev)
    (g, lo, n, mx), = pl.slices[0]
    ml = model.mem_len

    def one_pass():
        return model._prefill_pass(eng, blk, pad)

    def ev_ms(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), r

    pass_ms, copy_ms = [], []
    for _ in range(5):
        ms, pre = ev_ms(one_pass)
        pass_ms.append(ms)
        q = eng.new_queue_ring(sch.tables.shape[2], pl.lead, ml)
        torch.cuda.synchronize()
        ms, _ = ev_ms(lambda: eng.scatter_prefill(q, pre, desc, lo, n, mx, ml))
        copy_ms.append(ms)
        ring_bytes = pre.ring.slabs.numel() * pre.ring.slabs.element_size()
        kv, _ = pre.kv_rows
        kv_bytes = kv.numel() * kv.element_size()
        del pre, q
    d = eng.d
    rows = int(desc[lo:lo + n, 3].sum())
    copy_bytes = 2 * rows * ((d.n_layer + 1) * d.DP + d.n_layer * 2 * d.NH) * eng._es  # read + write
    return {"group_columns": blk.shape[1], "group_prompt_rows": blk.shape[0],
            "prefill_ring_GB": ring_bytes / 1e9, "prefill_kv_rows_GB": kv_bytes / 1e9,
            "pass_ms": statistics.median(pass_ms), "copy_descriptors": n, "copy_rows": rows,
            "copy_ms": statistics.median(copy_ms), "copy_GB_per_s": copy_bytes / (statistics.median(copy_ms) / 1e3) / 1e9}


def main():
    import mem_transformer as MT
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    model = build(dev)
    prompts, gens = queue()
    reqs = [MT.GenRequest(p, n, technique="topk", topk=32, temperature=0.95) for p, n in zip(prompts, gens)]
    kept = sum(gens)
    sch = MT.request_schedule([p.tolist() for p in prompts], gens, B)
    S_req = sch.tables.shape[1]
    sch_pre = MT.request_schedule([p.tolist() for p in prompts], gens, B, context_pass=True, mem_len=model.mem_len)
    S_pre = sch_pre.tables.shape[1]
    groups = []
    for i in range(0, N_REQ, B):
        ps, n = prompts[i:i + B], max(gens[i:i + B])
        T = max(len(p) for p in ps)
        start = torch.zeros(T, len(ps), dtype=torch.int64)
        for b, p in enumerate(ps):
            start[:len(p), b] = p
        groups.append((start.to(dev), [len(p) for p in ps], n))
    S_bat = sum(n for _, _, n in groups)

    def run_requests():
        model.generate_requests(reqs, B)

    def run_prefill():
        model.generate_requests(reqs, B, context_pass=True)

    def run_batched():
        for start, lens, n in groups:
            model.generate_batched(start, n, technique="topk", topk=32, temperature=0.95, prompt_lengths=lens)

    res = {"what": "generate_requests (one queue, a finished column takes the next request; prompts fed one token per "
                   "step, or context_pass=True: one context pass per group of 128 prompts and a row copy per "
                   "request) vs generate_batched over consecutive fixed groups of the same queue, each run to its "
                   "longest gen_len",
           "card": card(), "batch": B, "requests": N_REQ, "memory_length": 4146, "same_length": True,
           "dtype": "bf16", "sampling": "top-k 32, temperature 0.95",
           "prompt_length_range": [1, MAX_PROMPT], "gen_len_range": [GEN_LO, GEN_HI],
           "prompt_tokens": sum(len(p) for p in prompts), "generated_tokens": kept}
    with torch.no_grad():
        # warm-up: every kernel, allocation and ring layout of the timed runs
        model.generate_requests(reqs[:2 * B], B)
        model.generate_requests(reqs[:2 * B], B, context_pass=True)
        model.generate_batched(groups[0][0], 8, prompt_lengths=groups[0][1])
        legs = {"requests": run_requests, "requests_prefill": run_prefill, "batched": run_batched}
        out = {k: [] for k in legs}
        peak = {k: 0 for k in legs}
        for _ in range(args.reps):  # alternate the three paths
            for name, fn in legs.items():
                torch.cuda.reset_peak_memory_stats(dev)
                out[name].append(timed(fn))
                peak[name] = max(peak[name], torch.cuda.max_memory_allocated(dev))
        res["prefill_parts"] = prefill_parts(model, sch_pre)
    for name, steps in (("requests", S_req), ("requests_prefill", S_pre), ("batched", S_bat)):
        dev_ms = [d for d, _ in out[name]]
        host_ms = [h for _, h in out[name]]
        med = statistics.median(dev_ms)
        res[name] = {"steps": steps, "kept_column_step_share": kept / (steps * B),
                     "total_ms": {"median": med, "min": min(dev_ms), "max": max(dev_ms)},
                     "generated_tokens_per_s": kept / (med / 1e3),
                     "ms_per_step": med / steps,
                     "host_enqueue_ms_per_step": statistics.median(host_ms) / steps,
                     "max_memory_allocated_GB": peak[name] / 1e9}
    pl = sch_pre.prefill
    res["requests_prefill"]["context_passes"] = sum(t is not None for t in pl.steps)
    res["requests_prefill"]["scatter_launches"] = sum(len(v) for v in pl.slices.values())
    res["requests_prefill"]["start_steps"] = len({int(t) for t in sch_pre.start[sch_pre.req >= 0].unique()})
    res["requests_prefill"]["prefill_pass_share"] = (res["requests_prefill"]["context_passes"]
                                                     * res["prefill_parts"]["pass_ms"]
                                                     / res["requests_prefill"]["total_ms"]["median"])
    res["batched"]["context_passes"] = len(groups)
    res["requests_speedup"] = res["batched"]["total_ms"]["median"] / res["requests"]["total_ms"]["median"]
    res["requests_prefill_speedup"] = (res["batched"]["total_ms"]["median"]
                                       / res["requests_prefill"]["total_ms"]["median"])
    res["requests_prefill_vs_requests"] = (res["requests"]["total_ms"]["median"]
                                           / res["requests_prefill"]["total_ms"]["median"])
    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
