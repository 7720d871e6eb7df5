"""CPU: the host schedule of MemTransformerLM.generate_requests(context_pass=True)
(mem_transformer.request_schedule(..., context_pass=True)) on small cases worked out by hand: occupancy, forced
tokens, key floors P0 + t0 - n_r, start steps, the prefill groups with their prompt blocks, the step each pass is
enqueued at, the copy descriptors per start step and the initial empty-bar runs."""
import torch

import mem_transformer as MT

E = 37  # empty-bar token


def _cols(t):
    return [list(c) for c in t.t().tolist()]


def test_hand_worked_queue_with_long_and_one_token_prompts():
    # mem_len 3, 2 columns.  n_r = min(T - 1, 3): r0 2, r1 0 (one token), r2 3 (T - 1 = 5 > mem_len), r3 2.
    # P0 = min(3, max T - 1) = 3.  Each request holds its column for gen_len steps: r0 col 0 [0, 2), r1 col 1 [0, 3),
    # r2 col 0 [2, 4), r3 col 1 [3, 4).
    prompts = [[5, 6, 7], [9], [1, 2, 3, 4, 5, 6], [8, E, E]]
    gens = [2, 3, 2, 1]
    sch = MT.request_schedule(prompts, gens, 2, context_pass=True, mem_len=3, empty_tokens=[E] * 4)
    assert sch.tables.dtype == torch.int32 and sch.tables.shape == (5, 4, 2)
    assert _cols(sch.forced) == [[7, -1, 6, -1], [9, -1, -1, E]]  # prompt[-1] only, at the first step
    assert _cols(sch.req) == [[0, 0, 2, 2], [1, 1, 1, 3]]
    assert sch.out_base == [0, 2, 5, 7]
    assert _cols(sch.out_off) == [[0, 1, 5, 6], [2, 3, 4, 7]]  # every step of a request keeps its sample
    # floors P0 + t0 - n_r: r0 3 + 0 - 2, r1 3 + 0 - 0, r2 3 + 2 - 3, r3 3 + 3 - 2
    assert _cols(sch.key_start) == [[1, 1, 2, 2], [3, 3, 3, 4]]
    assert _cols(sch.start) == [[0, 0, 2, 2], [0, 0, 0, 3]]
    pl = sch.prefill
    assert pl.lead == 3
    # group 0 = r0, r1 (longest prompt[:-1]: 2 rows), group 1 = r2, r3 (5 rows); left-padded with token 0
    assert pl.blocks[0].tolist() == [[5, 0], [6, 0]] and pl.pads[0].tolist() == [0, 2]
    assert _cols(pl.blocks[1]) == [[1, 2, 3, 4, 5], [0, 0, 0, 8, E]] and pl.pads[1].tolist() == [0, 3]
    assert pl.steps == [0, 2]  # the start step of each group's first request
    # (source column, first source position = Tm - n_r, destination column, rows); r1 has no rows: no descriptor
    assert pl.desc.dtype == torch.int32
    assert pl.desc.tolist() == [[0, 0, 0, 2], [0, 2, 0, 3], [1, 3, 1, 2]]
    assert pl.slices == {0: [(0, 0, 1, 2)], 2: [(1, 1, 1, 3)], 3: [(1, 2, 1, 2)]}
    assert pl.run0.dtype == torch.int32 and pl.run0.tolist() == [0, 0, 0, 1]  # r3: [8, E] ends in one E


def test_run0_counts_only_the_trailing_run_of_the_request_s_own_empty_token():
    prompts = [[E, E, 4, E, E, E, 9], [E, E, E], [E], [3, 7, 7]]
    sch = MT.request_schedule(prompts, [1, 1, 1, 1], 4, context_pass=True, mem_len=8, empty_tokens=[E, E, E, 7])
    # prompt[:-1]: [E, E, 4, E, E, E] -> 3;  [E, E] -> 2;  [] -> 0;  [3, 7] with empty token 7 -> 1
    assert sch.prefill.run0.tolist() == [3, 2, 0, 1]
    assert MT.request_schedule(prompts, [1] * 4, 4, context_pass=True, mem_len=8).prefill.run0.tolist() == [0] * 4


def test_group_boundary_on_a_shared_start_step_and_idle_tail():
    # 2 columns, mem_len 4.  r0 col 0 [0, 1), r1 col 1 [0, 2), r2 col 0 [1, 2), r3 col 0 [2, 3), r4 col 1 [2, 6):
    # r3 (group 1) and r4 (group 2) start at step 2; column 0 idles from step 3 on.
    prompts = [[1, 2], [3, 4, 5], [6, 7, 8, 9], [10, 11], [12, 13, 14, 15, 16, 17, 18]]
    gens = [1, 2, 1, 1, 4]
    sch = MT.request_schedule(prompts, gens, 2, context_pass=True, mem_len=4)
    S = 6
    assert sch.tables.shape[1:] == (S, 2)
    assert _cols(sch.req) == [[0, 2, 3, -1, -1, -1], [1, 1, 4, 4, 4, 4]]
    pl = sch.prefill
    assert pl.lead == 4  # min(mem_len 4, max T - 1 = 6)
    # idle column 0: token 0, floored at its own row P0 + t, nothing kept
    assert _cols(sch.forced)[0][3:] == [0, 0, 0]
    assert _cols(sch.key_start)[0] == [4 - 1, 4 + 1 - 3, 4 + 2 - 1, 7, 8, 9]
    assert _cols(sch.out_off)[0][3:] == [-1, -1, -1]
    assert _cols(sch.key_start)[1] == [4 - 2] * 2 + [4 + 2 - 4] * 4  # r4: n_r = mem_len = 4
    assert pl.steps == [0, 1, 2]
    assert [b.shape[1] for b in pl.blocks] == [2, 2, 1]
    # first source position Tm - n_r: group 0 has Tm 2 (r0 n_r 1), group 1 Tm 3 (r3 n_r 1), group 2 Tm 6 (n_r 4)
    assert pl.desc.tolist() == [[0, 1, 0, 1], [1, 0, 1, 2], [0, 0, 0, 3], [1, 2, 0, 1], [0, 2, 1, 4]]
    # step 2: group 1's copy of r3 comes before group 2's (whose pass is enqueued at that step)
    assert pl.slices == {0: [(0, 0, 2, 2)], 1: [(1, 2, 1, 3)], 2: [(1, 3, 1, 1), (2, 4, 1, 4)]}


def test_all_one_token_prompts_need_no_pass_and_no_copy():
    sch = MT.request_schedule([[3], [4], [5]], [2, 1, 1], 2, context_pass=True, mem_len=6)
    pl = sch.prefill
    assert pl.lead == 0 and pl.blocks == [None, None] and pl.steps == [None, None]
    assert pl.desc.shape == (0, 4) and pl.slices == {}
    assert _cols(sch.key_start) == [[0, 0], [0, 1]]  # r2 starts at step 1 on no rows: floor 0 + 1 - 0
    assert _cols(sch.forced) == [[3, -1], [4, 5]]


def test_prefill_schedule_invariants_on_a_random_queue():
    g = torch.Generator().manual_seed(3)
    R, B, mem_len = 40, 5, 9
    lens = torch.randint(1, 20, (R,), generator=g).tolist()
    gens = torch.randint(1, 30, (R,), generator=g).tolist()
    prompts = [torch.randint(1, 300, (n,), generator=g).tolist() for n in lens]
    sch = MT.request_schedule(prompts, gens, B, context_pass=True, mem_len=mem_len)
    pl = sch.prefill
    S = sch.tables.shape[1]
    assert pl.lead == min(mem_len, max(lens) - 1)
    assert sum(gens) <= S * B
    starts = []
    for r, (p, k) in enumerate(zip(prompts, gens)):
        t, cs = (sch.req == r).nonzero(as_tuple=True)
        t0, c = int(t[0]), int(cs[0])
        starts.append(t0)
        assert len(set(cs.tolist())) == 1 and t.tolist() == list(range(t0, t0 + k))
        assert int(sch.forced[t0, c]) == p[-1] and (sch.forced[t0 + 1:t0 + k, c] == -1).all()
        assert (sch.key_start[t, c] == pl.lead + t0 - min(len(p) - 1, mem_len)).all()
        assert (sch.start[t, c] == t0).all()
        assert sch.out_off[t0:t0 + k, c].tolist() == list(range(sch.out_base[r], sch.out_base[r] + k))
    assert starts == sorted(starts)
    # every request with prompt rows has one descriptor, applied at its start step, reading its own block column
    applied = []
    for t, sl in sorted(pl.slices.items()):
        assert [e[0] for e in sl] == sorted(e[0] for e in sl)
        for gi, lo, n, mx in sl:
            assert pl.steps[gi] is not None and pl.steps[gi] <= t
            for i in range(lo, lo + n):
                j, pos, c, rows = pl.desc[i].tolist()
                r = gi * B + j
                assert starts[r] == t and rows == min(len(prompts[r]) - 1, mem_len) <= mx
                assert int(sch.req[t, c]) == r
                blk = pl.blocks[gi]
                assert pos + rows == blk.shape[0]
                assert blk[int(pl.pads[gi][j]):, j].tolist() == prompts[r][:-1]
                applied.append(r)
    assert applied == [r for r in range(R) if lens[r] > 1]
