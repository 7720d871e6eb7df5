"""CPU: the host schedule of MemTransformerLM.generate_requests (mem_transformer.request_schedule) on small cases
worked out by hand: which column serves which request at which step, the forced tokens, the key floor and the output
offsets."""
import torch

import mem_transformer as MT


def _cols(t):
    return [list(c) for c in t.t().tolist()]


def test_single_column_runs_the_queue_back_to_back():
    sch = MT.request_schedule([[5, 6, 7], [9]], [2, 3], 1)
    assert sch.tables.dtype == torch.int32 and sch.tables.shape == (4, 4 + 3, 1)
    # request 0: 3 prompt steps + 1 more, request 1 starts at step 4 and samples at its first step
    assert _cols(sch.forced) == [[5, 6, 7, -1, 9, -1, -1]]
    assert _cols(sch.req) == [[0, 0, 0, 0, 1, 1, 1]]
    assert _cols(sch.out_off) == [[-1, -1, 0, 1, 2, 3, 4]]
    assert _cols(sch.key_start) == [[0, 0, 0, 0, 4, 4, 4]]
    assert sch.out_base == [0, 2]


def test_assignment_goes_to_the_column_that_frees_first_ties_to_the_lowest():
    # steps T + g - 1: r0 = 4 on col 0, r1 = 2 on col 1, r2 = 2 on col 2; r3 -> col 1 (frees at 2, tie with col 2
    # broken low), r4 -> col 2 (frees at 2), r5 -> col 1 (frees at 3), r6 -> col 0 (frees at 4)
    prompts = [[1, 2, 3], [4], [5, 6], [7], [8, 9], [10], [11]]
    gens = [2, 2, 1, 1, 3, 2, 1]
    sch = MT.request_schedule(prompts, gens, 3)
    assert sch.tables.shape[1:] == (6, 3)
    assert _cols(sch.req) == [[0, 0, 0, 0, 6, -1],
                              [1, 1, 3, 5, 5, -1],
                              [2, 2, 4, 4, 4, 4]]
    assert _cols(sch.forced) == [[1, 2, 3, -1, 11, 0],
                                 [4, -1, 7, 10, -1, 0],
                                 [5, 6, 8, 9, -1, -1]]
    assert _cols(sch.key_start) == [[0, 0, 0, 0, 4, 5],
                                    [0, 0, 2, 3, 3, 5],
                                    [0, 0, 2, 2, 2, 2]]
    assert sch.out_base == [0, 2, 4, 5, 6, 9, 11]
    assert _cols(sch.out_off) == [[-1, -1, 0, 1, 11, -1],
                                  [2, 3, 5, 9, 10, -1],
                                  [-1, 4, -1, 6, 7, 8]]
    # every output slot is written exactly once
    offs = sch.out_off[sch.out_off >= 0]
    assert sorted(offs.tolist()) == list(range(sum(gens)))


def test_idle_tail_is_fed_a_valid_token_and_floored_at_its_own_row():
    sch = MT.request_schedule([[3] * 6, [4]], [2, 1], 2)
    S = 7
    assert sch.tables.shape[1:] == (S, 2)
    assert _cols(sch.req)[1] == [1] + [-1] * (S - 1)
    assert _cols(sch.forced)[1] == [4] + [0] * (S - 1)
    assert _cols(sch.out_off)[1] == [2] + [-1] * (S - 1)  # request 0 keeps outputs 0 and 1
    assert _cols(sch.key_start)[1] == list(range(S))


def test_fewer_requests_than_batch_size_use_one_column_each():
    sch = MT.request_schedule([[1, 2], [3]], [1, 4], 8)
    assert sch.tables.shape[1:] == (4, 2)
    assert _cols(sch.forced) == [[1, 2, 0, 0], [3, -1, -1, -1]]


def test_schedule_invariants_on_a_random_queue():
    g = torch.Generator().manual_seed(3)
    R, B = 40, 5
    lens = torch.randint(1, 20, (R,), generator=g).tolist()
    gens = torch.randint(1, 30, (R,), generator=g).tolist()
    prompts = [torch.randint(1, 300, (n,), generator=g).tolist() for n in lens]
    sch = MT.request_schedule(prompts, gens, B)
    S = sch.tables.shape[1]
    assert S >= max(n + k - 1 for n, k in zip(lens, gens))
    assert sum(n + k - 1 for n, k in zip(lens, gens)) <= S * B
    for r, (p, k) in enumerate(zip(prompts, gens)):
        t, c = (sch.req == r).nonzero(as_tuple=True)
        assert len(set(c.tolist())) == 1 and t.tolist() == list(range(int(t[0]), int(t[0]) + len(p) + k - 1))
        t0, c = int(t[0]), int(c[0])
        assert sch.forced[t0:t0 + len(p), c].tolist() == p
        assert (sch.forced[t0 + len(p):t0 + len(p) + k - 1, c] == -1).all()
        assert (sch.key_start[t, c] == t0).all()
        assert sch.out_off[t0 + len(p) - 1:t0 + len(p) + k - 1, c].tolist() == \
            list(range(sch.out_base[r], sch.out_base[r] + k))
    # a later request never starts before an earlier one (list order)
    starts = [int((sch.req == r).nonzero()[0, 0]) for r in range(R)]
    assert starts == sorted(starts)
