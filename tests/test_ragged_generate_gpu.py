"""GPU: batched generation from prompts of different lengths (MemTransformerLM.generate_batched(prompt_lengths=...)):
every sequence of the batch generates what it generates alone, and a memory that carries the key floor of the padded
prompts never reaches a training path."""
import pytest
import torch

import txl_oracle as O
from test_model_gpu import build

pytestmark = pytest.mark.gpu
V = 310


@pytest.mark.parametrize("technique,topk,k_empty", [("topk", 32, 0), ("topk", 6, 2)])
def test_ragged_generation_matches_each_prompt_alone(technique, topk, k_empty):
    """fp32 mode against generate.py restated with the oracle, each column on its own unpadded prompt, under the same
    injected uniforms (margin rule of test_sampling_gpu).  mem_len 12 < the longest prompt: the context pass drops the
    oldest rows, the window slides and the ring is re-laid out during the loop."""
    shape = O.TxlShape(n_layer=2, n_head=4, d_model=40, d_inner=72, n_token=V, mem_len=12, same_length=True)
    seed, G, temperature, empty_tok = 31, 20, 0.95, 37
    lens = [1, 2, 7, 13, 40]
    T0, B = 44, len(lens)
    model = build(shape, seed, 1, torch.float32).eval()
    g = torch.Generator().manual_seed(9)
    start = torch.randint(2, V, (T0, B), generator=g)  # right-padded: rows past each prompt must be ignored
    if k_empty:
        # column 0's one token is the empty token: the left padding repeats it, so counting pad rows into the
        # empty-bar run would suppress it at the first step (the prompt itself is a run of 1 < k)
        start[0, 0] = empty_tok
        with torch.no_grad():
            model.crit.out_layers[0].bias[empty_tok] += 6.0
    U = torch.rand(G, B, generator=g)
    ids, mems = model.generate_batched(start.cuda(), G, technique=technique, topk=topk, temperature=temperature,
                                       exclude_bos=True, empty_token=empty_tok, num_empty_tokens_to_ignore=k_empty,
                                       uniforms=U.cuda(), prompt_lengths=lens)
    torch.cuda.synchronize()
    ids = ids.cpu()
    # the window after max(lens) - 1 context rows and G single-token steps
    assert mems.key_start is not None and mems.length == shape.mem_len
    assert mems.pos0 == max(lens) - 1 + G - mems.length
    assert mems.key_start.cpu().tolist() == [max(lens) - n for n in lens]

    params = {k: v.double() for k, v in O.init_params(shape, seed).items()}
    if k_empty:
        params["crit.out_layers.0.bias"] = params["crit.out_layers.0.bias"].clone()
        params["crit.out_layers.0.bias"][empty_tok] += 6.0
    checked = suppressed = 0
    for b in range(B):
        seq = [int(t) for t in start[:lens[b], b]]
        om = None
        if lens[b] > 1:
            _, om = O.generate_logits(start[:lens[b] - 1, b:b + 1], None, params, shape)
        for t in range(G):
            lg, om = O.generate_logits(torch.tensor([[seq[-1]]]), om, params, shape)
            # suppressed after a run of k empty tokens (a one-token prompt is a run of one, however it is padded)
            sup = k_empty > 0 and len(seq) >= k_empty and all(s == empty_tok for s in seq[-k_empty:])
            suppressed += int(sup)
            probs = O.generation_probs(lg[-1, 0], temperature=temperature, technique=technique, topk=topk, p=0.0,
                                       exclude_bos=True, suppress_empty=sup, empty_bar_token=empty_tok)
            tok, margin = O.categorical_from_uniform(probs, float(U[t, b]))
            got = int(ids[t, b])
            if margin < 2e-4:  # u within the fp32 model error of a CDF step: either neighbour is a legitimate draw
                assert probs[got] > 0, (b, t, got)
            else:
                assert got == tok, (b, t, got, tok, margin)
                checked += 1
            assert got != 0 and not (sup and got == empty_tok)
            seq.append(got)
    assert checked > 0.85 * B * G
    assert not k_empty or suppressed > 0


def test_ragged_bf16_real_size_matches_single_prompt_runs():
    """bf16 at the real model size (6 x 500): the context pass over the longest prompt takes the tcgen05 kernel, the
    single-prompt runs mostly the SIMT kernels.  Per column, the logits of the first steps after the prompt and the
    real rows of the memory match a B = 1 run of that prompt alone (teacher-forced with the same tokens)."""
    shape = O.TxlShape(n_layer=6, n_head=10, d_model=500, d_inner=1000, n_token=V, mem_len=128, same_length=True)
    lens = [200, 150, 97, 33, 64, 1, 5, 181]
    T0, B, S = 200, len(lens), 3
    model = build(shape, 5, 1, torch.bfloat16).eval()
    g = torch.Generator().manual_seed(4)
    start = torch.randint(2, V, (T0, B), generator=g).cuda()
    forced = torch.randint(2, V, (S, B), generator=g).cuda()

    def run(prompt, lengths, cols):
        _, mems = model.generate_batched(prompt, 0, prompt_lengths=lengths)
        last = torch.stack([prompt[n - 1, c] for c, n in enumerate(lengths or [prompt.shape[0]] * prompt.shape[1])])
        steps = [last.view(1, -1)] + [forced[s:s + 1, cols] for s in range(S - 1)]
        logits = []
        for x in steps:
            lg, mems = model.forward_generate(x, mems)
            logits.append(lg[0].float())
        return torch.stack(logits), mems

    def chk(name, got, want):
        # 1e-2 of the values' scale: a B = 8 and a B = 1 run round differently in bf16 even without padding (logits
        # reach ~4, where one bf16 step is 0.016); a pad row leaking into the attention moves them by O(1)
        err = (got - want).abs().max().item()
        assert err <= 1e-2 * max(1.0, want.abs().max().item()), (name, err, want.abs().max().item())

    with torch.no_grad():
        lg_all, mems_all = run(start, lens, slice(None))
        mat_all = mems_all.materialize()
        torch.cuda.synchronize()
        assert mems_all.key_start is not None
        for b, n in enumerate(lens):
            lg_b, mems_b = run(start[:n, b:b + 1].contiguous(), None, slice(b, b + 1))
            chk(f"logits {b} (length {n})", lg_all[:, b], lg_b[:, 0])
            want = mems_b.materialize()[:, :, 0]
            pad_in_window = max(0, (T0 - n) - mems_all.pos0)
            got = mat_all[:, pad_in_window:, b]
            assert got.shape == want.shape, (b, got.shape, want.shape)
            chk(f"memory {b} (length {n})", got, want)


def test_split_generation_continues_through_the_returned_memory():
    shape = O.TxlShape(n_layer=2, n_head=4, d_model=40, d_inner=72, n_token=V, mem_len=10, same_length=True)
    model = build(shape, 3, 1, torch.float32).eval()
    lens = [3, 1, 9, 6]
    g = torch.Generator().manual_seed(2)
    start = torch.randint(2, V, (9, len(lens)), generator=g).cuda()
    U = torch.rand(16, len(lens), generator=g).cuda()
    ids, _ = model.generate_batched(start, 16, uniforms=U, prompt_lengths=lens)
    a, mems = model.generate_batched(start, 7, uniforms=U[:7], prompt_lengths=lens)
    b, _ = model.generate_batched(a[-1:], 9, uniforms=U[7:], mems=mems)
    torch.cuda.synchronize()
    assert torch.equal(ids, torch.cat([a, b]))


def test_bad_prompt_lengths_raise():
    shape = O.TxlShape(n_layer=2, n_head=4, d_model=40, d_inner=72, n_token=V, mem_len=10)
    model = build(shape, 3, 1, torch.float32).eval()
    start = torch.randint(2, V, (5, 3)).cuda()
    for lens in ([0, 2, 3], [1, 6, 2], [1, 2], [[1, 2, 3]] * 2):
        with pytest.raises(ValueError):
            model.generate_batched(start, 2, prompt_lengths=lens)
    _, mems = model.generate_batched(start, 2)
    with pytest.raises(ValueError):
        model.generate_batched(start, 2, prompt_lengths=[1, 2, 3], mems=mems)


def test_ragged_memory_never_reaches_training(tmp_path):
    """A memory with a key floor raises in every call that would train through it -- before any kernel launch."""
    from tgan_b200 import lib as L
    from test_gan_gpu import _build_gan
    gan, z, shape = _build_gan("gan_cnn_tiny", tmp_path, torch.float32)
    model = gan.generator
    B = 3
    start = torch.randint(2, shape.n_token, (max(shape.mem_len, 4) + 2, B)).cuda()
    # long enough to fill the memory: the captured MLE path takes only a full-length memory
    _, mems = model.generate_batched(start, 2, prompt_lengths=[start.shape[0], 2, 1])
    assert mems.key_start is not None and mems.length == model.mem_len
    data, target = start[:4], start[1:5]
    model.train()
    n0 = L.launch_count()
    with pytest.raises(L.TganError):
        model(data, target, None, mems)                        # eager MLE forward that saves activations
    with pytest.raises(L.TganError):
        model.forward_generate_gumbel(data[:1], 1.0, mems)     # sampling step of the GAN chain, with gradient
    model.use_cuda_graphs = True
    try:
        with pytest.raises(L.TganError):
            model(data, target, None, mems)                    # captured MLE step
    finally:
        model.use_cuda_graphs = False
    with pytest.raises(L.TganError):
        gan(data, target, None, ["mle", "gen"], mems=mems)     # TransformerGAN step (its MLE part takes the memory)
    assert L.launch_count() == n0
    # inference through the same memory still works
    with torch.no_grad():
        lg, _ = model.forward_generate(data[:1], mems)
    assert torch.isfinite(lg).all()
