"""Generate tests/golden/*.npz by running the UNMODIFIED reference (/root/reference/model) on CPU.

TEST INFRASTRUCTURE ONLY.  Run in the build container:  ``python oracle/make_goldens.py``.
Inputs are windows of the reference's own real-token fixture ``test/prefix_test.npy``; parameters are
regenerated from a seed by ``txl_oracle.init_params`` (so the 13.7 M-parameter real-size case needs no
55 MB file).  The reference runs in float64 (``model.double()``), dropout 0, so the goldens pin the
arithmetic far below any tolerance used later (fp32 mode 1e-4, bf16 1e-2).
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_harness  # noqa: E402
import txl_oracle as O  # noqa: E402

GOLD = os.path.join(os.path.dirname(HERE), "tests", "golden")
PREFIX = "/root/reference/test/prefix_test.npy"


def token_stream(B, total_len, offset=0):
    """[total_len+1, B] int64 windows of prefix_test.npy, one contiguous stretch per batch column."""
    a = np.load(PREFIX).astype(np.int64)
    per = (len(a) - offset) // B
    assert per > total_len
    cols = [a[offset + b * per: offset + b * per + total_len + 1] for b in range(B)]
    return torch.from_numpy(np.stack(cols, 1))


def run_mle_case(name, shape: O.TxlShape, seed, Q, B, nseg, reset_at=None, full_mems=True, grad_thin=1):
    """grad_thin: keep every grad_thin-th of the 2048 sampled entries of each large gradient (keeps the real-size
    fixtures under 1 MB)."""
    params = O.init_params(shape, seed, dtype=torch.float64)
    model = ref_harness.build_reference_lm(shape, params, Q, dtype=torch.float64)
    for p in model.parameters():
        p.requires_grad_(True)
    stream = token_stream(B, Q * nseg)
    mems = None
    out = {"seed": seed, "Q": Q, "B": B, "nseg": nseg,
           "shape": np.array([shape.n_layer, shape.n_head, shape.d_model, shape.d_inner, shape.n_token,
                              shape.mem_len, int(shape.same_length), shape.clamp_len, int(shape.pre_lnorm)])}
    model.zero_grad()
    for s in range(nseg):
        data = stream[s * Q:(s + 1) * Q].contiguous()
        target = stream[s * Q + 1:(s + 1) * Q + 1].contiguous()
        reset = torch.zeros(B, dtype=torch.bool)
        if reset_at is not None and s == reset_at[0]:
            reset[reset_at[1]] = True
        loss, mems = model(data, target, reset, mems)
        (loss.mean()).backward()
        out[f"data{s}"] = data.numpy()
        out[f"target{s}"] = target.numpy()
        out[f"reset{s}"] = reset.numpy()
        out[f"loss{s}"] = loss.detach().numpy()
    m = mems.detach().numpy()
    out["mems_shape"] = np.array(m.shape)
    if full_mems:
        out["mems"] = m
    else:
        out["mems_slice"] = m[:, :, :, ::7].astype(np.float64)
    sd_grads = {}
    for k, p in model.named_parameters():
        if k == "crit.out_layers.0.weight":
            continue
        sd_grads[k] = p.grad.detach()
    for k, g in sd_grads.items():
        key = k.replace(".", "/")
        out["gnorm:" + key] = np.array(g.norm().item())
        flat = g.reshape(-1)
        if flat.numel() <= 4096:
            out["grad:" + key] = g.numpy()
        else:
            idx = torch.linspace(0, flat.numel() - 1, 2048).long()[::grad_thin]
            out["gidx:" + key] = idx.numpy()
            out["gval:" + key] = flat[idx].numpy()
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)
    print("wrote", name, "loss0 mean", float(out["loss0"].mean()))


def run_generate_case(name, shape: O.TxlShape, seed, B, T, temperature):
    """forward_generate: incremental-with-memory vs one-shot (generate.py:309-327 invariance) and
    forward_generate_gumbel with injected uniform noise."""
    params = O.init_params(shape, seed, dtype=torch.float64)
    model = ref_harness.build_reference_lm(shape, params, 1, dtype=torch.float64)
    stream = token_stream(B, T, offset=1234)
    data = stream[:T].contiguous()
    out = {"seed": seed, "B": B, "T": T, "temperature": temperature, "data": data.numpy(),
           "shape": np.array([shape.n_layer, shape.n_head, shape.d_model, shape.d_inner, shape.n_token,
                              shape.mem_len, int(shape.same_length), shape.clamp_len, int(shape.pre_lnorm)])}
    with torch.no_grad():
        full_logits, full_mems = model.forward_generate(data, None)
        mems = None
        inc = []
        for t in range(T):
            lg, mems = model.forward_generate(data[t:t + 1], mems)
            inc.append(lg)
        inc = torch.cat(inc, 0)
        out["full_logits"] = full_logits.numpy()
        out["inc_logits"] = inc.numpy()
        out["full_mems"] = full_mems.numpy()
        out["inc_mems"] = mems.numpy()
        # gumbel: context of 3 tokens, then 4 sampled steps fed back as hard ids
        g = torch.Generator().manual_seed(seed + 1)
        U = [torch.rand(1, B, shape.n_token, generator=g, dtype=torch.float64) for _ in range(4)]
        _, mems = model.forward_generate(data[:3], None)
        inp = data[3:4]
        sts, ids = [], []
        with ref_harness.injected_uniform(U):
            for t in range(4):
                st, mems = model.forward_generate_gumbel(inp, temperature, mems)
                sts.append(st)
                inp = st.argmax(-1)
                ids.append(inp)
        out["gumbel_U"] = torch.cat(U, 0).numpy()
        out["gumbel_st"] = torch.cat(sts, 0).numpy()
        out["gumbel_ids"] = torch.cat(ids, 0).numpy()
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)
    print("wrote", name)


def run_gan_case(name, shape: O.TxlShape, seed, B, dis_type, loss_type, dis_tgt_len=16, context_len=5, chunks=2,
                 temperature=0.8):
    """One "dis_loss" and one "gen_loss" call of the UNMODIFIED reference TransformerGAN (fp32: its one-hot rows are
    hard-coded float32, transformer_gan.py:268-271) with injected Gumbel noise and GP alphas."""
    import tempfile
    V = shape.n_token
    bert_dir = ref_harness.tiny_bert_config_dir(os.path.join(tempfile.mkdtemp(), "bert"), V + 1)
    cfg = ref_harness.make_gan_cfg(shape, dis_tgt_len, shape.mem_len, dis_type, dis_tgt_len, shape.mem_len, context_len,
                                   chunks, loss_type, bert_path=bert_dir)
    params = O.init_params(shape, seed, dtype=torch.float32)
    torch.manual_seed(seed)
    model = ref_harness.build_reference_gan(cfg, V, params, dtype=torch.float32)
    dis_state = O.seeded_state(model.discriminator, seed + 1)
    model.discriminator.load_state_dict(dis_state, strict=False)
    if hasattr(model.discriminator, "dropout"):
        model.discriminator.dropout.p = 0.0  # RelGAN_D hard-codes dropout 0.25 (transformer_gan.py:52): off for a fixture
    model.temperature = temperature
    g = torch.Generator().manual_seed(seed + 2)
    data = token_stream(B, dis_tgt_len, offset=777)[:dis_tgt_len].contiguous()
    n_steps = dis_tgt_len - context_len
    U = [torch.rand(1, B, V, generator=g) for _ in range(n_steps)]
    alphas = [torch.rand(B, 1, 1, generator=g) for _ in range(chunks)]
    out = {"seed": seed, "B": B, "dis_type": dis_type, "loss_type": loss_type, "dis_tgt_len": dis_tgt_len,
           "context_len": context_len, "chunks": chunks, "temperature": temperature, "data": data.numpy(),
           "U": torch.cat(U, 0).numpy(), "alpha": torch.cat(alphas, 0).view(chunks, B).numpy(),
           "shape": np.array([shape.n_layer, shape.n_head, shape.d_model, shape.d_inner, shape.n_token,
                              shape.mem_len, int(shape.same_length), shape.clamp_len, int(shape.pre_lnorm)])}
    # discriminator weights are regenerated by txl_oracle.seeded_state(module, seed + 1) (keyed by tensor name)
    for mode in ("dis_loss", "gen_loss"):
        model.zero_grad()
        with ref_harness.injected_uniform(U, alphas):
            r = model(data, None, None, mode)
        for k in ("dis_loss", "gen_loss", "gp_loss"):
            if r.get(k) is not None:
                out[f"{mode}.{k}"] = np.array(float(r[k]))
        owner = model.discriminator if mode == "dis_loss" else model.generator
        for k, prm in owner.named_parameters():
            if prm.grad is not None and prm.numel() <= 40000:  # keep the fixture small: skip the 1.4 M highway matrix etc.
                out[f"{mode}.grad.{k}"] = prm.grad.numpy().copy()
        if mode == "dis_loss":
            assert all(prm.grad is None for prm in model.generator.parameters())
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)
    print("wrote", name, {k: float(v) for k, v in out.items() if k.endswith("_loss")})


def run_gan_ppo_case(name, shape: O.TxlShape, seed, B, dis_tgt_len=16, context_len=5, chunks=2, temperature=0.8):
    """The PPO variant of the GAN step (transformer_gan.py:184-201, :350-388) on the UNMODIFIED reference: BERT
    discriminator with loss_type 'ppo-gp', density-ratio classifier ``dis_D`` = RelGAN_D with one representation
    (PPO.dis_D_type 'cnn'; the reference's 'bert' branch reads self.discriminator before it exists, :140).  Calls, in
    train.py's order (:1037-1052): "classifier_loss" (P0 initialised), "gen_loss" with update_D0, "gen_loss" without,
    "dis_loss"."""
    import tempfile
    V = shape.n_token
    bert_dir = ref_harness.tiny_bert_config_dir(os.path.join(tempfile.mkdtemp(), "bert"), V + 1)
    cfg = ref_harness.make_gan_cfg(shape, dis_tgt_len, shape.mem_len, "bert", dis_tgt_len, shape.mem_len, context_len,
                                   chunks, "ppo-gp", bert_path=bert_dir)
    cfg.PPO.dis_D_type = "cnn"
    params = O.init_params(shape, seed, dtype=torch.float32)
    torch.manual_seed(seed)
    model = ref_harness.build_reference_gan(cfg, V, params, dtype=torch.float32)
    model.discriminator.load_state_dict(O.seeded_state(model.discriminator, seed + 1), strict=False)
    model.dis_D.load_state_dict(O.seeded_state(model.dis_D, seed + 3), strict=False)
    model.dis_D.dropout.p = 0.0  # RelGAN_D hard-codes dropout 0.25: off for a fixture
    model.temperature = temperature
    g = torch.Generator().manual_seed(seed + 2)
    data = token_stream(B, dis_tgt_len, offset=555)[:dis_tgt_len].contiguous()
    n_steps = dis_tgt_len - context_len
    U = [torch.rand(1, B, V, generator=g) for _ in range(n_steps)]
    alphas = [torch.rand(B, 1, 1, generator=g) for _ in range(chunks)]
    out = {"seed": seed, "B": B, "dis_type": "bert", "loss_type": "ppo-gp", "dis_tgt_len": dis_tgt_len,
           "context_len": context_len, "chunks": chunks, "temperature": temperature, "data": data.numpy(),
           "U": torch.cat(U, 0).numpy(), "alpha": torch.cat(alphas, 0).view(chunks, B).numpy(), "clip": cfg.PPO.clip_param,
           "shape": np.array([shape.n_layer, shape.n_head, shape.d_model, shape.d_inner, shape.n_token,
                              shape.mem_len, int(shape.same_length), shape.clamp_len, int(shape.pre_lnorm)])}
    calls = [("classifier_loss", "classifier_loss", False), ("gen_loss_d0", "gen_loss", True),
             ("gen_loss", "gen_loss", False), ("dis_loss", "dis_loss", False)]
    for tag, mode, upd in calls:
        model.zero_grad()
        with ref_harness.injected_uniform(U, alphas):
            r = model(data, None, None, mode, update_D0=upd)
        for k in ("dis_loss", "gen_loss", "gp_loss"):
            if r.get(k) is not None:
                out[f"{tag}.{k}"] = np.array(float(r[k]))
        out[f"{tag}.P0"] = model.P0.numpy().copy()
        owner = {"classifier_loss": model.dis_D, "dis_loss": model.discriminator}.get(mode, model.generator)
        for k, prm in owner.named_parameters():
            if prm.grad is not None and prm.numel() <= 40000:
                out[f"{tag}.grad.{k}"] = prm.grad.numpy().copy()
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)
    print("wrote", name, {k: float(v) for k, v in out.items() if k.endswith("_loss")})


def run_batches_case(name, seed=21, n_seq=37, B=5, bptt=8, n_train=60, n_dis=12):
    """Batches of the UNMODIFIED reference iterators (data_utils.py:206-434) on a seeded ragged corpus: the training
    iterator through two reshuffles, the one-pass (do_shuffle False) variant, eval_iterator with and without rank
    sharding, and get_dis_iterator under a seeded global numpy RNG."""
    sys.path.insert(0, "/root/reference/model")
    import data_utils as DU
    import data_oracle
    seqs = data_oracle.ragged_corpus(seed, n_seq)
    ds = DU.MusicDataset.__new__(DU.MusicDataset)  # bypass the directory loader: the iterators only read these fields
    ds._vocab = DU.BaseVocab(["<S>", "<PAD>"] + [f"t{i}" for i in range(308)])
    tens = [torch.from_numpy(a) for a in seqs]
    ds._train_data = ds._valid_data = ds._test_data = tens
    ds._train_seq_length = ds._valid_seq_length = ds._test_seq_length = np.array([len(a) for a in seqs], dtype=np.int32)
    ns = ref_harness._Node
    ds.cfg = ns(TRAIN=ns(append_note_status=False, random_crop=False, mem_length=16))
    out = {"seed": seed, "n_seq": n_seq, "B": B, "bptt": bptt, "pad_id": ds.vocab.pad_id}

    def dump(tag, it, n, has_target=True):
        k = 0
        for item in it:
            if k >= n:
                break
            out[f"{tag}.data{k}"] = item[0].numpy().copy()
            if has_target:
                out[f"{tag}.target{k}"] = item[1].numpy().copy()
                out[f"{tag}.reset{k}"] = np.asarray(item[2].numpy() if hasattr(item[2], "numpy") else item[2]).copy()
                out[f"{tag}.ntok{k}"] = np.array(int(item[3]))
            else:
                out[f"{tag}.ntok{k}"] = np.array(int(item[1]))
            k += 1
        out[f"{tag}.n"] = k

    dump("train", ds.get_iterator(B, bptt, "cpu", "train", True, seed=7)(), n_train)
    dump("once", ds.get_iterator(B, bptt, "cpu", "train", False)(), 10 ** 6)
    dump("eval", ds.eval_iterator(B, bptt, "cpu", "valid")(), 10 ** 6)
    dump("eval_r1", ds.eval_iterator(B, bptt, "cpu", "valid", local_rank=1, world_size=2)(), 10 ** 6)
    np.random.seed(99)  # get_dis_iterator draws its offsets from the GLOBAL numpy RNG (:349)
    dump("dis", ds.get_dis_iterator(B, bptt, "cpu", "train", True, seed=5)(), n_dis, has_target=False)
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)
    print("wrote", name, {k: out[k] for k in out if k.endswith(".n")})


def lamb_case_tensors(seed):
    """Seeded parameter / gradient tensors of the LAMB fixture: a matrix, an all-zero vector (trust ratio 1), a long
    vector whose norm exceeds the clamp at 10, and a tensor that spans several 16384-element chunks."""
    g = torch.Generator().manual_seed(seed)
    params = [torch.randn(7, 5, generator=g), torch.zeros(4), 20.0 * torch.randn(3000, generator=g),
              0.02 * torch.randn(150, 300, generator=g)]
    grads = [[torch.randn(p.shape, generator=g) * (0.5 + k) for p in params] for k in range(3)]
    return params, grads


def run_lamb_case(name, seed=23):
    """Three steps of the UNMODIFIED reference ``lamb.Lamb`` (lamb.py:57-118), weight decay 0.01."""
    sys.path.insert(0, "/root/reference/model")
    import warnings
    import lamb
    params, grads = lamb_case_tensors(seed)
    ps = [torch.nn.Parameter(p.clone()) for p in params]
    opt = lamb.Lamb(ps, lr=0.01, weight_decay=0.01)
    out = {"seed": seed, "lr": 0.01, "weight_decay": 0.01, "steps": len(grads)}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for k, gs in enumerate(grads):
            for p, g in zip(ps, gs):
                p.grad = g.clone()
            opt.step()
            out[f"trust{k}"] = np.array([float(opt.state[p]["trust_ratio"]) for p in ps])
            for i, p in enumerate(ps):
                out[f"p{k}.{i}"] = p.detach().numpy().copy()
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)
    print("wrote", name, out["trust2"])


def main():
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(8)
    only = sys.argv[1:]  # optional: regenerate just the named fixtures
    tiny = O.TxlShape(n_layer=2, n_head=4, d_model=40, d_inner=72, n_token=310, mem_len=16)
    tiny_sl = O.TxlShape(n_layer=2, n_head=4, d_model=40, d_inner=72, n_token=310, mem_len=12, same_length=True,
                         clamp_len=15)
    real = O.TxlShape(n_layer=6, n_head=10, d_model=500, d_inner=1000, n_token=310, mem_len=24)
    # Q = 32 is the smallest segment the tcgen05 attention kernels take: this fixture drives them (and the wrap of the
    # 64 + 32 ring) from the model-level golden test
    real_q32 = O.TxlShape(n_layer=6, n_head=10, d_model=500, d_inner=1000, n_token=310, mem_len=64)
    gen = O.TxlShape(n_layer=2, n_head=4, d_model=40, d_inner=72, n_token=310, mem_len=64, same_length=True)
    gan = O.TxlShape(n_layer=2, n_head=4, d_model=40, d_inner=72, n_token=310, mem_len=16)
    cases = {
        "mle_tiny": lambda n: run_mle_case(n, tiny, seed=11, Q=8, B=3, nseg=4, reset_at=(2, 1)),
        "mle_tiny_samelen": lambda n: run_mle_case(n, tiny_sl, seed=12, Q=8, B=2, nseg=4, reset_at=(1, 0)),
        "mle_real": lambda n: run_mle_case(n, real, seed=13, Q=16, B=2, nseg=3, reset_at=(2, 1), full_mems=False,
                                           grad_thin=2),
        "mle_real_q32": lambda n: run_mle_case(n, real_q32, seed=18, Q=32, B=2, nseg=4, reset_at=(3, 1), full_mems=False,
                                               grad_thin=3),
        "generate_tiny": lambda n: run_generate_case(n, gen, seed=14, B=2, T=12, temperature=0.7),
        "gan_bert_tiny": lambda n: run_gan_case(n, gan, seed=15, B=3, dis_type="bert", loss_type="wgan-gp"),
        "gan_cnn_tiny": lambda n: run_gan_case(n, gan, seed=16, B=2, dis_type="cnn", loss_type="rsgan"),
        "gan_ppo_tiny": lambda n: run_gan_ppo_case(n, gan, seed=17, B=3),
        "batches_tiny": lambda n: run_batches_case(n),
        "lamb_tiny": lambda n: run_lamb_case(n),
    }
    for name, fn in cases.items():
        if not only or name in only:
            fn(name)


if __name__ == "__main__":
    main()
