"""CPU: host-side plumbing of the engine that needs no device -- ring-buffer window arithmetic, the padded parameter
layout, batch sharding, the product path's refusal to run without CUDA, and the reference arm's JSON contract."""
import json
import os
import subprocess
import sys
import types

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_ring_window_segments_wrap_and_slide():
    from tgan_b200.engine import RingMems
    slabs = torch.zeros(3, 10, 2, 64)  # 3 slabs, capacity 10 positions
    ring = RingMems(slabs, start=7, length=6, d_model=50)
    assert ring.capacity == 10 and ring.bsz == 2
    assert ring.segments(0, 6) == [(7, 3), (0, 3)]            # logical rows 0..5 wrap around the end of the buffer
    assert ring.segments(2, 3) == [(9, 1), (0, 2)]
    assert ring.segments(4, 2) == [(1, 2)]
    assert ring.size() == (3, 6, 2, 50) and ring.shape[1] == 6
    # a window over the same slabs shares the projected-K/V cache state (decode calls hand it from step to step)
    nxt = RingMems(ring.slabs, 8, 6, 50, kv=ring.kv)
    assert nxt.kv is ring.kv


def test_param_layout_is_tma_friendly_and_covers_the_reference_state_dict():
    from tgan_b200.engine import ParamLayout, TxlDims
    d = TxlDims(n_layer=6, n_head=10, d_model=500, d_inner=1000, n_token=310)
    assert (d.d_head, d.DP, d.NH, d.DIP, d.VP) == (50, 512, 640, 1024, 320)
    lay = ParamLayout(d)
    for name, (off, rows, ld) in lay.mat.items():
        assert ld % 8 == 0 and off % 8 == 0, name   # 16-byte aligned rows: TMA / vector loads
    refs = [r for r, *_ in lay.reference_map()]
    assert len(refs) == len(set(refs)) == 4 + 11 * 6
    for must in ("word_emb.emb_layers.0.weight", "r_w_bias", "layers.5.dec_attn.qkv_net.weight",
                 "layers.0.pos_ff.CoreNet.3.bias", "crit.out_layers.0.bias"):
        assert must in refs
    # the padded gradient buffer holds every matrix once; weights additionally keep a transposed copy for dgrad
    assert lay.gmat_elems < lay.mat_elems


def test_batch_sharding_and_rank_seeds():
    from tgan_b200 import dp
    assert [dp.shard_columns(512, 8, r) for r in (0, 7)] == [(0, 64), (448, 512)]
    with pytest.raises(ValueError):
        dp.shard_columns(510, 8, 0)
    assert dp.rank_seed(1111, 3) == 4111  # train.py:224


def test_product_model_refuses_to_run_without_cuda():
    import mem_transformer as MT
    ns = types.SimpleNamespace
    cfg = ns(MODEL=ns(num_layers=1, num_heads=2, units=16, inner_size=32, dropout=0.0, attention_dropout=0.0,
                      tie_embedding=True, tie_proj=False, pre_lnorm=False, same_length=False, clamp_len=-1),
             TRAIN=ns(tgt_length=4, mem_length=4, pad_type="model", replace_start_with_pad=False, append_note_status=False))
    model = MT.MemTransformerLM(cfg, 20, 0)
    data = torch.randint(0, 20, (4, 2))
    with pytest.raises(RuntimeError, match="CUDA only"):
        model(data, data, torch.zeros(2, dtype=torch.bool), None)
    with pytest.raises(NotImplementedError):
        cfg.MODEL.pre_lnorm = True
        MT.MemTransformerLM(cfg, 20, 0)


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--cpu-batch", "1"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    # the default workload is the metric BASELINE.json names: the experiment_spanbert.yml GAN-step cycle (step 0 of the
    # timed region carries one discriminator + one generator update on the CPU: 123 sampling steps + HF BERT 5x768)
    assert d["impl"] == "reference" and d["metric"] == "train tokens/sec (GAN step)" and d["unit"] == "tokens/s"
    assert "experiment_spanbert.yml" in d["config"]["workload"]
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_dump_outputs_is_refused_with_more_than_one_rank(tmp_path):
    """The dump replays the captured MLE backward, which carries the bucket all-reduces: on one rank alone they would
    wait for the others forever, so bench.py refuses before it touches a device."""
    env = dict(os.environ, WORLD_SIZE="2", RANK="0", LOCAL_RANK="0")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "2", "--dump-outputs",
                          str(tmp_path / "dump")], capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode != 0 and "--dump-outputs runs on one GPU only" in out.stderr, out.stderr[-2000:]
    assert not (tmp_path / "dump").exists()


def test_lamb_chunk_table_covers_every_tensor_exactly_once():
    """FusedLamb cuts the flat parameter buffer into per-tensor chunks of <= 16384 elements (host logic, no kernel)."""
    import torch
    from tgan_b200 import dp
    ps = [torch.nn.Parameter(torch.zeros(7, 5)), torch.nn.Parameter(torch.zeros(40000)), torch.nn.Parameter(torch.zeros(3))]
    fp = dp.FlatParams(ps)
    opt = dp.FusedLamb(fp, 0.01)
    rows = opt.chunks.tolist()
    covered = torch.zeros(fp.numel(), dtype=torch.int32)
    for tid, off, cnt in rows:
        assert 0 < cnt <= dp.FusedLamb.CHUNK
        lo, n = fp.slices[tid]
        assert lo <= off and off + cnt <= lo + n
        covered[off:off + cnt] += 1
    assert bool((covered == 1).all())
    assert opt.norms.numel() == 2 * len(ps)


def test_device_dataset_refuses_cpu_and_unsupported_modes():
    import pytest
    from tgan_b200 import data, lib
    with pytest.raises(lib.TganError):
        data.DeviceSplit([[0, 5, 6]], "cpu")
    with pytest.raises(NotImplementedError):
        data.DeviceMusicDataset({}, 1, "cpu", random_crop=True)
