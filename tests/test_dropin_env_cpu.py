"""CPU: the environment shims under transformer-gan_b200/compat (SURVEY.md 8b "environment gaps") -- the yacs-compatible
CfgNode, and the start-up hooks that make the reference's unmodified scripts resolve the hot-path modules to this
package."""
import os
import subprocess
import sys
import textwrap

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COMPAT = os.path.join(ROOT, "transformer-gan_b200", "compat")


def _cfgnode():
    sys.path.insert(0, COMPAT)
    try:
        import importlib
        return importlib.import_module("yacs.config").CfgNode
    finally:
        sys.path.remove(COMPAT)


def test_cfgnode_merge_freeze_clone(tmp_path):
    CN = _cfgnode()
    cfg = CN()
    cfg.MODEL = CN()
    cfg.MODEL.units = 500
    cfg.MODEL.dropout = 0.1
    cfg.TRAIN = CN()
    cfg.TRAIN.lr = 0.004
    cfg.TRAIN.layers = ["0", "1"]
    f = tmp_path / "exp.yml"
    f.write_text("MODEL:\n  units: 64\nTRAIN:\n  lr: 1\n  layers: ['3']\n")
    cfg.freeze()
    cfg.merge_from_file(str(f))               # yacs merges through item assignment: allowed on a frozen node
    assert cfg.MODEL.units == 64 and cfg.TRAIN.lr == 1.0 and isinstance(cfg.TRAIN.lr, float) and cfg.TRAIN.layers == ["3"]
    with pytest.raises(AttributeError):
        cfg.MODEL.units = 3
    cfg.defrost()
    cfg.MODEL.units = 3
    c2 = cfg.clone()
    c2.MODEL.units = 7
    assert cfg.MODEL.units == 3 and c2.MODEL.units == 7
    cfg.merge_from_list(["MODEL.dropout", "0.25", "TRAIN.lr", 0.5])
    assert cfg.MODEL.dropout == 0.25 and cfg.TRAIN.lr == 0.5
    with pytest.raises(KeyError):
        cfg.merge_from_list(["MODEL.nope", 1])
    with pytest.raises(ValueError):
        cfg.merge_from_list(["MODEL.units", "abc"])
    bad = tmp_path / "bad.yml"
    bad.write_text("MODEL:\n  unknown_key: 1\n")
    with pytest.raises(KeyError):
        cfg.merge_from_file(str(bad))
    assert "units: 3" in cfg.dump()


def test_compat_resolves_hot_path_modules_to_this_package(tmp_path):
    """cwd = a script directory with its own mem_transformer.py / transformer_gan.py / discriminator.py /
    utils/proj_adaptive_softmax.py (as the reference's model/ has; here they raise when imported), only compat/ on
    PYTHONPATH: the hot-path modules come from this package, the AdamW alias and the nltk stand-in resolve, and
    TransformerGAN builds the experiment_cnn.yml generator."""
    (tmp_path / "utils").mkdir()  # a namespace package, as in the reference
    for rel in ("mem_transformer.py", "transformer_gan.py", "discriminator.py", "utils/proj_adaptive_softmax.py"):
        (tmp_path / rel).write_text("raise ImportError('the script directory copy was imported')\n")
    code = textwrap.dedent("""
        import types
        import transformer_gan, mem_transformer, discriminator
        import utils.proj_adaptive_softmax
        from transformers import AdamW
        import torch
        assert AdamW is torch.optim.AdamW
        for m in (transformer_gan, mem_transformer, discriminator, utils.proj_adaptive_softmax):
            assert "transformer-gan_b200" in m.__file__, m.__file__
        from nltk.translate.bleu_score import SmoothingFunction, sentence_bleu  # noqa: F401  (utils/bleu.py's imports)
        ns = types.SimpleNamespace
        cfg = ns(MODEL=ns(num_layers=6, num_heads=10, units=500, inner_size=1000, dropout=0.1, attention_dropout=0.1,
                          tie_embedding=True, tie_proj=False, pre_lnorm=False, same_length=False, clamp_len=-1),
                 TRAIN=ns(tgt_length=128, mem_length=1024, pad_type="model", replace_start_with_pad=False,
                          append_note_status=False),
                 DISCRIMINATOR=ns(type="cnn", tgt_len=128, mem_len=128, context_len=5, sample_chunks_mem=2,
                                  truncate_backprop=False, backprop_outside=True, gen_loss_factor=1.0,
                                  dis_loss_factor=1.0, batch_chunk=1, BERT=ns(loss_type="wgan-gp"),
                                  CNN=ns(embed_dim=64, hidden_dim=64, num_rep=64, init="uniform", loss_type="rsgan")))
        class V:
            vec_len = 0
            def __len__(self):
                return 310
        m = transformer_gan.TransformerGAN(cfg, V())
        n = sum(p.numel() for p in m.generator.parameters())
        assert n == 13677310, n
        sd = m.generator.state_dict()
        for k in ("word_emb.emb_layers.0.weight", "layers.5.dec_attn.qkv_net.weight", "r_w_bias", "crit.out_layers.0.bias"):
            assert k in sd, k
        print("DROPIN_OK")
    """)
    env = dict(os.environ, PYTHONPATH=COMPAT)
    out = subprocess.run([sys.executable, "-c", code], cwd=tmp_path, env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "DROPIN_OK" in out.stdout, out.stderr[-3000:]
