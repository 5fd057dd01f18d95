"""Config surface: the reference's examples/*.config load unchanged, and the generated configs are equivalent.

The reference's examples are represented by tests/golden/reference_example_configs.json.gz: what `load_pipeline_config`
made of each of them (`to_dict()`), written by tests/golden/make_golden_from_reference.py (`configs`)."""
import gzip
import json
import os

import pytest

from torcheasyrec_b200 import example_configs
from torcheasyrec_b200.config import config_to_kwargs, edit_config, load_pipeline_config, parse_text
from torcheasyrec_b200.features import create_features

with gzip.open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden",
                            "reference_example_configs.json.gz"), "rt") as _fh:
    REF_EXAMPLES = json.load(_fh)


def _reference_example(name, tmp_path):
    """The reference's examples/<name>.config as a pipeline config file (the JSON form the loader also accepts)."""
    path = tmp_path / (name + ".json")
    path.write_text(json.dumps(REF_EXAMPLES[name]))
    return str(path)


def test_all_reference_examples_parse(tmp_path):
    assert len(REF_EXAMPLES) >= 17
    for name in REF_EXAMPLES:
        cfg = load_pipeline_config(_reference_example(name, tmp_path))
        assert cfg.model_config.WhichOneof("model") is not None, name
        assert len(cfg.feature_configs) > 0


@pytest.mark.parametrize("name", list(example_configs.GENERATORS))
def test_generated_config_equals_reference_example(name):
    ours = parse_text(example_configs.GENERATORS[name]())
    assert ours.to_dict() == REF_EXAMPLES[name]


@pytest.mark.parametrize("name,groups", [
    ("dlrm_criteo", {"dense": 13, "sparse": 26}),
    ("deepfm_criteo", {"wide": 26, "fm": 26, "deep": 39}),
    ("mmoe_taobao", {"all": 16}),
    ("multi_tower_din_taobao", {"deep": 16, "seq": 6}),
])
def test_generated_configs_structure(name, groups):
    cfg = parse_text(example_configs.GENERATORS[name]())
    got = {g.group_name: len(g.feature_names) for g in cfg.model_config.feature_groups}
    assert got == groups
    assert cfg.train_config.sparse_optimizer.WhichOneof("optimizer") == "adagrad_optimizer"
    assert abs(cfg.train_config.sparse_optimizer.adagrad_optimizer.lr - 0.001) < 1e-12
    assert cfg.train_config.cuda_matmul_allow_tf32 is False  # train.proto field 14 default
    feats = create_features(list(cfg.feature_configs), fg_mode=cfg.data_config.fg_mode)
    assert len(feats) == sum(1 if fc.WhichOneof("feature") != "sequence_feature" else
                             len(fc.sequence_feature.features) for fc in cfg.feature_configs)


def test_text_format_features():
    cfg = parse_text('''
      # comment
      model_dir: 'a' "b"
      train_config { num_steps: 10 sparse_optimizer { sgd_optimizer { lr: 1e-2 } } }
      model_config {
        feature_groups { group_name: "g" feature_names: ["x", "y"] group_type: WIDE }
        dlrm { final { hidden_units: 8 hidden_units: 4 } }
      }
      unknown_block < inner: 3 inner: 4 >
    ''')
    assert cfg.model_dir == "ab"
    assert cfg.train_config.num_steps == 10 and cfg.train_config.save_checkpoints_steps == 1000
    assert cfg.train_config.sparse_optimizer.sgd_optimizer.lr == 0.01
    g = cfg.model_config.feature_groups[0]
    assert g.feature_names == ["x", "y"] and g.group_type == "WIDE"
    assert config_to_kwargs(cfg.model_config.dlrm.final)["hidden_units"] == [8, 4]
    assert cfg.model_config.dlrm.arch_with_sparse is True and not cfg.model_config.dlrm.HasField("dense_mlp")
    assert cfg.unknown_block.inner == [3, 4]
    edit_config(cfg, {"train_config.num_steps": 5, "model_config.feature_groups[0].group_name": "h"})
    assert cfg.train_config.num_steps == 5 and cfg.model_config.feature_groups[0].group_name == "h"


def test_sparse_optimizer_mapping_from_train_config():
    """tzrec/optim/optimizer_builder.py:30-97: every fused optimizer the kernels implement, with clipping."""
    from torcheasyrec_b200.config import parse_text
    from torcheasyrec_b200.kernels import OPT_ADAGRAD, OPT_ADAM, OPT_PARTIAL_ROWWISE_ADAM, OPT_ROWWISE_ADAGRAD, OPT_SGD
    from torcheasyrec_b200.rank_models import sparse_optimizer_from_config

    def spec(body):
        return sparse_optimizer_from_config(parse_text("train_config { sparse_optimizer { %s } }" % body).train_config)

    s = spec("adagrad_optimizer { lr: 0.001 }")
    assert (s.kind, s.max_gradient) == (OPT_ADAGRAD, 0.0) and abs(s.lr - 0.001) < 1e-9
    s = spec("sgd_optimizer { lr: 0.1 gradient_clipping: true max_gradient: 0.5 }")
    assert (s.kind, s.max_gradient) == (OPT_SGD, 0.5)
    s = spec("rowwise_adagrad_optimizer { lr: 0.02 }")
    assert s.kind == OPT_ROWWISE_ADAGRAD
    s = spec("adam_optimizer { lr: 0.01 beta1: 0.8 beta2: 0.95 weight_decay: 0.001 gradient_clipping: true }")
    assert s.kind == OPT_ADAM and abs(s.beta1 - 0.8) < 1e-6 and abs(s.beta2 - 0.95) < 1e-6
    assert abs(s.weight_decay - 0.001) < 1e-9 and s.max_gradient == 1.0        # proto default max_gradient
    s = spec("partial_rowwise_adam_optimizer { lr: 0.01 }")
    assert s.kind == OPT_PARTIAL_ROWWISE_ADAM and s.max_gradient == 0.0


@pytest.mark.parametrize("name", ["dlrm_criteo", "deepfm_criteo", "mmoe_taobao", "multi_tower_din_taobao",
                                  "multi_tower_taobao"])
def test_reference_example_config_runs_unchanged(name, tmp_path):
    """north_star: `examples/*.config` runs unchanged — the reference's own example is loaded (only the table sizes
    are capped, like the reference's --edit_config_json), the model is built and stepped twice on the CPU with the
    oracle as compute; the loss must be finite and move."""
    import sys

    import torch

    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from oracle_backend import OracleKernels

    from torcheasyrec_b200 import functional as Fn
    from torcheasyrec_b200.engine import Pipeline

    pipe = Pipeline(_reference_example(name, tmp_path), device="cpu", max_rows=200, seed=3)
    batch = pipe.synthetic_batch(24, seed=1)
    with Fn.use_backend(OracleKernels()):
        l0 = float(pipe.eager_step(batch))
        l1 = float(pipe.eager_step(batch))
    assert torch.isfinite(torch.tensor([l0, l1])).all()
    assert l1 < l0          # same batch twice: the sparse (Adagrad) and dense (Adam) updates reduce the loss
