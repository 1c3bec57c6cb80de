"""The experiment driver's host logic (no GPU): YAML forms, grid expansion, attribute access - checked on written-out
examples."""
import copy

import pytest

from deep_cbrs_amar_renaissance_b200 import experiment as ex
from deep_cbrs_amar_renaissance_b200.utilities.utils import make_grid, nested_dict_update


def test_yaml_reads_the_float_forms_of_yaml_1_2(tmp_path):
    p = tmp_path / "c.yaml"
    p.write_text("a: 1e-4\nb: [1e-5, 1e-3, 0.5, 3]\nc: '1e-4'\nd: null\ne: True\nf: 1.5e+2\n")
    cfg = ex.load_yaml(str(p))
    assert cfg == dict(a=1e-4, b=[1e-5, 1e-3, 0.5, 3], c='1e-4', d=None, e=True, f=150.0)
    assert isinstance(cfg["a"], float) and isinstance(cfg["b"][3], int)


def test_make_grid_and_update_written_out():
    grid = {"model": {"name": ["basic.BasicGCN", "basic.BasicGAT"], "n_hiddens": [[8, 8]], "l2_regularizer": [1e-5, 1e-4]},
            "dataset": {"type_adjacency": ["unary"]}}
    got = make_grid(grid)
    assert len(got) == 4
    assert got[0] == {"model": {"name": "basic.BasicGCN", "n_hiddens": [8, 8], "l2_regularizer": 1e-5}, "dataset": {"type_adjacency": "unary"}}
    assert [g["model"]["l2_regularizer"] for g in got] == [1e-5, 1e-4, 1e-5, 1e-4]   # last listed key varies fastest
    with pytest.raises(ValueError):
        make_grid({"model": {"name": "basic.BasicGCN"}})
    base = {"model": {"name": "x", "embedding_dim": 16}, "seed": 42}
    out = nested_dict_update(copy.deepcopy(base), got[1])
    assert out["model"] == {"name": "basic.BasicGCN", "embedding_dim": 16, "n_hiddens": [8, 8], "l2_regularizer": 1e-4}
    assert out["seed"] == 42 and out["dataset"] == {"type_adjacency": "unary"}


def test_config_attribute_access():
    c = ex.Config({"model": {"name": "basic.BasicGCN", "n_hiddens": [8, 8]}, "seed": 1})
    assert c.model.name == "basic.BasicGCN" and c.seed == 1 and c.plain() == {"model": {"name": "basic.BasicGCN", "n_hiddens": [8, 8]}, "seed": 1}
    with pytest.raises(AttributeError):
        c.nope
