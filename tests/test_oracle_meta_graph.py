"""Pins the CPU oracle to the graphs the reference itself serialized: the forward sub-graphs of the shipped
`models/*.ckpt.meta` MetaGraphDefs (tests/golden/meta/*.json, extracted by scripts/make_meta_fixture.py) are executed op by
op by an independent numpy interpreter (tests/tf_graph_interp.py) on the shipped checkpoint weights, and the oracle must
give the same numbers - final output and every layer - in float64.  That fixes, from reference-held bytes: op order and
wiring, SAME padding, NHWC / HWIO, the [B2, A1] concat order, DepthToSpace block sizes, Up-PS bias-without-activation,
R-CNN1 without bias, the PReLU form, and dropout = identity at keep 1 (both dropout sub-graph generations)."""
import os

import numpy as np
import pytest
import torch

import dcscn_oracle as O
from conftest import GOLDEN, MODEL_FLAGS, ROOT, load_golden_weights
from tf_graph_interp import GraphInterpreter

META_MODELS = ["dcscn_L7_F32to8_G1.20_NIN_A24_B8_PS_R1F32", "dcscn_L7_F32to8_G1.20_Sc3_NIN_A24_B8_PS_R1F32",
               "dcscn_L7_F32to8_G1.20_Sc4_NIN_A24_B8_PS_R1F32", "dcscn_L7_F32to8_G1.20_Sc4_NIN_A24_B8_PS_DS_R1F32"]


def _fixture(model):
    return os.path.join(GOLDEN, "meta", model + ".json")


@pytest.mark.parametrize("model", META_MODELS)
def test_variables_of_the_shipped_graph_are_the_oracles(model):
    g = GraphInterpreter(_fixture(model))
    cfg = O.OracleConfig(**MODEL_FLAGS[model])
    shapes = g.variables()
    expect = {}
    for scope, k, cin, cout, bias, prelu in O.layer_table(cfg):
        base = scope.split("/")[-1]
        if cfg.depthwise_separable:      # the dead conv_W is not on the forward path (tf_graph.py:183)
            expect[scope + "/depthwise_W"] = (k, k, cin, 1)
            expect[scope + "/pointwise_W"] = (1, 1, cin, cout)
        else:
            expect[scope + "/conv_W"] = (k, k, cin, cout)
        if bias:
            expect[scope + "/conv_B"] = (cout,)
        if prelu:
            expect["%s/prelu/%s_prelu" % (scope, base)] = (cout,)
    assert shapes == expect


@pytest.mark.parametrize("model", META_MODELS)
def test_oracle_equals_the_shipped_graph_executed_op_by_op(model):
    g = GraphInterpreter(_fixture(model))
    kw = MODEL_FLAGS[model]
    cfg = O.OracleConfig(**kw)
    w = load_golden_weights(model)
    s = cfg.scale
    rs = np.random.RandomState(len(model))
    x = rs.rand(2, 9, 11, 1) * 255
    x2 = rs.rand(2, 9 * s, 11 * s, 1) * 255
    L = cfg.layers
    # the node that carries each layer's output (post-dropout where the graph has dropout): two dropout generations
    def out_of(scope):
        for cand in (scope + "/dropout/mul_1", scope + "/dropout/mul"):
            if cand in g.nodes and (cand.endswith("mul_1") or (scope + "/dropout/mul_1") not in g.nodes):
                return cand
        raise KeyError(scope)
    fetch = {"CNN%d" % (i + 1): out_of("CNN%d" % (i + 1)) for i in range(L)}
    fetch.update({"A1": out_of("A1"), "B1": out_of("B1"), "B2": out_of("B2"), "Up-PS": "Up-PS/DepthToSpace"})
    if s == 4:
        fetch["Up-PS2"] = "Up-PS2/DepthToSpace"
    res = g.run({"x": x, "x2": x2, "dropout_keep_rate": 1.0}, w, fetch=[g.root] + list(fetch.values()))
    y64, inter = O.Oracle(cfg, w, torch.float64).forward(x, x2, return_intermediates=True)
    for name, node in fetch.items():
        ref = res[node]
        assert inter[name].shape == ref.shape, name
        assert np.abs(inter[name] - ref).max() <= 1e-9 * max(1.0, np.abs(ref).max()), name
    assert np.abs(y64 - res[g.root]).max() <= 1e-9 * max(1.0, np.abs(y64).max())
    # wiring facts read straight off the serialized graph
    cat = g.nodes["Concat/H_concat"]["input"][:-1]
    assert cat == [fetch["CNN%d" % (i + 1)] for i in range(L)]
    assert g.nodes["Concat2"]["input"][:-1] == [fetch["B2"], fetch["A1"]]          # B2 first (DCSCN.py:281)
    assert "R-CNN1/conv_B" not in g.nodes and "Up-PS/Up-PS_CNN/prelu/Relu" not in g.nodes
    assert set(g.nodes[g.root]["input"]) == {"R-CNN1/R-CNN1_conv", "x2"}


@pytest.mark.parametrize("model", META_MODELS)
def test_fixture_is_what_the_reference_ships(model, tmp_path):
    """Re-extract the sub-graph from the reference's shipped .meta (stored byte for byte, xz-compressed, under
    tests/golden/models) and require the committed fixture."""
    import importlib.util
    import json
    import lzma
    spec = importlib.util.spec_from_file_location("make_meta_fixture", os.path.join(ROOT, "scripts", "make_meta_fixture.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    with lzma.open(os.path.join(GOLDEN, "models", model + ".ckpt.meta.xz")) as f:
        nodes, _ = mod.graph_nodes(f.read())
    root, keep = mod.forward_subgraph(nodes)
    doc = json.load(open(_fixture(model)))
    assert doc["root"] == root and doc["nodes"] == json.loads(json.dumps(keep))
