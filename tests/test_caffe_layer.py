"""The reference-facing plugin surface: prototxt parsing (CPU) and the layer vs the oracle (GPU)."""
import os

import numpy as np
import pytest

from npairloss_b200 import caffe_layer, synth

REF_USAGE_BLOCK = '''
layer {
    bottom: "pool5/7x7_s1"
    name: "loss3/pool5/7x7_s1/norm"
    type: "L2Normalize"
    top: "loss3/pool5/7x7_s1/norm"
}
.
.
layer {
    bottom: "loss3/pool5/7x7_s1/norm"
    #bottom: "pool5/7x7_s1"
    bottom: "label_type_mb"
    name: "loss3/type_mb"
    type: "NPairMultiClassLoss"
    top: "loss3/type_npair_mc"
    top: "loss3/type_npair_mc_retrieve_top1"
    top: "loss3/type_npair_mc_retrieve_top5"
    top: "loss3/type_npair_mc_retrieve_top10"
    top: "loss3/feature_asum"
    loss_weight: 1
    loss_weight: 1
    loss_weight: 1
    loss_weight: 1
    loss_weight: 1
    npair_loss_param {
        margin_ident: 0.0
        margin_diff: -0.05
        identsn: -0.0
        diffsn: -0.3 # inert for absolute selection
        ap_mining_region: GLOBAL
        ap_mining_method: RELATIVE_HARD
        an_mining_region: LOCAL
        an_mining_method: HARD # RELATIVE_HARD
    }
    #loss_weight: 1
    #include {
    #    phase: TRAIN
    #}
}
'''


def test_parse_reference_usage_block():
    """The layer block in the format of usage/def.prototxt:115-151 (comments, '.' elision marks, a foreign layer)."""
    p = caffe_layer.parse_only(REF_USAGE_BLOCK)
    assert p["n_layers"] == 2 and p["num_tops"] == 5 and p["n_loss_weights"] == 5
    assert p["margin_ident"] == 0.0 and p["margin_diff"] == pytest.approx(-0.05) and p["diffsn"] == pytest.approx(-0.3)
    assert p["identsn"] == 0.0 and np.signbit(np.float32(p["identsn"]))           # -0.0 survives
    assert (p["ap_region"], p["ap_method"], p["an_region"], p["an_method"]) == (0, 3, 1, 0)


def test_parse_reference_prototxt_file_unchanged():
    """usage/def.prototxt of the reference, stored byte for byte as tests/golden/usage_def.prototxt."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "usage_def.prototxt")
    txt = open(path, encoding="utf-8", errors="replace").read()
    p = caffe_layer.parse_only(txt)
    assert p["num_tops"] == 5 and p["n_loss_weights"] == 5
    assert (p["ap_region"], p["ap_method"], p["an_region"], p["an_method"]) == (0, 3, 1, 0)
    assert p["margin_diff"] == pytest.approx(-0.05)


def test_proto_defaults_and_errors():
    p = caffe_layer.parse_only('layer { type: "NPairMultiClassLoss" bottom: "a" bottom: "b" top: "l" }')
    # caffe.proto:4-7,19-22
    assert (p["margin_ident"], p["margin_diff"], p["identsn"], p["diffsn"]) == (0.0, 0.0, -1.0, -1.0)
    assert (p["ap_region"], p["ap_method"], p["an_region"], p["an_method"]) == (1, 2, 1, 2)
    with pytest.raises(ValueError):
        caffe_layer.parse_only('layer { type: "NPairMultiClassLoss" npair_loss_param { ap_mining_method: SEMI_HARD } }')
    with pytest.raises(ValueError):
        caffe_layer.parse_only('layer { type: "Other" }')


@pytest.mark.gpu
def test_layer_matches_oracle_on_usage_block(oracle):
    Q, D = 120, 1024                     # the reference's own per-rank batch and embedding dim (usage/def.prototxt:21-27,115-123)
    x, lab = synth.make_inputs(Q, D, seed=42, noise=2.5)
    layer = caffe_layer.Layer(REF_USAGE_BLOCK, Q, D)
    assert layer.type() == "NPairMultiClassLoss" and layer.num_tops == 5
    assert all(layer.loss_weight(t) == 1.0 for t in range(5))
    layer.bottom_data(0)[:] = x.ravel()
    layer.bottom_data(1)[:] = lab
    tops, weighted = layer.forward()
    layer.backward()
    dx = layer.bottom_diff().copy()
    cfg = oracle.make_config(Q, D, faithful_sorts=1, **synth.USAGE_MINING)
    tops_o, dx_o = oracle.step_world(x, lab, cfg, 1.0)
    np.testing.assert_allclose(tops[0], tops_o[0, 0], rtol=2e-5)
    assert abs(tops[1] - tops_o[0, 1]) * Q <= 1 and abs(tops[3] - tops_o[0, 3]) * Q <= 1
    np.testing.assert_allclose(tops[4], tops_o[0, 4], rtol=2e-6)
    assert weighted == pytest.approx(sum(tops), rel=1e-6)          # five loss_weight: 1 entries (usage/def.prototxt:132-136)
    assert np.linalg.norm(dx - dx_o) <= 5e-5 * np.linalg.norm(dx_o)
    # a second step with new data reuses the same layer (batch size frozen at setup)
    x2, _ = synth.make_inputs(Q, D, seed=43, noise=2.5)
    layer.bottom_data(0)[:] = x2.ravel()
    t2 = layer.step_host()
    assert t2[0] != tops[0]
    layer.close()


@pytest.mark.gpu
def test_layer_contract(oracle):
    mining = synth.DEFAULT_MINING
    with pytest.raises(caffe_layer.LayerError):                     # MaxTopBlobs = 5 (.hpp:34)
        caffe_layer.Layer(caffe_layer.layer_prototxt(mining, 5).replace('top: "loss3/feature_asum"', 'top: "a"\n top: "b"'), 8, 4)
    layer = caffe_layer.Layer(caffe_layer.layer_prototxt(mining, 3, loss_weights=False), 16, 8)
    x, lab = synth.make_inputs(16, 8, seed=3)
    layer.bottom_data(0)[:] = x.ravel()
    layer.bottom_data(1)[:] = lab
    tops, weighted = layer.forward()
    t_o, _ = oracle.forward(x, lab, oracle.make_config(16, 8, num_tops=3))
    np.testing.assert_allclose(tops[:3], t_o[:3], rtol=2e-5)
    assert weighted == 0.0                                          # LossLayer::LayerSetUp is not chained: no implicit loss_weight (Q13)
    with pytest.raises(caffe_layer.LayerError) as e:                # no CPU path, loudly
        layer.forward_cpu_mode()
    assert "no CPU path" in str(e.value)
    layer.close()


REF_TRAIN_NET = '''
name: "GoogleNet"
layer {
    name: "data_mb"
    type: "MultibatchData"
    top: "data_mb"
    top: "label_type_mb"
    include { phase: TRAIN }
    multi_batch_data_param {
        batch_size: 120
        shuffle: true
        identity_num_per_batch: 60
        img_num_per_identity: 2
        rand_identity: true
    }
}
layer {
    name: "data_mb"
    type: "MultibatchData"
    top: "data_mb"
    top: "label_type_mb"
    include { phase: TEST }
    multi_batch_data_param { batch_size: 30 identity_num_per_batch: 15 img_num_per_identity: 2 }
}
.
.
''' + REF_USAGE_BLOCK


def test_train_net_prototxt_is_parsed():
    """The data-layer block format of usage/def.prototxt:2-59 next to the loss block: both phases, nested messages captured."""
    p = caffe_layer.parse_only(REF_TRAIN_NET)
    assert p["n_layers"] == 4 and p["num_tops"] == 5


@pytest.mark.gpu
def test_solver_loop_trains_through_the_reference_chain():
    """SURVEY 8f-4: MultibatchData -> [synthetic trunk] -> L2Normalize -> NPairMultiClassLoss for a few hundred SGD iterations with the
    solver settings of usage/solver.prototxt (momentum 0.9, step policy); the learning rate is scaled for the toy embedding table.
    The loss must come down and top-1 retrieval must go up: forward, backward and both layers' gradients act together."""
    solver = "base_lr: 4000\nlr_policy: \"step\"\nstepsize: 200\ngamma: 0.5\nmomentum: 0.9\nweight_decay: 0.00002\ndisplay: 20\nmax_iter: 400\nsolver_mode: GPU\n"
    log = caffe_layer.solver_run(REF_TRAIN_NET, solver, feature_dim=64, num_identities=240, imgs_per_identity=4, seed=3, noise=2.5)
    assert len(log) >= 20 and log[0, 0] == 0 and log[-1, 0] == 399
    first, last = log[:3].mean(axis=0), log[-3:].mean(axis=0)
    print("solver loop: loss", first[2], "->", last[2], " top1", first[3], "->", last[3])
    assert np.isfinite(log).all()
    assert last[2] < 0.8 * first[2], (first[2], last[2])
    assert last[3] > first[3] + 0.1, (first[3], last[3])
    assert abs(last[6] - first[6]) < 0.2 * first[6]          # feature_asum of unit rows stays put
