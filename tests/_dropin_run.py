"""Helper executed in a fresh interpreter by tests/test_dropin_reference.py (install() rewires
sys.modules, so it must not run inside the pytest process).

    python tests/_dropin_run.py <reference_root> <device>

Imports the REFERENCE's own models/{classifier,segmenter,autoencoder}.py — from the bytecode
build product oracle/_ref/pyref — on top of sonet_b200's networks/layers/losses/som/index_max,
and on a CUDA device runs their unmodified
Model.set_input()/test_model() against the golden vectors the reference itself produced."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "so-net_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

ref_root, device = sys.argv[1], sys.argv[2]

import sonet_b200.install as inst  # noqa: E402
from sonet_b200 import networks, ops, synth  # noqa: E402

inst.install(ref_root)
from models import autoencoder, classifier, segmenter  # noqa: E402  (the reference's files)
import models.networks as n  # noqa: E402

assert n is networks and classifier.networks is networks
for mod in (classifier, segmenter, autoencoder):
    assert os.path.abspath(mod.__file__).startswith(os.path.abspath(ref_root)), mod.__file__
print("reference Model files from", os.path.dirname(classifier.__file__))

if device == "cpu":
    # construction works anywhere; the CUDA-only hot path must refuse CPU tensors loudly
    opt = synth.make_opt("classifier", batch_size=2, input_pc_num=64)
    m = classifier.Model(opt)
    assert type(m.encoder).__module__ == "sonet_b200.networks"
    inp = synth.synth_inputs(2, 64)
    m.set_input(inp["pc"], inp["sn"], inp["label"], inp["node"], inp["node_knn_I"])
    try:
        m.test_model()
        raise SystemExit("expected the CUDA-only encoder to refuse CPU tensors")
    except RuntimeError as e:
        assert "no CPU fallback" in str(e)
    s = segmenter.Model(synth.make_opt("segmenter", batch_size=2, input_pc_num=64))
    assert type(s.segmenter).__module__ == "sonet_b200.networks"
    a = autoencoder.Model(synth.make_opt("autoencoder", batch_size=2, input_pc_num=64))
    assert type(a.chamfer_criteria).__module__ == "sonet_b200.losses"
    print("DROPIN_OK")
    raise SystemExit(0)

from helpers import (assert_close, assert_golden, build_states, golden, golden_case,  # noqa: E402
                     to_ref_slot_order)
from oracle import oracle  # noqa: E402  (checker only)


def gpu_opt(opt):
    opt.device = torch.device(device)
    opt.gpu_id = torch.device(device).index or 0
    return opt


def check_encoder(g, enc, opt):
    assert np.array_equal(oracle.canon_sets(enc.min_idx.cpu(), opt.k).numpy(), g["knn_sets"])
    for name in ("som_node", "first_pn_out_masked_max", "final_pn_out", "feature"):
        assert_golden(g, name, getattr(enc, name))
    if opt.som_k >= 2:
        assert_golden(g, "knn_feature_1", enc.knn_feature_1)


# ---- models/classifier.py:64-105, unmodified ------------------------------------------------------
g = golden("classifier_b2_n256")
opt, inp, seed = golden_case(g, "classifier")
st = build_states("classifier", opt, seed)
m = classifier.Model(gpu_opt(opt))
assert type(m.encoder).__module__ == "sonet_b200.networks"
m.encoder.load_state_dict(st["encoder"])
m.classifier.load_state_dict(st["head"])
m.set_input(inp["pc"], inp["sn"], inp["label"], inp["node"], inp["node_knn_I"])
c0 = ops.LAUNCHES
m.test_model()                       # the reference calls this WITHOUT torch.no_grad()
assert ops.LAUNCHES - c0 >= 10, "the reference's test_model did not reach the CUDA kernels"
assert m.score.grad_fn is None
check_encoder(g, m.encoder, opt)
assert_golden(g, "score", m.score)
assert torch.isfinite(m.loss)
print("classifier.Model ok: %d kernel-API calls" % (ops.LAUNCHES - c0))

# ---- models/segmenter.py:66-135, unmodified (per-point torch.gather + reference head signature) ----
g = golden("segmenter_b2_n128")
opt, inp, seed = golden_case(g, "segmenter")
st = build_states("segmenter", opt, seed)
m = segmenter.Model(gpu_opt(opt))
m.encoder.load_state_dict(st["encoder"])
m.segmenter.load_state_dict(st["head"])
seg = torch.zeros(int(g["B"]), int(g["N"]), dtype=torch.int64)
for rep in range(2):                 # 2nd forward: the encoder has learnt that first_pn_out is read
    m.set_input(inp["pc"], inp["sn"], inp["label"], seg, inp["node"], inp["node_knn_I"])
    m.test_model()
    check_encoder(g, m.encoder, opt)
    assert_golden(g, "score_segmenter", m.score_segmenter)
    assert_golden(g, "first_pn_out",
                  to_ref_slot_order(m.encoder.first_pn_out, m.encoder.min_idx, g, opt.k))
assert torch.isfinite(m.loss_segmenter)
print("segmenter.Model ok")

# ---- models/autoencoder.py:56-126, unmodified ------------------------------------------------------
g = golden("autoencoder_b2_n256")
opt, inp, seed = golden_case(g, "autoencoder")
st = build_states("autoencoder", opt, seed)
m = autoencoder.Model(gpu_opt(opt))
assert type(m.chamfer_criteria).__module__ == "sonet_b200.losses"
m.encoder.load_state_dict(st["encoder"])
m.decoder.load_state_dict(st["head"])
m.set_input(inp["pc"], inp["sn"], inp["label"], inp["node"], inp["node_knn_I"])
m.test_model()
check_encoder(g, m.encoder, opt)
assert_golden(g, "predicted_pc", m.predicted_pc)
assert_close(m.loss_chamfer, g["loss_chamfer"], "loss_chamfer")
assert_close(m.loss, g["loss"], "loss")
print("autoencoder.Model ok")
print("DROPIN_OK")
