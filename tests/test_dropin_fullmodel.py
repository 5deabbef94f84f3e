"""BASELINE config 1 and the true drop-in case (INTEGRATION.md section 2).

CPU: the drop-in MultiModalModel with the full seeded ResNeXt-50 trunk keeps the reference's parameter paths,
attributes and temperature (tests/golden/state_dict_keys.json) and, run on the host, gives the trunk-boundary
activations and image features the unmodified reference gave on the same seeded trunk and images.

GPU: the full model (seeded ResNeXt-50 trunk as the stock torch module + this library's head) through
calculate_contrastive_loss / forward / encode_image against goldens produced by the unmodified reference
(oracle/make_golden_fullmodel.py), flat and spatial (mean, max)."""
import argparse
import json
import os

import numpy as np
import pytest
import torch

from _util import GOLD, O, ROOT, assert_logits_close, golden, t
from oracle.make_golden import case_inputs
from oracle.make_golden_fullmodel import load_trunk, seeded_images, seeded_trunk


def _load_head(model, inp, embedding_type):
    with torch.no_grad():
        if embedding_type == "flat":
            model.image_embed.model.fc.weight.copy_(torch.from_numpy(inp["W"]))
            model.image_embed.model.fc.bias.copy_(torch.from_numpy(inp["b"]))
        else:
            conv = list(model.image_embed.model.children())[-1]
            conv.weight.copy_(torch.from_numpy(inp["W"])[:, :, None, None])
            conv.bias.copy_(torch.from_numpy(inp["b"]))
        model.text_embed.embedding.weight.copy_(torch.from_numpy(inp["table"]))


@pytest.mark.parametrize("embedding_type,sim,fix", [("flat", "mean", False), ("flat", "mean", True), ("spatial", "max", False)])
def test_dropin_full_model_matches_reference_cpu(embedding_type, sim, fix):
    import multimodal_baby_b200 as cv
    name = "fullmodel_flat_b8" if embedding_type == "flat" else "fullmodel_spatial_%s_b8" % sim
    g = golden(name)
    args = argparse.Namespace(embedding_type=embedding_type, embedding_dim=int(g["E"]), normalize_features=True,
                              fix_temperature=fix, temperature=0.07, text_encoder="embedding",
                              cnn_model="resnext50_32x4d", finetune_cnn=False, sim=sim)
    vocab = {str(i): i for i in range(2350)}
    mine = cv.MultiModalModel(cv.VisionEncoder(args, trunk="resnext"), cv.TextEncoder(vocab, 2048, args), args)
    # the trunk parameters sit at torchvision's paths (load_trunk rejects missing or unexpected trunk keys) ...
    load_trunk(mine.image_embed, seeded_trunk(), embedding_type)
    assert len(mine.state_dict()) > 300                    # the whole ResNeXt trunk is in there
    # ... and everything outside the trunk where the reference keeps it
    with open(os.path.join(GOLD, "state_dict_keys.json")) as fh:
        ref = json.load(fh)["%s_fix%d" % (embedding_type, int(fix))]
    ref_keys = [k[len("model."):] for k in ref["state_dict"] if k.startswith("model.")]
    assert sorted(k for k in mine.state_dict() if not k.startswith("image_embed.")) == \
        [k for k in ref_keys if not k.startswith("image_embed.")]
    for attr in ("normalize_features", "sim", "embedding_type", "fix_temperature", "image_embed", "text_embed",
                 "logit_neg_log_temperature"):
        assert hasattr(mine, attr)
    assert isinstance(mine.logit_neg_log_temperature, torch.nn.Parameter) == ref["temperature_is_parameter"] == (not fix)
    assert mine.logit_neg_log_temperature.item() == pytest.approx(ref["temperature_value"])
    # the head parameters are found where the reference keeps them
    w, b = mine._head()
    assert tuple(w.shape) == (512, 2048) and tuple(b.shape) == (512,)
    # trunk boundary on CPU (the trunk is a stock torch module) and the head on top of it: what the reference computed
    inp = case_inputs(int(g["seed"]), int(g["B"]), int(g["E"]), embedding_type)
    _load_head(mine, inp, embedding_type)
    mine.eval()
    x = seeded_images(int(g["seed"]) + 1)
    with torch.no_grad():
        boundary, fmap = cv.split_trunk_forward(mine.image_embed, x, run_head=False)
        feats = O.encode_image(boundary, w, b, embedding_type)
    assert tuple(fmap.shape) == tuple(g["feature_map_shape"])
    assert abs(float(fmap.mean()) - float(g["feature_map_mean"])) <= 1e-5 * abs(float(g["feature_map_mean"]))
    assert abs(float(fmap.abs().max()) - float(g["feature_map_abs_max"])) <= 1e-5 * float(g["feature_map_abs_max"])
    if embedding_type == "flat":
        assert torch.allclose(boundary, fmap.mean((2, 3)), atol=1e-6)
        assert float((boundary[:, :16] - torch.from_numpy(g["pooled_head"])).abs().max()) <= \
            1e-5 * float(np.abs(g["pooled_head"]).max())
        assert float((feats - torch.from_numpy(g["image_features"])).abs().max()) <= 1e-5
    else:
        assert torch.equal(boundary, fmap)
        assert float((feats[:2, :, :2, :2] - torch.from_numpy(g["image_features_slice"])).abs().max()) <= 1e-5
    # the CUDA-only contract: CPU tensors raise instead of silently taking another path
    with pytest.raises(RuntimeError):
        mine.calculate_contrastive_loss(x, t(inp["ids"]), t(inp["lens"]))


def _mirror_model(name, dev):
    import multimodal_baby_b200 as cv
    g = golden(name)
    et, sim = str(g["embedding_type"]), str(g["sim"])
    args = argparse.Namespace(embedding_type=et, embedding_dim=int(g["E"]), normalize_features=True, fix_temperature=True,
                              temperature=0.07, text_encoder="embedding", cnn_model="resnext50_32x4d", finetune_cnn=False,
                              sim=sim)
    vocab = {str(i): i for i in range(2350)}
    m = cv.MultiModalModel(cv.VisionEncoder(args, trunk="resnext"), cv.TextEncoder(vocab, 2048, args), args)
    load_trunk(m.image_embed, seeded_trunk(), et)
    inp = case_inputs(int(g["seed"]), int(g["B"]), int(g["E"]), et)
    _load_head(m, inp, et)
    return g, inp, m.to(dev).eval()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["fullmodel_flat_b8", "fullmodel_spatial_mean_b8", "fullmodel_spatial_max_b8"])
def test_full_model_matches_reference_golden(name):
    torch.backends.cudnn.allow_tf32 = False; torch.backends.cuda.matmul.allow_tf32 = False
    dev = "cuda"
    g, inp, m = _mirror_model(name, dev)
    x = seeded_images(int(g["seed"]) + 1).to(dev)
    ids, lens = t(inp["ids"], dev), t(inp["lens"], dev)
    with torch.no_grad():
        out = m.calculate_contrastive_loss(x, ids, lens)
        lpi, lpt = m(x, ids, lens)
        feats, fmap = m.encode_image(x)
    # the trunk itself (stock torch on the GPU vs the reference on CPU)
    assert tuple(fmap.shape) == tuple(g["feature_map_shape"])
    assert abs(float(fmap.mean()) - float(g["feature_map_mean"])) <= 1e-3 * abs(float(g["feature_map_mean"]))
    assert abs(out[0].item() - float(g["loss"])) <= 1e-3 * abs(float(g["loss"]))
    assert abs(out[3].item() - float(g["image_entropy"])) <= 2e-3 and abs(out[4].item() - float(g["text_entropy"])) <= 2e-3
    assert abs(out[1].item() - float(g["image_accuracy"])) <= 0.125 + 1e-6       # 8 rows, near-tied random-init logits
    assert_logits_close(out[5].cpu().numpy(), g["logits_per_image"])
    assert_logits_close(out[6].cpu().numpy(), g["logits_per_text"])
    assert_logits_close(lpi.cpu().numpy(), g["logits_per_image"])
    assert_logits_close(lpt.cpu().numpy(), g["logits_per_text"])
    if "image_features" in g:
        assert float((feats.cpu() - torch.from_numpy(g["image_features"])).abs().max()) <= 6e-3
        assert float((fmap.mean((2, 3))[:, :16].cpu() - torch.from_numpy(g["pooled_head"])).abs().max()) <= \
            1e-3 * float(np.abs(g["pooled_head"]).max())
    else:
        assert float((feats[:2, :, :2, :2].cpu() - torch.from_numpy(g["image_features_slice"])).abs().max()) <= 6e-3


@pytest.mark.gpu
def test_full_model_training_step_updates_only_the_head():
    """frozen trunk (finetune_cnn=False, multimodal.py:175-177): calculate_contrastive_loss + backward leaves gradients on
    fc / embedding only, and they equal the head-only step on the trunk-boundary features."""
    import multimodal_baby_b200 as cv
    dev = "cuda"
    g, inp, m = _mirror_model("fullmodel_flat_b8", dev)
    m.train(); m.image_embed.model.eval()                  # BatchNorm on its running statistics, as in the golden
    x = seeded_images(int(g["seed"]) + 1).to(dev)
    ids, lens = t(inp["ids"], dev), t(inp["lens"], dev)
    out = m.calculate_contrastive_loss(x, ids, lens)
    out[0].backward()
    with_grad = sorted(n for n, p in m.named_parameters() if p.grad is not None)
    assert with_grad == ["image_embed.model.fc.bias", "image_embed.model.fc.weight", "text_embed.embedding.weight"]
    with torch.no_grad():
        pooled, _ = cv.split_trunk_forward(m.image_embed, x, run_head=False)
    W = m.image_embed.model.fc.weight.detach().clone().requires_grad_(True)
    b = m.image_embed.model.fc.bias.detach().clone().requires_grad_(True)
    tab = m.text_embed.embedding.weight.detach().clone().requires_grad_(True)
    loss2 = cv.ops.flat_contrastive_loss(pooled, ids, lens, W, b, tab, m.logit_neg_log_temperature, True)[0]
    loss2.backward()
    assert abs(loss2.item() - out[0].item()) <= 1e-6 * abs(out[0].item())
    assert torch.equal(W.grad, m.image_embed.model.fc.weight.grad)
    assert torch.equal(tab.grad, m.text_embed.embedding.weight.grad)
