"""CPU suite (-m "not gpu"): host-side mirror of the reference interface and the C-ABI surface.
No compute call is made (there is no CPU path); what is checked is everything around it:
symbol export, prototypes, state_dict key parity with the reference, tokenisation, argument
semantics and loud failure modes."""
import argparse
import ctypes
import json
import os
import re

import pytest
import torch

from _util import GOLD, ROOT

import multimodal_baby_b200 as cv


def _args(**kw):
    d = dict(embedding_type="flat", embedding_dim=64, normalize_features=True, fix_temperature=False,
             temperature=0.07, text_encoder="embedding", sim="mean", dropout_o=0.0)
    d.update(kw)
    return argparse.Namespace(**d)


def _lit(**kw):
    a = _args(**kw)
    vocab = {"<pad>": 0, "<unk>": 1, "<sos>": 2, "<eos>": 3, **{"w%d" % i: i for i in range(4, 2350)}}
    return cv.MultiModalLitModel(cv.VisionEncoder(a, trunk="pooled"), cv.TextEncoder(vocab, 2048, a), a,
                                 vocab=vocab)


# ------------------------------------------------------------------------------ C ABI surface
def test_library_exports_every_declared_symbol_at_the_header_abi_version():
    hdr = open(os.path.join(ROOT, "include", "cvcl_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(cvcl_[a-z0-9_]+)\s*\(", hdr)))
    assert len(declared) >= 25
    lib = ctypes.CDLL(cv._cabi.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), "libcvcl_b200.so does not export %s" % name
    # the ctypes prototype table covers exactly the header
    assert sorted(cv._cabi.PROTOTYPES) == declared
    # library, bindings and header agree on the ABI version (6: per-row diagonal of G in the InfoNCE backward)
    header_abi = int(re.search(r"#define CVCL_ABI_VERSION (\d+)", hdr).group(1))
    assert cv._cabi.load().cvcl_abi_version() == cv._cabi.ABI_VERSION == header_abi == 6


def test_library_links_no_torch_and_is_sm100a():
    import subprocess
    out = subprocess.run(["ldd", cv._cabi.LIB_PATH], capture_output=True, text=True).stdout
    assert "libtorch" not in out and "libc10" not in out
    cu = subprocess.run(["cuobjdump", "-lelf", cv._cabi.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in cu


def test_sass_shows_the_sm100a_instructions_the_design_claims():
    """static evidence (no GPU): the built library contains tcgen05 MMAs with TMEM loads, TMA tensor loads and
    stores, the 1-D bulk copy of the streaming eval kernel, cluster barriers, 16-byte fp32 vector atomics, and
    the system-scope release / acquire accesses of the peer-memory barriers (DESIGN sections 3 and 5)."""
    import subprocess
    sass = subprocess.run(["cuobjdump", "-sass", cv._cabi.LIB_PATH], capture_output=True, text=True).stdout
    for mnemonic in ("UTCHMMA", "LDTM", "UTMALDG.2D", "UTMASTG.2D", "UBLKCP", "UCGABAR_WAIT", "SYNCS.PHASECHK",
                     "REDG.E.ADD.F32x4", "STG.E.STRONG.SYS", "LDG.E.STRONG.SYS", "LDG.E.128.STRONG.SYS",
                     "MEMBAR.SC.SYS"):
        assert mnemonic in sass, "missing %s in the SASS of libcvcl_b200.so" % mnemonic
    names = subprocess.run(["cuobjdump", "-elf", cv._cabi.LIB_PATH], capture_output=True, text=True).stdout
    for kernel in ("peer_allreduce_push_f32_kernel", "peer_allgather_push_kernel", "eval_nway_stream_kernel",
                   "text_encoder_flat_wide_kernel", "featgrad_finish_kernel", "gradcam_cam_kernel",
                   "gemm_bf16_persistent_kernel",
                   # round 2: the one-kernel step, the one-pass similarity epilogue, compacted spatial backward, eval forms
                   "flat_step_kernel", "EpiSimStats1P", "token_row_offsets_kernel", "token_rows_scatter_kernel",
                   "spatial_pool_bwd_kernel", "linear_f32_kernel", "row_argmax_f32_kernel", "normalize_rows_f32_kernel"):
        assert kernel in names, "kernel %s not in the library" % kernel
    # the one-kernel step itself issues tcgen05 MMAs, TMEM loads and TMA traffic (not a wrapper around other launches)
    import re
    body = sass[sass.index("flat_step_kernel"):]
    nxt = re.search(r"\n\s*Function : ", body[100:])
    body = body[:100 + nxt.start()] if nxt else body
    for mnemonic in ("UTCHMMA", "LDTM", "UTMALDG.2D", "UTMASTG.2D", "STG.E.STRONG.SYS"):
        assert mnemonic in body, "flat_step_kernel lacks %s" % mnemonic


def test_missing_library_is_loud(monkeypatch):
    monkeypatch.setattr(cv._cabi, "_lib", None)
    with pytest.raises(cv.CvclLibraryMissing):
        cv._cabi.load("/nonexistent/libcvcl_b200.so")
    monkeypatch.undo()
    cv._cabi.load()


def test_cpu_tensors_raise_no_fallback():
    lit = _lit()
    ids, lens = lit.tokenize(["w5 w6"])
    with pytest.raises(RuntimeError, match="no CPU"):
        lit(torch.randn(2, 2048), ids, lens)
    with pytest.raises(RuntimeError, match="no CPU"):
        lit.model.calculate_contrastive_loss(torch.randn(1, 2048), ids, lens)
    with pytest.raises(RuntimeError, match="no CPU"):
        cv.ops.eval_nway(torch.randn(8, 64), torch.randn(2, 64), None, 4, True, 0.0)


def test_package_never_imports_oracle():
    pkg = os.path.join(ROOT, "multimodal-baby_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), fn


# ------------------------------------------------------------------------------ reference interface
@pytest.mark.parametrize("et", ["flat", "spatial"])
@pytest.mark.parametrize("fix", [False, True])
def test_state_dict_keys_match_reference(et, fix):
    with open(os.path.join(GOLD, "state_dict_keys.json")) as fh:
        g = json.load(fh)["%s_fix%d" % (et, int(fix))]
    lit = _lit(embedding_type=et, fix_temperature=fix)
    assert sorted(lit.state_dict().keys()) == g["state_dict"]
    assert sorted(n for n, p in lit.named_parameters() if p.requires_grad) == g["trainable"]
    s = lit.model.logit_neg_log_temperature
    assert isinstance(s, torch.nn.Parameter) == g["temperature_is_parameter"]
    assert abs(float(s) - g["temperature_value"]) < 1e-7
    assert s.dim() == 0 and s.dtype == torch.float32
    # tied LM head and shared encoders, as in the reference
    assert lit.language_model.output_layer.weight is lit.text_encoder.embedding.weight
    assert lit.model.image_embed is lit.vision_encoder and lit.model.text_embed is lit.text_encoder


def test_tokenize_matches_reference_golden():
    """tokenize == the reference's tokenize on the same texts, with the entries of the reference's vocab.json that
    these texts use (tokenize_vocab.json): <sos> / <eos>, <unk> for an unknown word, truncation to 25, padding."""
    vocab = cv.load_vocab(os.path.join(GOLD, "tokenize_vocab.json"))
    with open(os.path.join(GOLD, "tokenize.json")) as fh:
        g = json.load(fh)
    a = _args()
    lit = cv.MultiModalLitModel(cv.VisionEncoder(a, trunk="pooled"), cv.TextEncoder(vocab, 2048, a), a,
                                vocab=vocab)
    ids, lens = lit.tokenize(g["texts"])
    assert ids.dtype == torch.int64 and lens.dtype == torch.int64
    assert ids.tolist() == g["ids"] and lens.tolist() == g["lens"]
    one, n = lit.tokenize(g["texts"][0])            # a bare string is one utterance
    assert one.tolist() == [g["ids"][0]] and n.tolist() == [g["lens"][0]]


def test_unsupported_configurations_raise():
    with pytest.raises(NotImplementedError):
        cv.TextEncoder({"<pad>": 0}, 2048, _args(text_encoder="lstm"))
    with pytest.raises(NotImplementedError):
        _lit(lambda_lm=0.5)
    lit = _lit(dropout_o=0.3)
    lit.train()
    ids, lens = lit.tokenize(["w5"])
    with pytest.raises(NotImplementedError, match="dropout_o"):
        lit.model.encode_text(ids, lens)
    with pytest.raises(NotImplementedError):
        cv.VisionEncoder(_args(vit_dino=True), trunk="pooled")


def test_defaults_follow_reference_argparse():
    p = argparse.ArgumentParser()
    cv.MultiModalModel.add_to_argparse(p)
    a = p.parse_args([])
    assert (a.embedding_type, a.embedding_dim, a.normalize_features, a.sim, a.temperature,
            a.fix_temperature) == ("flat", 128, False, "max", 0.07, False)   # multimodal.py:17-29


def test_trunk_split_keeps_reference_semantics():
    """split_trunk_forward(run_head=True) == the stock module forward, and run_head=False hands the
    kernels the input of the head (flat: pooled activations; spatial: the layer4 map)."""
    a = _args()
    ve = cv.VisionEncoder(a, trunk="pooled")
    x = torch.randn(3, 2048)
    feats, fmap = cv.split_trunk_forward(ve, x, run_head=True)
    assert torch.allclose(feats, ve.model.fc(x)) and torch.equal(fmap, x)
    pooled, fmap2 = cv.split_trunk_forward(ve, x, run_head=False)
    assert torch.equal(pooled, x) and isinstance(ve.model.fc, torch.nn.Linear)
    vs = cv.VisionEncoder(_args(embedding_type="spatial"), trunk="pooled")
    xs = torch.randn(2, 2048, 7, 7)
    b, f = cv.split_trunk_forward(vs, xs, run_head=False)
    assert torch.equal(b, xs) and torch.equal(f, xs)


def test_full_resnext_trunk_split_matches_torchvision():
    a = _args()
    ve = cv.VisionEncoder(a, trunk="resnext").eval()
    x = torch.randn(1, 3, 64, 64)
    with torch.no_grad():
        pooled, fmap = cv.split_trunk_forward(ve, x, run_head=False)
        ref = ve.model(x)
        assert pooled.shape == (1, 2048) and fmap.shape[1] == 2048
        assert torch.allclose(ve.model.fc(pooled), ref, atol=1e-5)
    assert not any(p.requires_grad for n, p in ve.model.named_parameters() if not n.startswith("fc."))
    assert all(p.requires_grad for p in ve.model.fc.parameters())


# ------------------------------------------------------------------------------ bench.py contract
def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the B200 arm) prints ONE JSON line with
    the metric of BASELINE.json, its own cpu_baseline and a zero-copy e2e object; no GPU needed."""
    import json
    import subprocess
    import sys
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3",
                          "--warmup", "3", "--pairs-per-gpu", "64"], capture_output=True, text=True, timeout=600,
                         cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert d["impl"] == "reference" and d["metric"] == base["metric"] and d["unit"] == "pairs/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 3 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]


# ------------------------------------------------------------------------------ input staging (SURVEY 8f item 3)
@pytest.mark.parametrize("name", ["collate_long", "collate_short"])
def test_collate_matches_reference_golden(name):
    """multiModalDataset_collate_fn mirror == the reference's own function (multimodal_data_module.py:98-109) on a
    batch with lengths around and beyond 25 (golden written by oracle/make_golden.py from the live reference)."""
    from oracle.make_golden import collate_batch
    with open(os.path.join(GOLD, name + ".json")) as fh:
        g = json.load(fh)
    batch = collate_batch()
    if not g["long"]:
        batch = [b for b in batch if b[2] <= 12]
    img, ids, lens, raw = cv.multiModalDataset_collate_fn(batch)
    assert list(img.shape) == g["img_shape"] and [float(v) for v in img[:, 0, 0, 0]] == g["img_first"]
    assert str(ids.dtype) == g["ids_dtype"] and str(lens.dtype) == g["lens_dtype"]
    assert ids.tolist() == g["ids"] and lens.tolist() == g["lens"] and raw == g["raw"]


def test_pinned_stager_holds_what_the_reference_collate_hands_to_the_model():
    """fixed-shape [B,25] staging: same ids (zero-padded to 25) and the same clamped lengths as the reference's
    collate, from per-sample rows and from an already padded tensor; PAD beyond every length; stale contents of a
    previous batch never leak."""
    from oracle.make_golden import collate_batch
    with open(os.path.join(GOLD, "collate_long.json")) as fh:
        g = json.load(fh)
    batch = collate_batch()
    B = len(batch)
    st = cv.PinnedBatchStager(B, feat_shape=(8,), feat_dtype=torch.bfloat16, pin=False)
    st.ids_host.fill_(7)                                       # garbage from an earlier batch
    feats = torch.arange(B * 8, dtype=torch.float32).reshape(B, 8)
    ids, lens = st.stage([b[1] for b in batch], [b[2] for b in batch], feats)
    want = torch.zeros(B, 25, dtype=torch.int64)
    gi = torch.tensor(g["ids"])
    want[:, :gi.shape[1]] = gi
    assert ids.shape == (B, 25) and ids.dtype == torch.int64 and torch.equal(ids, want)
    assert lens.tolist() == g["lens"] and lens.dtype == torch.int64
    assert st.x_host.dtype == torch.bfloat16 and torch.equal(st.x_host.float(), feats.to(torch.bfloat16).float())
    pos = torch.arange(25)[None, :]
    assert bool((ids[pos >= lens[:, None]] == 0).all())
    # the same from the reference-style padded tensor (short batch: width 12 < 25)
    with open(os.path.join(GOLD, "collate_short.json")) as fh:
        gs = json.load(fh)
    st2 = cv.PinnedBatchStager(len(gs["lens"]), pin=False)
    st2.ids_host.fill_(9)
    ids2, lens2 = st2.stage(torch.tensor(gs["ids"]), gs["lens"])
    assert ids2[:, :12].tolist() == gs["ids"] and bool((ids2[:, 12:] == 0).all()) and lens2.tolist() == gs["lens"]
    with pytest.raises(ValueError):
        st2.stage(torch.tensor(gs["ids"])[:2], gs["lens"])


def test_batch_trials_shares_label_rows_and_keeps_trial_order():
    """Labeled-S items (imgs [4,3,H,W] target first, label row, len, [raw]) -> stacked frames + distinct label rows
    + per-trial index: decoding the index gives back every trial's own label row; frames keep trial-major order."""
    g = torch.Generator().manual_seed(0)
    vocab = {"ball": 71, "car": 90, "kitty": 76}
    names = ["ball", "car", "ball", "kitty", "car", "ball"]
    items = []
    for i, nm in enumerate(names):
        imgs = torch.full((4, 3, 2, 2), float(i)) + torch.arange(4, dtype=torch.float32)[:, None, None, None] / 10
        label = torch.tensor([2, vocab[nm], 3]) if i % 2 == 0 else torch.tensor([vocab[nm]])   # with / without sos-eos
        items.append((imgs, label, label.numel(), [nm]))
    frames, ids, lens, index, raw = cv.batch_trials(items)
    assert frames.shape == (24, 3, 2, 2) and ids.dtype == torch.int64 and index.dtype == torch.int32
    assert raw == names and index.shape == (6,)
    assert ids.shape[0] == len({tuple(it[1].tolist()) for it in items}) < len(items)      # rows are shared
    for i, it in enumerate(items):
        row = ids[index[i]]
        n = int(lens[index[i]])
        assert row[:n].tolist() == it[1].tolist() and bool((row[n:] == 0).all())
        assert torch.equal(frames[4 * i:4 * i + 4], it[0])                                  # target stays first
    with pytest.raises(ValueError):
        cv.batch_trials(items + [(torch.zeros(3, 3, 2, 2), torch.tensor([5]), 1, ["x"])])
    with pytest.raises(ValueError):
        cv.batch_trials(items, max_len=2)


def test_lit_epoch_end_hooks_log_example_weighted_means():
    """joint_loss_epoch_end / *_epoch_end (multimodal_lit.py:376-444, 450-541): example-weighted means of the step
    outputs under the reference's metric names; validation_step routes dataloaders >= 2 to the test split."""
    lit = _lit(fix_temperature=True)
    logged = {}
    lit.log = lambda name, value, *a, **k: logged.__setitem__(name, (float(value), k))
    outs = [dict(batch_size=2, loss=torch.tensor(1.0), infonce_loss=torch.tensor(1.0), image_accuracy=torch.tensor(0.5),
                 text_accuracy=torch.tensor(0.0), image_entropy=torch.tensor(2.0), text_entropy=torch.tensor(4.0)),
            dict(batch_size=6, loss=torch.tensor(3.0), infonce_loss=torch.tensor(3.0), image_accuracy=torch.tensor(1.0),
                 text_accuracy=torch.tensor(1.0), image_entropy=torch.tensor(0.0), text_entropy=torch.tensor(0.0))]
    lit.training_epoch_end(outs)
    assert logged["train_loss_epoch"][0] == pytest.approx(2.5) and logged["train_image_accuracy_epoch"][0] == pytest.approx(0.875)
    assert logged["train_loss_epoch"][1] == dict(on_step=False, on_epoch=True)
    logged.clear()
    lit.validation_epoch_end([outs, [], outs[:1], []])
    assert logged["val_loss"][0] == pytest.approx(2.5) and logged["val_text_entropy"][0] == pytest.approx(1.0)
    assert logged["test_loss"][0] == pytest.approx(1.0)
    for name in ("infonce_loss", "image_accuracy", "text_accuracy", "image_entropy", "text_entropy", "loss"):
        assert "val_" + name in logged and "test_" + name in logged
    calls = []
    lit.validation_test_step = lambda stage, batch, idx, dataloader_idx=0: calls.append((stage, dataloader_idx))
    lit.validation_step(None, 0, 1); lit.validation_step(None, 0, 3)
    assert calls == [("val", 1), ("test", 1)]
