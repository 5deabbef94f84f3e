"""`MultiModalLitModel` mirror for the contrastive path (reference: multimodal/multimodal_lit.py).

Keeps the caller-facing API of the reference's Lightning wrapper that touches the hot path:

    MultiModalLitModel(vision_encoder, text_encoder, args)      multimodal_lit.py:40-74
      .forward(x, y, y_len)            -> logits_per_image, logits_per_text     :130-131
      .encode_image(x) / .encode_text(y, y_len)                                  :151-159
      .tokenize(texts) -> (ids int64 [N,25], lens int64 [N])                     :161-190
      .calculate_joint_loss(batch, stage, log)   (contrastive branch)            :227-375
      .training_step / .validation_test_step (Labeled-S 4-way trial)             :445-511
      .joint_loss_epoch_end / *_epoch_end  (example-weighted epoch metrics)      :376-444, :450-541
      .configure_optimizers()                                                    :112-128
      .evaluate_trials(...)  batched replacement of the per-trial loop of eval.py:175-266
      .evaluate_retrieval(...)  image->text / text->image top-K, ranks and recall@K over a held-out split

pytorch_lightning is optional (absent in this image): the class derives from
`pl.LightningModule` when importable, else from `nn.Module` with no-op `log` /
`save_hyperparameters`.  The language-model / text-generation branches (lambda_lm, lambda_ar,
multimodal_lit.py:266-358) are outside the hot path and raise NotImplementedError.
"""
from __future__ import annotations

import functools
import json
import math
import os

import torch
import torch.nn as nn

from . import ops
from .multimodal import (MultiModalModel, MAX_LEN_UTTERANCE, PAD_TOKEN_ID, SOS_TOKEN_ID,
                         EOS_TOKEN_ID, _args_dict)

N_VAL_DATALOADERS_PER_SPLIT = 2                    # multimodal_data_module.py:32

try:                                               # pragma: no cover - not installed here
    import pytorch_lightning as pl
    _Base = pl.LightningModule
except Exception:                                  # noqa: BLE001
    class _Base(nn.Module):
        def save_hyperparameters(self, *a, **k):
            pass

        def log(self, *a, **k):
            pass

OPTIMIZER = torch.optim.AdamW
LR = 3e-4
FACTOR = 0.1
PATIENCE = 20
WEIGHT_DECAY = 0.01

_VOCAB_CANDIDATES = (
    os.path.join(os.path.dirname(os.path.abspath(__file__)), "vocab.json"),
    "/root/reference/multimodal/vocab.json",
)


class WhitespaceTokenizer:
    """Stand-in for spaCy's en_core_web_sm (not installable offline): whitespace split.  Token-id
    parity with the reference holds for pre-tokenised text only (SURVEY Appendix A)."""

    def __call__(self, text):
        return text.split()


def load_vocab(path=None):
    for p in ((path,) if path else _VOCAB_CANDIDATES):
        if p and os.path.exists(p):
            with open(p) as f:
                return json.load(f)
    raise FileNotFoundError("vocab.json not found; pass vocab= or vocab_path=")


class LanguageModelHead(nn.Module):
    """Parameter holder mirroring the reference LanguageModel's state_dict entries
    (multimodal.py:825-843: `text_encoder` shared, `output_layer` tied to the embedding, bias [V])
    so checkpoints load with identical keys.  The LM loss itself is outside the hot path."""

    def __init__(self, text_encoder, args):
        super().__init__()
        a = _args_dict(args)
        self.text_encoder = text_encoder
        self.output_layer = nn.Linear(text_encoder.hidden_dim, text_encoder.vocab_size,
                                      bias=a.get("bias", True))
        if a.get("tie", True):
            self.output_layer.weight = self.text_encoder.embedding.weight

    def forward(self, *a, **k):
        raise NotImplementedError("the language-model branch is outside the cvcl_b200 hot path")


class MultiModalLitModel(_Base):
    def __init__(self, vision_encoder, text_encoder, args, vocab=None, tokenizer=None):
        super().__init__()
        self.args = _args_dict(args)
        self.optimizer_class = self.args.get("optimizer", OPTIMIZER)
        self.lr = self.args.get("lr", LR)
        self.lr_scheduler = self.args.get("lr_scheduler", False)
        self.factor = self.args.get("factor", FACTOR)
        self.patience = self.args.get("patience", PATIENCE)
        self.weight_decay = self.args.get("weight_decay", WEIGHT_DECAY)
        self.lambda_mm = self.args.get("lambda_mm", 1.)
        self.lambda_lm = self.args.get("lambda_lm", 0.)
        self.lambda_ar = self.args.get("lambda_ar", 0.)
        self.optimize_unused = self.args.get("optimize_unused", False)
        if self.lambda_lm or self.lambda_ar:
            raise NotImplementedError("language-model / attention-regularisation losses "
                                      "(lambda_lm, lambda_ar) are outside the cvcl_b200 hot path")
        self.vision_encoder = vision_encoder
        self.text_encoder = text_encoder
        self.model = MultiModalModel(self.vision_encoder, self.text_encoder, args)
        self.language_model = LanguageModelHead(self.text_encoder, args)
        self.vocab = vocab if vocab is not None else getattr(text_encoder, "vocab", None) or load_vocab()
        self.nlp = tokenizer if tokenizer is not None else WhitespaceTokenizer()
        self.save_hyperparameters()

    # -- optimiser (multimodal_lit.py:112-128) ------------------------------------------------
    def configure_optimizers(self):
        optimizer = self.optimizer_class(self.parameters(), lr=self.lr, weight_decay=self.weight_decay)
        if not self.lr_scheduler:
            return optimizer
        sched = torch.optim.lr_scheduler.ReduceLROnPlateau(optimizer, factor=self.factor,
                                                           patience=self.patience)
        return {"optimizer": optimizer, "lr_scheduler": {"scheduler": sched, "monitor": "val_loss"}}

    # -- inference API (multimodal_lit.py:130-190) ---------------------------------------------
    def forward(self, x, y, y_len):
        return self.model(x, y, y_len)

    def encode_image(self, x):
        image_features, _ = self.model.encode_image(x)
        return image_features

    def encode_text(self, y, y_len=None):
        text_features, _ = self.model.encode_text(y, y_len)
        return text_features

    def attention_maps(self, image, text, text_length, text_index=None, out_size=None):
        return self.model.spatial_attention_maps(image, text, text_length, text_index, out_size)

    def tokenize(self, texts):
        """multimodal_lit.py:161-190: [<sos>] + ids + [<eos>], truncated to 25, padded with 0."""
        max_seq_len = MAX_LEN_UTTERANCE
        if isinstance(texts, str):
            texts = [texts]
        all_tokens, token_lengths = [], []
        for text in texts:
            word_tokens = [getattr(t, "text", t) for t in self.nlp(text)]
            if len(word_tokens) > max_seq_len - 2:
                word_tokens = word_tokens[:max_seq_len - 2]
            token_lengths.append(len(word_tokens) + 2)
            all_tokens.append(
                [self.vocab["<sos>"]] + [self.vocab.get(t, self.vocab["<unk>"]) for t in word_tokens]
                + [self.vocab["<eos>"]] + [self.vocab["<pad>"]] * (max_seq_len - len(word_tokens) - 2))
        return (torch.tensor(all_tokens, dtype=torch.long),
                torch.tensor(token_lengths, dtype=torch.long))

    # -- training (multimodal_lit.py:227-375, contrastive branch) ------------------------------
    def calculate_joint_loss(self, batch, stage, log, eval_textgen=False, ce_weight=None):
        x, y, y_len, raw_y = batch
        ret = {'batch_size': x.size(0)}
        infonce_loss, image_accuracy, text_accuracy, image_entropy, text_entropy, *_ = \
            self.model.calculate_contrastive_loss(x, y, y_len)
        log(f"{stage}_infonce_loss", infonce_loss)
        log(f"{stage}_image_accuracy", image_accuracy)
        log(f"{stage}_text_accuracy", text_accuracy)
        log(f"{stage}_image_entropy", image_entropy)
        log(f"{stage}_text_entropy", text_entropy)
        # multimodal_lit.py:252 (one D2H read when the temperature is a CUDA parameter, as in the reference)
        log("temperature", math.exp(-ops._scalar(self.model.logit_neg_log_temperature)))
        ret.update({
            'infonce_loss': infonce_loss.detach(),
            'image_accuracy': image_accuracy,
            'text_accuracy': text_accuracy,
            'image_entropy': image_entropy.detach(),
            'text_entropy': text_entropy.detach(),
        })
        loss = self.lambda_mm * infonce_loss
        log(f"{stage}_loss", loss)
        ret.update({'loss': loss})
        return ret

    def joint_loss_epoch_end(self, outputs, stage, log, eval_textgen=False):
        """multimodal_lit.py:376-444, contrastive branch: example-weighted means of the step outputs."""
        n = sum(o['batch_size'] for o in outputs)

        def mean(name):
            return sum(float(o[name]) * o['batch_size'] for o in outputs) / n
        for name in ('infonce_loss', 'image_accuracy', 'text_accuracy', 'image_entropy', 'text_entropy'):
            log(f"{stage}_{name}", mean(name))
        log(f"{stage}_loss", mean('loss'))

    def training_step(self, batch, batch_idx):
        return self.calculate_joint_loss(batch, 'train', self.log)

    def training_epoch_end(self, outputs):
        ops.check_token_ids()            # a token id outside the vocabulary reached the kernels this epoch -> IndexError
        def log(name, value, *a, **k):
            return self.log(f"{name}_epoch", value, *a, on_step=False, on_epoch=True, **k)
        return self.joint_loss_epoch_end(outputs, 'train', log)

    # -- Labeled-S trial (multimodal_lit.py:466-511) --------------------------------------------
    def validation_test_step(self, stage, batch, batch_idx, dataloader_idx=0):
        log = functools.partial(self.log, on_step=False, on_epoch=True)
        ret = {}
        if dataloader_idx == 0:
            ret.update(self.calculate_joint_loss(batch, stage, lambda *a, **k: None))
        elif dataloader_idx == 1:
            x, y, y_len, raw_y = batch
            x = x.view(-1, *x.shape[-3:])
            logits_per_image, logits_per_text = self.model(x, y, y_len)
            logits = logits_per_text[0]
            pred = torch.argmax(logits).item()
            accuracy = int(pred == 0)                  # the target is always the first candidate
            log_p = torch.log_softmax(logits, dim=-1)  # utils.get_entropy (utils.py:106-108)
            entropy = (torch.softmax(log_p, dim=-1) * -log_p).sum(dim=-1)
            log(f"{stage}_accuracy", accuracy)
            log(f"{stage}_entropy", entropy)
            log(f"{stage}_accuracy_{raw_y[0][0]}", accuracy)      # per-category metric
            ret.update({'accuracy': accuracy})
        return ret

    def validation_test_epoch_end(self, stage, outputs):
        ops.check_token_ids()
        log = functools.partial(self.log, on_step=False, on_epoch=True)
        return self.joint_loss_epoch_end(outputs[0], stage, log)

    def validation_step(self, batch, batch_idx, dataloader_idx=0):
        if dataloader_idx < N_VAL_DATALOADERS_PER_SPLIT:
            return self.validation_test_step('val', batch, batch_idx, dataloader_idx)
        return self.test_step(batch, batch_idx, dataloader_idx - N_VAL_DATALOADERS_PER_SPLIT)

    def validation_epoch_end(self, outputs):
        self.validation_test_epoch_end('val', outputs[:N_VAL_DATALOADERS_PER_SPLIT])
        if len(outputs) > N_VAL_DATALOADERS_PER_SPLIT:
            self.test_epoch_end(outputs[N_VAL_DATALOADERS_PER_SPLIT:])

    def test_step(self, batch, batch_idx, dataloader_idx=0):
        return self.validation_test_step('test', batch, batch_idx, dataloader_idx)

    def test_epoch_end(self, outputs):
        return self.validation_test_epoch_end('test', outputs)

    # -- batched n-way evaluation (replaces the per-trial loop, eval.py:175-266) -----------------
    @torch.no_grad()
    def evaluate_trials(self, trial_features, label_ids, label_lens, label_index=None, n_way=4,
                        from_trunk_boundary=True, want_logits=True):
        """trial_features (target first): flat models take [N, n_way, 2048] trunk-boundary activations or,
        with from_trunk_boundary=False, [N, n_way, E] head outputs before normalisation; spatial models
        (embedding_type="spatial", sim "max" or "mean") take [N, n_way, 2048, H, W] layer4 maps or
        [N, n_way, E, H, W] head outputs before normalisation.
        label_ids / label_lens: [C, L] / [C] token rows; label_index [N] picks the row per trial
        (None: C == N).  Returns (pred int32 [N], logits fp32 [N, n_way] | empty), the logits being
        `logits_per_text[0]` of the reference's per-trial forward; fp32 end to end, first maximum wins."""
        m = self.model
        if m.embedding_type == "spatial":
            img = self._spatial_head_outputs(trial_features, (n_way,), from_trunk_boundary, "evaluate_trials")
            txt = self._spatial_text(label_ids, label_lens, img.shape[1])
            return ops.eval_nway_spatial(img, txt, label_lens, label_index, n_way, m.sim, bool(m.normalize_features),
                                         ops._scalar(m.logit_neg_log_temperature), want_logits)
        table = m.text_embed.embedding.weight
        s = ops._scalar(m.logit_neg_log_temperature)
        txt = ops.text_features_flat(label_ids, label_lens, table, normalize=False)
        N = trial_features.shape[0]
        feats = trial_features.reshape(N * n_way, -1).float()
        if from_trunk_boundary:
            w, b = m._head()
            feats = ops.linear_f32(feats, w, b)                           # fp32 head (exact mode), own kernel
        return ops.eval_nway(feats, txt, label_index, n_way, bool(m.normalize_features), s, want_logits)

    @torch.no_grad()
    def classify_frames(self, frame_features, label_ids, label_lens, from_trunk_boundary=True, want_logits=True):
        """n-category classification (the reference's other Labeled-S form, multimodal_saycam_data_module.py:545-606:
        every frame against ALL C category labels, argmax over the categories).  frame_features [N, 2048] trunk-
        boundary rows (or [N, E] head outputs with from_trunk_boundary=False); spatial models take [N, 2048, H, W]
        layer4 maps (or [N, E, H, W] head outputs).  label_ids / label_lens [C, L] / [C].
        -> (pred int32 [N] = category row, logits_per_image fp32 [N, C] | empty); fp32 end to end."""
        m = self.model
        s = ops._scalar(m.logit_neg_log_temperature)
        if m.embedding_type == "spatial":
            img = self._spatial_head_outputs(frame_features, (), from_trunk_boundary, "classify_frames")
            txt = self._spatial_text(label_ids, label_lens, img.shape[1])
            return ops.classify_ncat_spatial(img, txt, label_lens, m.sim, bool(m.normalize_features), s, want_logits)
        txt = ops.text_features_flat(label_ids, label_lens, m.text_embed.embedding.weight, normalize=False)
        feats = frame_features.reshape(-1, frame_features.shape[-1]).float()
        if from_trunk_boundary:
            w, b = m._head()
            feats = ops.linear_f32(feats, w, b)
        return ops.classify_ncat(feats, txt, bool(m.normalize_features), s, want_logits)

    @torch.no_grad()
    def evaluate_retrieval(self, frame_features, text_ids, text_lens, frame_group=None, text_group=None, k=10,
                           recall_at=(1, 5, 10), from_trunk_boundary=True, block_bytes=1 << 30):
        """Image->text and text->image retrieval over a held-out split: for every frame, where its utterances rank
        among all N_txt utterances, and for every utterance, where its frames rank among all N_img frames.
        frame_features as classify_frames takes them ([N_img, 2048] trunk-boundary rows or [N_img, E] head outputs;
        spatial models [N_img, 2048, H, W] layer4 maps or [N_img, E, H, W] head outputs); text_ids / text_lens
        [N_txt, L] / [N_txt].  The scores are the fp32 values classify_frames takes its arg-max of.  Without groups
        frame i and text i are the pair (N_img == N_txt); with frame_group [N_img] / text_group [N_txt] (int64) every
        text of a frame's group is a positive of it and the other way round: give repeated utterances one id, or use
        the category of each frame with the category labels as the texts.  Exact: keys ordered as
        torch.sort(descending=True, stable=True) orders them, 1 <= k <= min(64, N_img, N_txt).  The score blocks
        stay under block_bytes.  -> {"image_to_text": d, "text_to_image": d} with d holding "topk", "logits", "rank",
        "recall" {K: R@K}, "median_rank", "mean_rank", "n_queries" (see ops.retrieval_f32)."""
        m = self.model
        w, b = m._head()
        if text_ids.dim() != 2 or tuple(text_lens.shape) != (text_ids.shape[0],):
            raise ValueError("evaluate_retrieval: text_ids %s / text_lens %s are not [N_txt, L] / [N_txt]"
                             % (tuple(text_ids.shape), tuple(text_lens.shape)))
        spatial = m.embedding_type == "spatial"
        chans = w.shape[1] if from_trunk_boundary else w.shape[0]
        if frame_features.dim() != (4 if spatial else 2) or frame_features.shape[1] != chans:
            raise ValueError("evaluate_retrieval: a %s model takes %s of shape [N, %d%s], got %s"
                             % ("spatial" if spatial else "flat", "head outputs" if not from_trunk_boundary else
                                "layer4 maps" if spatial else "trunk-boundary rows", chans, ", H, W" if spatial else "",
                                tuple(frame_features.shape)))
        recall_at = tuple(recall_at)
        ops.check_retrieval_args(frame_features.shape[0], text_ids.shape[0], frame_group, text_group, k, recall_at,
                                 block_bytes, "evaluate_retrieval")
        s = ops._scalar(m.logit_neg_log_temperature)
        if spatial:
            img = self._spatial_head_outputs(frame_features, (), from_trunk_boundary, "evaluate_retrieval")
            txt = self._spatial_text(text_ids, text_lens, img.shape[1])
            return ops.retrieval_f32(img, txt, text_lens, m.sim, bool(m.normalize_features), s, frame_group,
                                     text_group, k, recall_at, block_bytes)
        txt = ops.text_features_flat(text_ids, text_lens, m.text_embed.embedding.weight, normalize=False)
        feats = frame_features.float()
        if from_trunk_boundary:
            feats = ops.linear_f32(feats, w, b)
        return ops.retrieval_f32(feats, txt, None, "flat", bool(m.normalize_features), s, frame_group, text_group, k,
                                 recall_at, block_bytes)

    def _spatial_head_outputs(self, x, lead, from_trunk_boundary, who):
        """[N, *lead, channels, H, W] -> head outputs before normalisation as NHWC rows [N*prod(lead), H*W, E]:
        the fp32 1x1-conv head on layer4 maps (channels = 2048), or the given head outputs (channels = E)."""
        w, b = self.model._head()
        chans = w.shape[1] if from_trunk_boundary else w.shape[0]
        want = "[N, %s%d, H, W]" % ("".join("%d, " % d for d in lead), chans)
        what = "layer4 maps" if from_trunk_boundary else "head outputs"
        if (x.dim() != len(lead) + 4 or tuple(x.shape[1:1 + len(lead)]) != tuple(lead)
                or x.shape[1 + len(lead)] != chans):
            raise ValueError("%s: a spatial model takes %s of shape %s, got %s"
                             % (who, what, want, tuple(x.shape)))
        H, W = x.shape[-2:]
        x = x.reshape(-1, chans, H, W)
        if from_trunk_boundary:
            rows = ops.conv1x1_f32(x, w, b)                               # fp32 head, NCHW read in place
        else:
            rows = x.float().permute(0, 2, 3, 1).reshape(-1, chans)        # NHWC rows
        return rows.view(x.shape[0], H * W, -1)

    def _spatial_text(self, label_ids, label_lens, hw):
        """text side of the spatial scores from the model's own table: per-token features ("max") or the pooled
        factor sum_l tok / (HW len) ("mean"), normalised per token iff normalize_features."""
        m = self.model
        table = m.text_embed.embedding.weight
        if m.sim == "max":
            tok, _ = ops.text_features_spatial(label_ids, label_lens, table, m.normalize_features)
            return tok
        _, pooled = ops.text_features_spatial(label_ids, label_lens, table, m.normalize_features, 1.0 / hw,
                                              want_tok=False)
        return pooled

