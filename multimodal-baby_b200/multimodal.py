"""Drop-in `MultiModalModel` for CVCL whose contrastive head runs on hand-written sm_100a kernels.

Mirrors the public surface of the reference's multimodal/multimodal.py (class and attribute
names, argument meaning, return tuples, error behaviour) for the hot path only:

    MultiModalModel(vision_encoder, text_encoder, args)                       multimodal.py:691-715
      .encode_image(image)            -> (image_features, image_feature_map)  multimodal.py:732-737
      .encode_text(text, text_length) -> (text_features, text_outputs)        multimodal.py:739-744
      .forward(image, text, text_length, return_image_features=False,
               return_text_outputs=False)                                     multimodal.py:746-794
      .calculate_contrastive_loss(x, y, y_len) -> 10-tuple                    multimodal.py:796-822

`vision_encoder` / `text_encoder` may be the REFERENCE's own VisionEncoder / TextEncoder objects
(that is the drop-in case: replace the MultiModalModel import in multimodal_lit.py) or the minimal
mirrors defined below, which keep the same parameter attribute paths so that state_dict keys are
identical.  The ResNeXt trunk stays a stock torch module; everything after its pooled / layer4
output and after the token ids goes through `ops` (libcvcl_b200.so).  There is no CPU path: calling
the model with CPU tensors raises.

Out of scope (raise NotImplementedError instead of silently differing): text encoders other than
"embedding" (cbow / lstm / bilstm / transformer, multimodal.py:505-573), dropout_o > 0 in training
mode (multimodal.py:575-580), the ViT trunk (`vit_dino`).
"""
from __future__ import annotations

import contextlib
import math

import numpy as np
import torch
import torch.nn as nn

from . import ops

# defaults of the reference's argparse (multimodal.py:17-29)
TEXT_ENCODER = "embedding"
EMBEDDING_TYPE = "flat"
EMBEDDING_DIM = 128
CRANGE = 1
DROPOUT_I = 0.0
DROPOUT_O = 0.0
NORMALIZE_FEATURES = False
SIM = "max"
TEMPERATURE = 0.07
FIX_TEMPERATURE = False
CNN_MODEL = "resnext50_32x4d"
LAST_CNN_OUT_DIM = 2048          # multimodal.py:116-126

# special tokens (multimodal_data_module.py:37-50)
PAD_TOKEN_ID, UNK_TOKEN_ID, SOS_TOKEN_ID, EOS_TOKEN_ID = 0, 1, 2, 3
MAX_LEN_UTTERANCE = 25


def _args_dict(args):
    if args is None:
        return {}
    return dict(args) if isinstance(args, dict) else vars(args)


class PooledTrunk(nn.Module):
    """Trunk stand-in fed with trunk-boundary features ([B,2048] pooled activations): keeps the
    `layer4` / `fc` attribute paths of a torchvision ResNet so the head parameters live where the
    reference keeps them (`image_embed.model.fc.*`)."""

    def __init__(self, in_dim, embedding_dim):
        super().__init__()
        self.layer4 = nn.Identity()
        self.fc = nn.Linear(in_dim, embedding_dim)

    def forward(self, x):
        return self.fc(self.layer4(x))


class VisionEncoder(nn.Module):
    """Mirror of the reference VisionEncoder (multimodal.py:56-194) for the CNN branch: a frozen
    torchvision ResNeXt-50 32x4d trunk plus a trainable projection head -- `model.fc =
    Linear(2048, E)` for flat embeddings (:186-192), a 1x1 `Conv2d(2048, E)` appended after layer4
    for spatial embeddings (:181-185).  `trunk="pooled"` builds only the head (inputs are then
    trunk-boundary features), which is what the benchmarks and parity tests feed."""

    def __init__(self, args, trunk="resnext"):
        super().__init__()
        self.args = _args_dict(args)
        self.embedding_type = self.args.get("embedding_type", EMBEDDING_TYPE)
        self.embedding_dim = self.args.get("embedding_dim", EMBEDDING_DIM)
        self.cnn_model = self.args.get("cnn_model", CNN_MODEL)
        self.finetune_cnn = self.args.get("finetune_cnn", False)
        self.vit_dino = False
        if self.args.get("vit_dino", False):
            raise NotImplementedError("vit_dino trunk is outside the cvcl_b200 hot path")
        if trunk == "pooled":
            if self.embedding_type == "flat":
                self.model = PooledTrunk(LAST_CNN_OUT_DIM, self.embedding_dim)
            else:
                self.model = nn.Sequential(nn.Identity(),
                                           nn.Conv2d(LAST_CNN_OUT_DIM, self.embedding_dim, 1))
        else:
            import torchvision
            name = self.cnn_model if hasattr(torchvision.models, str(self.cnn_model)) else CNN_MODEL
            model = getattr(torchvision.models, name)(weights=None)
            if not self.finetune_cnn:                       # multimodal.py:175-177
                for p in model.parameters():
                    p.requires_grad = False
            if self.embedding_type == "spatial":
                model = nn.Sequential(*list(model.children())[:-2],
                                      nn.Conv2d(LAST_CNN_OUT_DIM, self.embedding_dim, 1))
            else:
                model.fc = nn.Linear(LAST_CNN_OUT_DIM, self.embedding_dim)
            self.model = model

    @property
    def last_cnn_out_dim(self):
        return LAST_CNN_OUT_DIM

    def forward(self, x):
        """Reference semantics (multimodal.py:88-104): (features incl. head, layer4 map).  Kept
        for callers that use the encoder on its own; MultiModalModel does not route through it."""
        feats, fmap = split_trunk_forward(self, x)
        return feats, fmap


class TextEncoder(nn.Module):
    """Mirror of the reference TextEncoder (multimodal.py:278-364) restricted to the embedding
    branch: `nn.Embedding(V, E, padding_idx=0)` and the attributes other reference classes read."""

    def __init__(self, vocab, image_feature_map_dim, args):
        super().__init__()
        self.args = _args_dict(args)
        self.text_encoder = self.args.get("text_encoder", TEXT_ENCODER)
        if self.text_encoder != "embedding":
            raise NotImplementedError(
                "cvcl_b200 implements the 'embedding' text encoder only (got %r)" % self.text_encoder)
        self.embedding_type = self.args.get("embedding_type", EMBEDDING_TYPE)
        self.embedding_dim = self.args.get("embedding_dim", EMBEDDING_DIM)
        self.hidden_dim = self.embedding_dim
        self.input_dim = self.embedding_dim
        self.crange = self.args.get("crange", CRANGE)
        self.dropout_i = self.args.get("dropout_i", DROPOUT_I)
        self.dropout_o = self.args.get("dropout_o", DROPOUT_O)
        self.vocab = vocab
        self.word2idx = vocab
        self.idx2word = {idx: word for word, idx in vocab.items()}
        self.embedding = nn.Embedding(self.vocab_size, self.embedding_dim, padding_idx=PAD_TOKEN_ID)

    @property
    def vocab_size(self):
        return len(self.vocab)

    @property
    def regressional(self):
        return False

    @property
    def captioning(self):
        return False

    @property
    def has_attention(self):
        return False

    def forward(self, x, x_len, image_features=None, image_feature_map=None):
        """(ret, output, attns) as multimodal.py:493-584, embedding branch."""
        _check_dropout(self)
        table = self.embedding.weight
        output = ops.text_outputs(x, table)
        if self.embedding_type == "flat":
            ret = ops.text_features_flat(x, x_len, table, normalize=False)
        else:
            ret = output
        return ret, output, None


def _check_dropout(text_embed):
    p = getattr(text_embed, "dropout_o", 0.0) or 0.0
    if p > 0 and text_embed.training:
        raise NotImplementedError(
            "dropout_o=%g in training mode is not implemented by the cvcl_b200 kernels "
            "(all shipped CVCL configs use dropout_o=0)" % p)


@contextlib.contextmanager
def _swapped(module, name, new):
    old = getattr(module, name)
    setattr(module, name, new)
    try:
        yield old
    finally:
        setattr(module, name, old)


def split_trunk_forward(image_embed, x, run_head=True):
    """Run the vision encoder's trunk and (optionally) its stock torch head.
    Returns (features_or_pooled, feature_map).  With run_head=False the first element is the
    trunk-boundary activation that feeds the kernels: pooled [B,2048] (flat) or the layer4 map
    [B,2048,H,W] (spatial)."""
    model = image_embed.model
    if getattr(image_embed, "vit_dino", False):
        raise NotImplementedError("vit_dino trunk is outside the cvcl_b200 hot path")
    if isinstance(model, PooledTrunk):             # trunk-boundary features fed directly
        if x.dim() > 2:                            # e.g. a Labeled-S trial viewed as [n_way, 1, 1, 2048]
            x = x.reshape(-1, x.shape[-1])
        return (model.fc(x) if run_head else x), x
    if image_embed.embedding_type == "spatial":
        fmap = x
        for layer in list(model.children())[:-1]:
            fmap = layer(fmap)
        if not run_head:
            return fmap, fmap
        return list(model.children())[-1](fmap), fmap
    captured = {}
    handle = model.layer4.register_forward_hook(lambda m, i, o: captured.__setitem__("fmap", o))
    try:
        if run_head:
            out = model(x)
        else:
            with _swapped(model, "fc", nn.Identity()):
                out = model(x)
    finally:
        handle.remove()
    return out, captured.get("fmap")


class MultiModalModel(nn.Module):
    """B200 drop-in for the reference MultiModalModel (multimodal.py:691-822)."""

    def __init__(self, vision_encoder, text_encoder, args):
        super().__init__()
        self.args = _args_dict(args)
        self.sim = self.args.get("sim", SIM)
        self.embedding_type = self.args.get("embedding_type", EMBEDDING_TYPE)
        self.normalize_features = self.args.get("normalize_features", NORMALIZE_FEATURES)
        self.initial_temperature = self.args.get("temperature", TEMPERATURE)
        self.fix_temperature = self.args.get("fix_temperature", FIX_TEMPERATURE)

        self.image_embed = vision_encoder
        self.text_embed = text_encoder
        if getattr(text_encoder, "text_encoder", "embedding") != "embedding":
            raise NotImplementedError("cvcl_b200 implements the 'embedding' text encoder only")

        # multimodal.py:711-715: a plain CPU 0-dim tensor when fixed (not a buffer, not in the
        # state_dict), an nn.Parameter otherwise.
        self.logit_neg_log_temperature = torch.ones([]) * - np.log(self.initial_temperature)
        if not self.fix_temperature:
            self.logit_neg_log_temperature = nn.Parameter(self.logit_neg_log_temperature)

        # API-fidelity switches.  The reference returns the B x B logits and the [B,L,E]
        # text_outputs from calculate_contrastive_loss although its trainer ignores them
        # (multimodal_lit.py:241-266).  True = materialise them (faithful); False = return None in
        # those tuple slots and keep the step fully fused.
        self.materialize_logits = True
        self.materialize_text_outputs = True
        self.materialize_features = True
        # "fused": one C call computes loss and all head gradients (flat embeddings, frozen trunk);
        # "ops": op-by-op autograd path (always used for spatial embeddings / finetune_cnn).
        self.train_path = "fused"
        self.process_group = None         # set to a torch.distributed group to shard the batch
        # spatial "max" similarity: "split_bf16" evaluates head and scores with two-term bf16 operands (fp32-grade,
        # 3x the tensor work) so that the arg-max over the 7x7 locations agrees with the reference's fp32
        # arithmetic; "bf16" is the fast single-term form (near-tied locations may flip, moving gradient rows)
        self.spatial_max_precision = "split_bf16"

    # -- helpers ---------------------------------------------------------------------------
    def _head(self):
        model = self.image_embed.model
        if self.embedding_type == "spatial":
            conv = list(model.children())[-1]
            return conv.weight.view(conv.weight.shape[0], -1), conv.bias
        return model.fc.weight, model.fc.bias

    def _log_scale(self):
        return self.logit_neg_log_temperature

    def _trunk(self, image):
        with torch.set_grad_enabled(torch.is_grad_enabled()):
            return split_trunk_forward(self.image_embed, image, run_head=False)

    def _split(self):
        return self.embedding_type == "spatial" and self.sim == "max" and self.spatial_max_precision == "split_bf16"

    def _image_features_from_trunk(self, boundary):
        w, b = self._head()
        if self.embedding_type == "flat":
            return ops.head_features(boundary, w, b, self.normalize_features)
        B, K, H, W = boundary.shape
        rows = boundary.permute(0, 2, 3, 1).reshape(B * H * W, K)          # NHWC rows
        feat = ops.head_features(rows, w, b, self.normalize_features, split=self._split())      # [B*H*W, E]
        return feat.view(B, H, W, -1)                                      # NHWC

    # -- reference API ---------------------------------------------------------------------
    def encode_image(self, image):
        boundary, fmap = self._trunk(image)
        feat = self._image_features_from_trunk(boundary)
        if self.embedding_type == "spatial":
            feat = feat.permute(0, 3, 1, 2)                 # [B,E,H,W] view, as the reference returns
        return feat, fmap

    def encode_text(self, text, text_length):
        _check_dropout(self.text_embed)
        table = self.text_embed.embedding.weight
        text_outputs = ops.text_outputs(text, table) if self.materialize_text_outputs else None
        if self.embedding_type == "flat":
            feat = ops.text_features_flat(text, text_length, table, self.normalize_features)
        else:
            feat, _ = ops.text_features_spatial(text, text_length, table, self.normalize_features)
        return feat, text_outputs

    def _match_logits(self, image_features, text, text_length):
        """(logits_per_image, logits_per_text) for already-encoded image features."""
        s = self._log_scale()
        table = self.text_embed.embedding.weight
        if self.embedding_type == "flat":
            txt = ops.text_features_flat(text, text_length, table, self.normalize_features)
            return ops.sim_logits(image_features, txt, s)
        B, E, H, W = image_features.shape
        nhwc = image_features.permute(0, 2, 3, 1).reshape(B, H * W, E)
        if self.sim == "mean":
            _, tpool = ops.text_features_spatial(text, text_length, table, self.normalize_features,
                                                 1.0 / (H * W), want_tok=False)
            return ops.sim_logits(ops.spatial_pool(nhwc), tpool, s)
        tok, _ = ops.text_features_spatial(text, text_length, table, self.normalize_features)
        match = ops.spatial_max_similarity(nhwc, tok, text_length, text, split=self._split())
        scale = s.exp() if torch.is_tensor(s) else math.exp(s)
        scale = scale.to(match.device) if torch.is_tensor(scale) else scale
        return match * scale, match.t() * scale

    def forward(self, image, text, text_length, return_image_features=False,
                return_text_outputs=False):
        image_features, image_feature_map = self.encode_image(image)
        logits_per_image, logits_per_text = self._match_logits(image_features, text, text_length)
        ret = logits_per_image, logits_per_text
        if return_image_features:
            ret = ret + (image_features, image_feature_map)
        if return_text_outputs:
            table = self.text_embed.embedding.weight
            ret = ret + (ops.text_outputs(text, table),)
        return ret

    def calculate_contrastive_loss(self, x, y, y_len):
        """10-tuple of multimodal.py:796-822: (infonce_loss, image_accuracy, text_accuracy,
        image_entropy, text_entropy, logits_per_image, logits_per_text, image_features,
        image_feature_map, text_outputs)."""
        _check_dropout(self.text_embed)
        s = self._log_scale()
        table = self.text_embed.embedding.weight
        boundary, fmap = self._trunk(x)
        fused_ok = (self.embedding_type == "flat" and self.train_path == "fused"
                    and not boundary.requires_grad)
        if fused_ok:
            # one fused pass: loss + all head gradients (already summed over ranks when sharded)
            w, b = self._head()
            loss, iacc, tacc, ient, tent, img_f, txt_f = ops.flat_contrastive_loss(
                boundary, y, y_len, w, b, table, s, self.normalize_features,
                want_features=self.materialize_features, group=self.process_group)
            image_features = img_f if self.materialize_features else None
        else:
            image_features = self._image_features_from_trunk(boundary)
            if self.embedding_type == "flat":
                img_f = image_features
                txt_f = ops.text_features_flat(y, y_len, table, self.normalize_features)
            else:
                B, H, W, E = image_features.shape
                nhwc = image_features.reshape(B, H * W, E)
                image_features = image_features.permute(0, 3, 1, 2)
                if self.sim == "mean":
                    img_f, txt_f = ops.spatial_mean_factors(nhwc, y, y_len, table, self.normalize_features)
                else:
                    img_f = txt_f = None
            if img_f is not None:
                # flat features are unit vectors when normalize_features is on (one similarity pass at large batch);
                # the pooled spatial factors are not
                unit = self.embedding_type == "flat" and bool(self.normalize_features)
                loss, iacc, tacc, ient, tent, _, _ = ops.sim_infonce(img_f, txt_f, s, self.process_group, unit)
            elif self.process_group is None:
                tok, _ = ops.text_features_spatial(y, y_len, table, self.normalize_features)
                match = ops.spatial_max_similarity(nhwc, tok, y_len, y, split=self._split())
                loss, iacc, tacc, ient, tent, lpi, lpt = ops.infonce_from_match(match, s)
            else:
                # global-batch loss; the logits are this rank's [b,b] block, as on the sharded mean path
                tok, _ = ops.text_features_spatial(y, y_len, table, self.normalize_features)
                loss, iacc, tacc, ient, tent, _, _, mloc = ops.spatial_max_infonce(
                    nhwc, tok, y_len, y, s, self.process_group, split=self._split(), local_match=True)
                lpi = mloc * math.exp(ops._scalar(s))
                lpt = lpi.t()
        logits_per_image = logits_per_text = None
        if self.materialize_logits and img_f is not None and img_f.numel() == 0:
            raise RuntimeError("materialize_logits=True needs materialize_features=True on the fused path")
        if self.materialize_logits:
            if self.embedding_type == "spatial" and self.sim == "max":
                logits_per_image, logits_per_text = lpi, lpt
            else:
                with torch.no_grad():
                    logits_per_image, logits_per_text = ops.sim_logits(img_f, txt_f, ops._scalar(s))
        text_outputs = ops.text_outputs(y, table) if self.materialize_text_outputs else None
        return (loss, iacc, tacc, ient, tent, logits_per_image, logits_per_text,
                image_features, fmap, text_outputs)

    @staticmethod
    def add_to_argparse(parser):
        """Same flags as multimodal.py:717-730."""
        parser.add_argument("--embedding_type", type=str, default=EMBEDDING_TYPE,
                            choices=["spatial", "flat"],
                            help="type of embeddings to use (spatial or flat embedding)")
        parser.add_argument("--embedding_dim", type=int, default=EMBEDDING_DIM,
                            help="size of embedding representations")
        parser.add_argument("--normalize_features", action="store_true",
                            help="normalize feature embeddings after encoding")
        parser.add_argument("--sim", type=str, default=SIM, choices=["mean", "max"],
                            help="type of similarity to use (mean or max over image patches per word)")
        parser.add_argument("--temperature", type=float, default=TEMPERATURE,
                            help="initial temperature")
        parser.add_argument("--fix_temperature", action="store_true",
                            help="fix the temperature so it is not trained")
