"""CPU oracle for the VQAModel eval-mode forward path.

TEST INFRASTRUCTURE ONLY.  Nothing in the product package may import this
module: only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs use it, and there only as the
checker / CPU baseline, never as the thing shipped.

It is a plain functional restatement (torch fp32 tensor ops on CPU, no
``nn.Module``, no import of the reference) of the algorithm in
``/root/reference/models/*.py`` driven directly by the reference's 225-key
``state_dict``.  Every function cites the reference lines it follows.

Parity status: PINNED.  ``tests/golden/make_golden.py`` imports the real
reference in the build container, runs it on seeded inputs and commits the
outputs under ``tests/golden/``; ``tests/test_oracle.py`` checks this oracle
against those vectors (and, when ``/root/reference`` is present, against the
live reference).  The reference itself ships no numerical golden vectors
(SURVEY.md section 8c), only the integer known answers for the tokenizer /
answer vocabulary, which ``tests/test_text_utils.py`` covers.
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Tuple

import torch
import torch.nn.functional as F

BN_EPS = 1e-5  # torch default used by every BatchNorm2d (models/cnn_backbone.py:152,159,246,351)
LN_EPS = 1e-5  # torch default for nn.LayerNorm

IMAGENET_MEAN = (0.485, 0.456, 0.406)  # data/preprocess.py:34
IMAGENET_STD = (0.229, 0.224, 0.225)   # data/preprocess.py:35


# --------------------------------------------------------------------------- helpers
def _bn(sd, p, x):
    """Eval-mode BatchNorm2d with running statistics."""
    w, b = sd[p + ".weight"], sd[p + ".bias"]
    m, v = sd[p + ".running_mean"], sd[p + ".running_var"]
    s = w / torch.sqrt(v + BN_EPS)
    return x * s.view(1, -1, 1, 1) + (b - m * s).view(1, -1, 1, 1)


def _ln(sd, p, x):
    return F.layer_norm(x, (x.shape[-1],), sd[p + ".weight"], sd[p + ".bias"], LN_EPS)


def _lin(sd, p, x):
    return F.linear(x, sd[p + ".weight"], sd.get(p + ".bias"))


# --------------------------------------------------------------------------- image side
def preprocess_u8(images_u8_hwc: torch.Tensor) -> torch.Tensor:
    """uint8 [B,H,W,3] (already 224x224) -> normalised fp32 NCHW.

    ToTensor (/255, HWC->CHW) then Normalize (data/preprocess.py:117-121).  For a
    224x224 input the PIL resize in that pipeline is the identity (SURVEY T8).
    """
    x = images_u8_hwc.to(torch.float32).div(255.0).permute(0, 3, 1, 2)
    mean = torch.tensor(IMAGENET_MEAN, dtype=torch.float32).view(1, 3, 1, 1)
    std = torch.tensor(IMAGENET_STD, dtype=torch.float32).view(1, 3, 1, 1)
    return ((x - mean) / std).contiguous()


def stem(sd, x, p="image_encoder.stem"):
    """conv7x7/2 -> BN -> ReLU -> maxpool3x3/2 (models/cnn_backbone.py:349-354)."""
    x = F.conv2d(x, sd[p + ".0.weight"], None, stride=2, padding=3)
    x = F.relu(_bn(sd, p + ".1", x))
    return F.max_pool2d(x, kernel_size=3, stride=2, padding=1)


def block_conv1(sd, p, x, stride):
    """First half of ResidualBlock.forward (models/cnn_backbone.py:164-197): conv1 -> bn1 -> ReLU."""
    out = F.conv2d(x, sd[p + ".conv1.weight"], None, stride=stride, padding=1)
    return F.relu(_bn(sd, p + ".bn1", out))


def block_tail(sd, p, x, mid, stride):
    """Second half of ResidualBlock.forward (models/cnn_backbone.py:164-197): conv2 -> bn2 on ``mid`` (the output of
    block_conv1), plus the identity or downsampled shortcut of the block input ``x``, then ReLU."""
    out = F.conv2d(mid, sd[p + ".conv2.weight"], None, stride=1, padding=1)
    out = _bn(sd, p + ".bn2", out)
    if (p + ".downsample.0.weight") in sd:  # built at models/cnn_backbone.py:243-249
        idn = F.conv2d(x, sd[p + ".downsample.0.weight"], None, stride=stride)
        idn = _bn(sd, p + ".downsample.1", idn)
    else:
        idn = x
    return F.relu(out + idn)


def residual_block(sd, p, x, stride):
    """ResidualBlock.forward (models/cnn_backbone.py:164-197)."""
    return block_tail(sd, p, x, block_conv1(sd, p, x, stride), stride)


def se_scale(sd, p, x):
    """The per-channel scale [B, C] of SEAttention.forward (models/attention_modules.py:91-136); no biases (:84-85)."""
    sq = x.mean(dim=(2, 3))
    ex = F.relu(F.linear(sq, sd[p + ".fc1.weight"]))
    return torch.sigmoid(F.linear(ex, sd[p + ".fc2.weight"]))


def se_attention(sd, p, x):
    """SEAttention.forward (models/attention_modules.py:91-136)."""
    return x * se_scale(sd, p, x).view(x.shape[0], -1, 1, 1)


def spatial_map(sd, p, x):
    """The sigmoid attention map [B, 1, H, W] of SpatialAttention.forward (models/attention_modules.py:198-243);
    [max, avg] order (:230)."""
    mx = x.max(dim=1, keepdim=True)[0]
    av = x.mean(dim=1, keepdim=True)
    w = sd[p + ".conv.weight"]
    return torch.sigmoid(F.conv2d(torch.cat([mx, av], dim=1), w, None, padding=w.shape[-1] // 2))


def spatial_attention(sd, p, x):
    """SpatialAttention.forward (models/attention_modules.py:198-243)."""
    return x * spatial_map(sd, p, x)


def residual_stage(sd, p, x, stride, taps=None):
    """ResidualStage.forward: blocks, then SE, then spatial (models/cnn_backbone.py:267-279,
    models/attention_modules.py:427-433)."""
    b = 0
    while (p + f".blocks.{b}.conv1.weight") in sd:
        x = residual_block(sd, p + f".blocks.{b}", x, stride if b == 0 else 1)
        b += 1
    if taps is not None:
        taps[p + ".blocks"] = x
    if (p + ".attention.se.fc1.weight") in sd:
        x = se_attention(sd, p + ".attention.se", x)
    if (p + ".attention.spatial.conv.weight") in sd:
        x = spatial_attention(sd, p + ".attention.spatial", x)
    return x


def image_encoder(sd, images, taps=None):
    """CustomResNet.forward (models/cnn_backbone.py:440-463): NCHW fp32 -> [B,512,7,7]."""
    x = stem(sd, images)
    if taps is not None:
        taps["image_encoder.stem"] = x
    for s, stride in ((1, 1), (2, 2), (3, 2), (4, 2)):
        x = residual_stage(sd, f"image_encoder.stage{s}", x, stride, taps)
        if taps is not None:
            taps[f"image_encoder.stage{s}"] = x
    return x


# --------------------------------------------------------------------------- text side
def sinusoidal_pe(max_length: int, embed_dim: int) -> torch.Tensor:
    """PositionalEncoding buffer (models/text_encoder.py:76-96)."""
    pe = torch.zeros(max_length, embed_dim)
    pos = torch.arange(0, max_length, dtype=torch.float).unsqueeze(1)
    div = torch.exp(torch.arange(0, embed_dim, 2).float() * (-math.log(10000.0) / embed_dim))
    pe[:, 0::2] = torch.sin(pos * div)
    pe[:, 1::2] = torch.cos(pos * div)
    return pe.unsqueeze(0)


def _mha(q, k, v, num_heads, key_mask=None):
    """Scaled dot-product attention over heads; returns (context [B,Lq,D], weights [B,H,Lq,Lk]).

    Self-attention: models/text_encoder.py:229-259 (mask fill -inf at :244).
    Cross-attention: models/cross_attention.py:164-197.
    """
    B, Lq, D = q.shape
    Lk = k.shape[1]
    hd = D // num_heads
    q = q.view(B, Lq, num_heads, hd).transpose(1, 2)
    k = k.view(B, Lk, num_heads, hd).transpose(1, 2)
    v = v.view(B, Lk, num_heads, hd).transpose(1, 2)
    s = torch.matmul(q, k.transpose(-2, -1)) / math.sqrt(hd)
    if key_mask is not None:
        s = s.masked_fill(key_mask.unsqueeze(1).unsqueeze(2) == 0, float("-inf"))
    w = F.softmax(s, dim=-1)
    ctx = torch.matmul(w, v).transpose(1, 2).contiguous().view(B, Lq, D)
    return ctx, w


def text_embed(sd, token_ids, p="text_encoder"):
    """Token embedding * sqrt(D) + sinusoidal position (models/text_encoder.py:504-507, :108-112)."""
    emb = sd[p + ".token_embedding.weight"]
    D = emb.shape[1]
    x = F.embedding(token_ids, emb) * math.sqrt(D)                      # :504-507
    return x + sd[p + ".positional_encoding.pe"][:, : x.shape[1], :]     # :108-112


def text_layer(sd, lp, x, attention_mask, num_heads):
    """One pre-norm encoder layer of TransformerTextEncoder (models/text_encoder.py:390-397)."""
    n = _ln(sd, lp + ".norm1", x)                                        # pre-norm, :390
    q = _lin(sd, lp + ".self_attention.W_q", n)
    k = _lin(sd, lp + ".self_attention.W_k", n)
    v = _lin(sd, lp + ".self_attention.W_v", n)
    ctx, _ = _mha(q, k, v, num_heads, attention_mask)
    x = x + _lin(sd, lp + ".self_attention.W_o", ctx)                    # :392
    n = _ln(sd, lp + ".norm2", x)                                        # :395
    return x + _lin(sd, lp + ".ffn.fc2", F.relu(_lin(sd, lp + ".ffn.fc1", n)))  # :320-323,:397


def text_encoder(sd, token_ids, attention_mask, num_heads, p="text_encoder"):
    """TransformerTextEncoder.forward (models/text_encoder.py:479-529)."""
    x = text_embed(sd, token_ids, p)
    layer = 0
    while (p + f".layers.{layer}.norm1.weight") in sd:
        x = text_layer(sd, p + f".layers.{layer}", x, attention_mask, num_heads)
        layer += 1
    enc = _ln(sd, p + ".final_norm", x)                                  # :519
    if attention_mask is not None:                                       # :523-527
        m = attention_mask.unsqueeze(-1).float()
        pooled = (enc * m).sum(dim=1) / m.sum(dim=1).clamp(min=1)
    else:
        pooled = enc.mean(dim=1)
    return enc, pooled


# --------------------------------------------------------------------------- fusion + head
def image_projector(sd, feats, p="fusion.image_projector"):
    """ImageFeatureProjector.forward (models/fusion.py:82-112)."""
    B, C, H, W = feats.shape
    x = feats.view(B, C, H * W).permute(0, 2, 1)
    x = _ln(sd, p + ".projection.1", _lin(sd, p + ".projection.0", x))
    return x + sd[p + ".position_embedding"][:, : H * W, :]


def cross_layer(sd, lp, q, kv, num_heads):
    """MultiHeadCrossAttention.forward (models/cross_attention.py:265-299)."""
    nq = _ln(sd, lp + ".norm_query", q)
    nkv = _ln(sd, lp + ".norm_kv", kv)
    Q = _lin(sd, lp + ".cross_attention.W_q", nq)
    K = _lin(sd, lp + ".cross_attention.W_k", nkv)
    V = _lin(sd, lp + ".cross_attention.W_v", nkv)
    ctx, w = _mha(Q, K, V, num_heads, None)          # key_value_mask=None (models/fusion.py:292-297)
    q = q + _lin(sd, lp + ".cross_attention.W_o", ctx)
    n = _ln(sd, lp + ".norm_ffn", q)
    q = q + _lin(sd, lp + ".ffn.3", F.relu(_lin(sd, lp + ".ffn.0", n)))  # :257-263
    return q, w


def fusion(sd, feats, text_features, text_mask, num_heads, p="fusion"):
    """MultimodalFusion.forward (models/fusion.py:252-336)."""
    img = image_projector(sd, feats)
    q = text_features
    weights = []
    layer = 0
    while (p + f".cross_attention.layers.{layer}.norm_query.weight") in sd:
        q, w = cross_layer(sd, p + f".cross_attention.layers.{layer}", q, img, num_heads)
        weights.append(w)
        layer += 1
    fused, att_pooled, txt_pooled = fusion_tail(sd, q, text_features, text_mask, p)
    aux = {"cross_attention_weights": weights, "image_projected": img,
           "attended_pooled": att_pooled, "text_pooled": txt_pooled}
    return fused, aux


def fusion_tail(sd, q, text_features, text_mask, p="fusion"):
    """MultimodalFusion.forward after the cross-attention layers (models/fusion.py:303-326): masked mean pools of the
    attended and the plain text features, gate (or sum), output LayerNorm -> (fused, att_pooled, txt_pooled)."""
    if text_mask is not None:                                            # :303-313
        m = text_mask.unsqueeze(-1).float()
        den = m.sum(dim=1).clamp(min=1)
        att_pooled = (q * m).sum(dim=1) / den
        txt_pooled = (text_features * m).sum(dim=1) / den
    else:
        att_pooled = q.mean(dim=1)
        txt_pooled = text_features.mean(dim=1)
    if (p + ".gate.gate.0.weight") in sd:                                # :159-166
        g = torch.sigmoid(_lin(sd, p + ".gate.gate.0", torch.cat([att_pooled, txt_pooled], dim=-1)))
        fused = g * att_pooled + (1 - g) * txt_pooled
    else:
        fused = att_pooled + txt_pooled                                  # :322
    return _ln(sd, p + ".output_norm", fused), att_pooled, txt_pooled   # :326


def answer_head(sd, fused, p="answer_head.classifier"):
    """AnswerHead.forward: 256->512->256->1000 (models/vqa_model.py:73-83,94-104)."""
    x = F.relu(_lin(sd, p + ".0", fused))
    x = F.relu(_lin(sd, p + ".3", x))
    return _lin(sd, p + ".6", x)


# --------------------------------------------------------------------------- whole model
def vqa_forward(sd: Dict[str, torch.Tensor], images: torch.Tensor, token_ids: torch.Tensor,
                attention_mask: Optional[torch.Tensor] = None, num_heads: int = 8,
                return_aux: bool = False, taps: Optional[dict] = None
                ) -> Tuple[torch.Tensor, Optional[dict]]:
    """VQAModel.forward in eval mode (models/vqa_model.py:243-311).

    ``sd`` is the reference ``state_dict`` (fp32 CPU tensors).  ``num_heads`` is the
    only hyper-parameter not recoverable from tensor shapes.
    """
    with torch.no_grad():
        feats = image_encoder(sd, images.float(), taps)
        text_features, text_pooled = text_encoder(sd, token_ids, attention_mask, num_heads)
        fused, faux = fusion(sd, feats, text_features, attention_mask, num_heads)
        logits = answer_head(sd, fused)
    if not return_aux:
        return logits, None
    aux = {"image_features": feats, "text_features": text_features,
           "text_pooled": text_pooled, "fused": fused}
    aux.update(faux)  # fusion's own text_pooled overrides (models/vqa_model.py:301-309)
    return logits, aux


def predict_topk(logits: torch.Tensor, top_k: int = 5):
    """softmax + topk (models/vqa_model.py:336-337, api/inference.py:231-234)."""
    probs = F.softmax(logits, dim=-1)
    top_probs, top_idx = probs.topk(top_k, dim=-1)
    return top_idx, top_probs
