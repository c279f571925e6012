"""cnn_linear heads on the B200 backend -- drop-in for deepards/models/torch_cnn_linear_network.py.

`CNNLinearNetwork(breath_block, sequence_size, metadata_features)` (torch_cnn_linear_network.py:92-113) and
`CNNSingleBreathLinearNetwork(breath_block)` (:49-67): same attributes (`breath_block`, `linear_final`,
`seq_size`), same `forward(x, metadata)` contract and error for a wrong window length.

Where the reference loops over the batch in Python and calls the backbone once per 20-breath sequence (so that
BatchNorm sees one sequence at a time), this implementation runs ALL B*20 breaths through one kernel plan whose
BatchNorm kernels take their statistics per group of 20 consecutive breaths -- same numbers, one launch
sequence, no O(B^2) torch.cat.
"""
import torch
import torch.nn as nn

from . import autograd as _ag
from .resnet import _Picklable


def _drop_key(backbone):
    feats = getattr(backbone, "features", None)
    return feats._drop_key() if feats is not None and hasattr(feats, "_drop_key") else ()


class _HeadBase(_Picklable, nn.Module):
    def _check(self, x):
        # input should be in shape: (batches, breaths in seq, chans, 224)
        if x.shape[-1] != 224:
            raise Exception('input breaths must have sequence length of 224')
        if x.dim() != 4 or x.shape[2] != 1:
            raise NotImplementedError("deepards_b200 heads take (B, breaths, 1, 224) inputs, got %s" % (tuple(x.shape),))
        if not hasattr(self.breath_block, "network_name") or not hasattr(self.breath_block, "precision"):
            raise TypeError("breath_block must be a deepards_b200 backbone (resnet18 / densenet18 from this package)")

    def _sequence_features(self, x):
        """(B, S, 1, 224) -> pooled backbone features (B, S, F): ONE batched plan with BatchNorm group S, i.e. what the
        reference's `breath_block(x[i])` loop + torch.cat produces (torch_cnn_linear_network.py:22-24)."""
        self._check(x)
        feat = _ag.run_plan(self, self.breath_block, None, x, x.shape[1], "backbone", _drop_key(self.breath_block))
        return feat.view(x.shape[0], x.shape[1], -1)

    @property
    def precision(self):
        return self.breath_block.precision

    @precision.setter
    def precision(self, value):
        self.breath_block.precision = value


class CNNLinearNetwork(_HeadBase):
    """Flatten the 20 x F features of each sequence and classify it with one Linear layer."""

    def __init__(self, breath_block, sequence_size, metadata_features):
        super(CNNLinearNetwork, self).__init__()
        self.seq_size = 224
        self.breath_block = breath_block
        self.linear_final = nn.Linear(self.breath_block.n_out_filters * sequence_size + metadata_features, 2)

    def forward(self, x, metadata=None):
        self._check(x)
        return _ag.run_plan(self, self.breath_block, self.linear_final, x, x.shape[1], "cnn_linear",
                            _drop_key(self.breath_block))

    def _head(self, feat):
        """(B, S, F) features -> (B, 2) logits in torch: what the plan's fused linear computes.  DataParallelTrainer uses
        it with a caller-supplied criterion; forward() keeps the fused head."""
        return self.linear_final(feat.reshape(feat.shape[0], -1))


class CNNSingleBreathLinearNetwork(_HeadBase):
    """One prediction per breath: Linear(F, 2) on every breath's pooled features -> (B, breaths, 2)."""

    def __init__(self, breath_block):
        super(CNNSingleBreathLinearNetwork, self).__init__()
        self.seq_size = 224
        self.breath_block = breath_block
        self.linear_final = nn.Linear(self.breath_block.n_out_filters, 2)

    def forward(self, x, metadata=None):
        self._check(x)
        return _ag.run_plan(self, self.breath_block, self.linear_final, x, x.shape[1], "per_breath",
                            _drop_key(self.breath_block))

    def _head(self, feat):
        """(B, S, F) features -> (B, S, 2) logits in torch (see CNNLinearNetwork._head)."""
        return self.linear_final(feat)


# ---- sibling heads on the same backbone (SURVEY.md 8f-4): the backbone runs as one batched plan, the few-kB head
# ---- arithmetic behind it stays in torch.  `_head(feat)` is that arithmetic: forward() and DataParallelTrainer both
# ---- call it on the plan's pooled features ----------------------------------------------------------------------
class CNNLinearToMean(_HeadBase):
    """Linear(F, 2) on the mean of the sequence's breath features (torch_cnn_linear_network.py:7-25)."""

    def __init__(self, breath_block):
        super(CNNLinearToMean, self).__init__()
        self.seq_size = 224
        self.breath_block = breath_block
        self.linear_final = nn.Linear(self.breath_block.n_out_filters, 2)

    def forward(self, x, metadata=None):
        return self._head(self._sequence_features(x))

    def _head(self, feat):
        return self.linear_final(torch.mean(feat, dim=1))


class CNNLinearComprToRF(_HeadBase):
    """Linear(F, 2) on the per-feature median over the sequence (torch_cnn_linear_network.py:28-46)."""

    def __init__(self, breath_block):
        super(CNNLinearComprToRF, self).__init__()
        self.seq_size = 224
        self.breath_block = breath_block
        self.linear_final = nn.Linear(self.breath_block.n_out_filters, 2)

    def forward(self, x, metadata=None):
        return self._head(self._sequence_features(x))

    def _head(self, feat):
        return self.linear_final(torch.median(feat, dim=1)[0])


class CNNDoubleLinearNetwork(_HeadBase):
    """Linear(F, 2) per breath, then Linear(2 * S, 2) per sequence (torch_cnn_linear_network.py:70-89)."""

    def __init__(self, breath_block, sequence_size, metadata_features):
        super(CNNDoubleLinearNetwork, self).__init__()
        self.seq_size = 224
        self.breath_block = breath_block
        self.linear_intermediate = nn.Linear(self.breath_block.n_out_filters, 2)
        self.linear_final = nn.Linear(2 * sequence_size + metadata_features, 2)

    def forward(self, x, metadata=None):
        return self._head(self._sequence_features(x))

    def _head(self, feat):
        return self.linear_final(self.linear_intermediate(feat).reshape(feat.shape[0], -1))


class CNNRegressor(_HeadBase):
    """Linear(F, n_final_features) on a FLAT batch of breaths: BatchNorm group = the whole batch
    (torch_cnn_bm_regressor.py:6-19).  x: (N, 1, 224)."""

    def __init__(self, breath_block, n_final_features):
        super(CNNRegressor, self).__init__()
        self.seq_size = 224
        self.breath_block = breath_block
        self.linear_final = nn.Linear(breath_block.n_out_filters, n_final_features)

    def forward(self, x, metadata=None):
        # input should be in shape: (batches, chans, 224)
        if x.shape[-1] != 224:
            raise Exception('input breaths must have sequence length of 224')
        return self._head(self.breath_block(x))

    def _head(self, feat):
        return self.linear_final(feat.squeeze())


class CNNLSTMNetwork(_HeadBase):
    """LSTM over the sequence's breath features, Linear(hidden, 2) on every step (torch_cnn_lstm_combo.py:6-50).
    forward(x, metadata, hx_cx) -> (B, S, 2), (hx, cx).  Breath metadata is not supported on this backend (the reference
    ignores it when it is NaN, which is what the cnn_lstm experiment files feed, torch_cnn_lstm_combo.py:36)."""

    def __init__(self, breath_block, metadata_features, bm_to_linear, lstm_hidden_units):
        super(CNNLSTMNetwork, self).__init__()
        if metadata_features:
            raise NotImplementedError("deepards_b200: metadata_features > 0 is not implemented")
        self.seq_size = 224
        self.breath_block = breath_block
        self.lstm_hidden_units = lstm_hidden_units
        self.lstm_layers = 1
        self.bm_to_linear = bm_to_linear
        self.lstm = nn.LSTM(breath_block.n_out_filters, self.lstm_hidden_units, num_layers=self.lstm_layers, batch_first=True)
        self.linear_final = nn.Linear(self.lstm_hidden_units, 2)

    def forward(self, x, metadata=None, hx_cx=None):
        if metadata is not None and not torch.any(torch.isnan(metadata)):
            raise NotImplementedError("deepards_b200: breath metadata is not implemented on this backend")
        return self._head(self._sequence_features(x), hx_cx)

    def _head(self, feat, hx_cx=None):
        # the fp32 path promises the reference's fp32 numbers: keep cuDNN's LSTM GEMMs out of TF32 (its default)
        with torch.backends.cudnn.flags(allow_tf32=_ag.module_precision(self) == "bf16"):
            out, (hx, cx) = self.lstm(feat, hx_cx)
        return self.linear_final(out), (hx, cx)


# ---- transformer head (deepards/models/cnn_transformer.py:8-44 over deepards/models/transformer.py) -------------------
class _SelfAttention(nn.Module):
    """Multi-head scaled dot-product attention with the reference's parameter names (transformer.py:13-58)."""

    def __init__(self, input_size, hidden_size, num_heads):
        super(_SelfAttention, self).__init__()
        if hidden_size % num_heads:
            raise ValueError("hidden_size must be a multiple of num_heads")
        self.num_heads, self.head_size = num_heads, hidden_size // num_heads
        self.q_linear = nn.Linear(input_size, hidden_size)
        self.k_linear = nn.Linear(input_size, hidden_size)
        self.v_linear = nn.Linear(input_size, hidden_size)
        self.joint_linear = nn.Linear(hidden_size, input_size)
        self.weights = None

    def forward(self, x):
        b, s, _ = x.shape
        split = lambda t: t.view(b, s, self.num_heads, self.head_size).permute(0, 2, 1, 3)  # noqa: E731
        q, k, v = split(self.q_linear(x)), split(self.k_linear(x)), split(self.v_linear(x))
        att = torch.softmax(torch.einsum("bhid,bhjd->bhij", q, k) / float(self.head_size) ** 0.5, dim=-1)
        self.weights = att  # the reference keeps the last attention map for visualisation
        mixed = torch.einsum("bhij,bhjd->bihd", att, v).reshape(b, s, self.num_heads * self.head_size)
        return self.joint_linear(mixed)


class _TransformerBlock(nn.Module):
    """attention -> dropout -> +x -> LayerNorm; feed-forward(ReLU) -> dropout -> +x (the block INPUT, as the reference
    does, transformer.py:89-91) -> LayerNorm."""

    def __init__(self, input_size, hidden_size, num_heads, dropout):
        super(_TransformerBlock, self).__init__()
        self.attention = _SelfAttention(input_size, hidden_size, num_heads)
        self.attention_norm = nn.LayerNorm(input_size)
        self.attention_dropout = nn.Dropout(dropout)
        self.ff = nn.Sequential(nn.Linear(input_size, hidden_size), nn.ReLU(), nn.Linear(hidden_size, input_size),
                                nn.Dropout(dropout))
        self.ff_norm = nn.LayerNorm(input_size)

    def forward(self, x):
        attended = self.attention_norm(self.attention_dropout(self.attention(x)) + x)
        return self.ff_norm(self.ff(attended) + x)


class _Transformer(nn.Module):
    def __init__(self, input_size, hidden_size, num_blocks, num_heads, dropout=.2):
        super(_Transformer, self).__init__()
        self.blocks = nn.Sequential(*[_TransformerBlock(input_size, hidden_size, num_heads, dropout)
                                      for _ in range(num_blocks)])

    def forward(self, x):
        return self.blocks(x)


class CNNTransformerNetwork(_HeadBase):
    """Transformer over the sequence's breath features, Linear(F, 2) on every position -> (B, S, 2)
    (cnn_transformer.py:8-44).  The backbone is ONE batched plan with BatchNorm group S; the transformer (a few hundred
    kB of weights, S = 20 tokens) stays in torch.  Breath metadata is not supported on this backend (the reference skips
    it when it is NaN, which is what the experiment files feed, cnn_transformer.py:31)."""

    def __init__(self, breath_block, metadata_features, bm_to_linear, hidden_units, num_blocks):
        super(CNNTransformerNetwork, self).__init__()
        if metadata_features:
            raise NotImplementedError("deepards_b200: metadata_features > 0 is not implemented")
        self.seq_size = 224
        self.breath_block = breath_block
        self.bm_to_linear = bm_to_linear
        self.transformer = _Transformer(breath_block.n_out_filters, hidden_units, num_blocks, 4)
        self.linear_final = nn.Linear(breath_block.n_out_filters, 2)

    def forward(self, x, metadata=None):
        if metadata is not None and not torch.any(torch.isnan(metadata)):
            raise NotImplementedError("deepards_b200: breath metadata is not implemented on this backend")
        return self._head(self._sequence_features(x))

    def _head(self, feat):
        with _no_tf32(self):
            return self.linear_final(self.transformer(feat))


class _no_tf32(object):
    """fp32 plans promise the reference's fp32 numbers: keep cuBLAS out of TF32 for the head's small GEMMs."""

    def __init__(self, mod):
        self.on = _ag.module_precision(mod) != "bf16"

    def __enter__(self):
        self.prev = torch.backends.cuda.matmul.allow_tf32
        if self.on:
            torch.backends.cuda.matmul.allow_tf32 = False

    def __exit__(self, *a):
        torch.backends.cuda.matmul.allow_tf32 = self.prev
