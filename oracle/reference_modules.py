"""fp32 torch.nn restatement of the reference's hot-path MODULES — TEST INFRASTRUCTURE, NOT PRODUCT CODE.

`visual_encoder_oracle.py` restates the reference's forward as functions on a state dict; the training tests need the
reference as modules instead: the same module tree and attribute names (so forward hooks, `named_parameters()` and
state dicts line up key for key with the drop-ins), batch-statistics BatchNorm under `model.train()`, and the
reference's dropout modules at the reference's call sites, drawn in the reference's order (so a seeded run draws the
same masks).  Autograd through these modules is the reference's own gradient.

Classes and line citations follow SBL_Multilingual_Lip_reading/transformer/ (video_frontend.py, encoder.py,
attention.py, module.py, utils.py) and, for `Stage1Transformer`, the stage-1 sub-project's transformer/transformer.py;
that sub-project's frontend and encoder classes are the same as SBL's (SURVEY.md §2.1).

Pinning: tests/test_oracle_golden.py runs these modules on the golden inputs and checks them against the outputs the
reference modules themselves produced (tests/golden/reference_outputs.npz) and against the reference's state-dict
contract (tests/golden/state_dict_contract.json).  Only `tests/` import this file.
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F


# ----------------------------------------------------------------------------------------------
# visual frontend  (transformer/video_frontend.py)
# ----------------------------------------------------------------------------------------------
def conv3x3(in_planes, out_planes, stride=1):
    """:10-12"""
    return nn.Conv2d(in_planes, out_planes, kernel_size=3, stride=stride, padding=1, bias=False)


class BasicBlock(nn.Module):
    """:15-41"""
    expansion = 1

    def __init__(self, inplanes, planes, stride=1, downsample=None):
        super().__init__()
        self.conv1 = conv3x3(inplanes, planes, stride)
        self.bn1 = nn.BatchNorm2d(planes)
        self.relu = nn.ReLU(inplace=True)
        self.conv2 = conv3x3(planes, planes)
        self.bn2 = nn.BatchNorm2d(planes)
        self.downsample = downsample
        self.stride = stride

    def forward(self, x):
        residual = x
        out = self.conv1(x)
        out = self.bn1(out)
        out = self.relu(out)
        out = self.conv2(out)
        out = self.bn2(out)
        if self.downsample is not None:
            residual = self.downsample(x)
        out += residual
        out = self.relu(out)
        return out


class ResNet(nn.Module):
    """ResNet trunk without stem, :44-89."""

    def __init__(self, block, layers):
        self.inplanes = 64
        super().__init__()
        self.layer1 = self._make_layer(block, 64, layers[0])
        self.layer2 = self._make_layer(block, 128, layers[1], stride=2)
        self.layer3 = self._make_layer(block, 256, layers[2], stride=2)
        self.layer4 = self._make_layer(block, 512, layers[3], stride=2)
        self.avgpool = nn.AdaptiveAvgPool2d(1)
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                n = m.kernel_size[0] * m.kernel_size[1] * m.out_channels
                m.weight.data.normal_(0, math.sqrt(2. / n))
            elif isinstance(m, (nn.BatchNorm2d, nn.BatchNorm1d)):
                m.weight.data.fill_(1)
                m.bias.data.zero_()

    def _make_layer(self, block, planes, blocks, stride=1):
        downsample = None
        if stride != 1 or self.inplanes != planes * block.expansion:
            downsample = nn.Sequential(
                nn.Conv2d(self.inplanes, planes * block.expansion, kernel_size=1, stride=stride, bias=False),
                nn.BatchNorm2d(planes * block.expansion),
            )
        layers = [block(self.inplanes, planes, stride, downsample)]
        self.inplanes = planes * block.expansion
        for _ in range(1, blocks):
            layers.append(block(self.inplanes, planes))
        return nn.Sequential(*layers)

    def forward(self, x):
        x = self.layer1(x)
        x = self.layer2(x)
        x = self.layer3(x)
        x = self.layer4(x)
        x = self.avgpool(x)
        return x.view(x.size(0), -1)


class Lipreading(nn.Module):
    """:91-157.  forward(x [N,1,T,88,88]) -> [N,T,512], with the always-on `F.dropout(x, p=0.5)` of :122 (the functional
    default training=True: active under model.eval() too); `_frontend_forward` is everything before it."""

    def __init__(self):
        super().__init__()
        self.inputDim = 512
        self.frontend3D = nn.Sequential(
            nn.Conv3d(1, 64, kernel_size=(5, 7, 7), stride=(1, 2, 2), padding=(2, 3, 3), bias=False),
            nn.BatchNorm3d(64),
            nn.ReLU(True),
            nn.MaxPool3d(kernel_size=(1, 3, 3), stride=(1, 2, 2), padding=(0, 1, 1)),
        )
        self.resnet18 = ResNet(BasicBlock, [2, 2, 2, 2])
        self._initialize_weights()

    def _frontend_forward(self, x):
        x = self.frontend3D(x)
        x = x.transpose(1, 2).contiguous()
        x = x.view(-1, 64, x.size(3), x.size(4))
        return self.resnet18(x)

    def forward(self, x):
        frame_len = x.size(2)
        x = self._frontend_forward(x)
        x = F.dropout(x, p=0.5)
        return x.view(-1, frame_len, self.inputDim)

    def _initialize_weights(self):
        for m in self.modules():
            if isinstance(m, (nn.Conv3d, nn.Conv2d, nn.Conv1d)):
                n = math.prod(m.kernel_size) * m.out_channels
                m.weight.data.normal_(0, math.sqrt(2. / n))
                if m.bias is not None:
                    m.bias.data.zero_()
            elif isinstance(m, (nn.BatchNorm3d, nn.BatchNorm2d, nn.BatchNorm1d)):
                m.weight.data.fill_(1)
                m.bias.data.zero_()


# ----------------------------------------------------------------------------------------------
# transformer encoder  (transformer/encoder.py, attention.py, module.py, utils.py)
# ----------------------------------------------------------------------------------------------
def get_non_pad_mask(padded_input, input_lengths):
    """utils.py:98-113 -> [N,T,1], 1 where t < length."""
    mask = padded_input.new_ones(padded_input.size()[:-1])
    for i in range(padded_input.size(0)):
        mask[i, input_lengths[i]:] = 0
    return mask.unsqueeze(-1)


def get_attn_pad_mask(padded_input, input_lengths, expand_length):
    """utils.py:140-147 -> bool [N,expand_length,T], True where KEY t >= length."""
    pad_mask = get_non_pad_mask(padded_input, input_lengths).squeeze(-1).lt(1)
    return pad_mask.unsqueeze(1).expand(-1, expand_length, -1)


class PositionalEncoding(nn.Module):
    """module.py:8-32"""

    def __init__(self, d_model, max_len=5000):
        super().__init__()
        pe = torch.zeros(max_len, d_model, requires_grad=False)
        position = torch.arange(0, max_len).unsqueeze(1).float()
        div_term = torch.exp(torch.arange(0, d_model, 2).float() * -(math.log(10000.0) / d_model))
        pe[:, 0::2] = torch.sin(position * div_term)
        pe[:, 1::2] = torch.cos(position * div_term)
        self.register_buffer("pe", pe.unsqueeze(0))

    def forward(self, input):
        return self.pe[:, :input.size(1)]


class ScaledDotProductAttention(nn.Module):
    """attention.py:63-83: the attention-probability dropout is drawn on [n_head*N, T, T]."""

    def __init__(self, temperature, attn_dropout=0.1):
        super().__init__()
        self.temperature = temperature
        self.dropout = nn.Dropout(attn_dropout)
        self.softmax = nn.Softmax(dim=2)

    def forward(self, q, k, v, mask=None):
        attn = torch.bmm(q, k.transpose(1, 2)) / self.temperature
        if mask is not None:
            attn = attn.masked_fill(mask, -np.inf)
        attn = self.softmax(attn)
        attn = self.dropout(attn)
        return torch.bmm(attn, v), attn


class MultiHeadAttention(nn.Module):
    """attention.py:9-60"""

    def __init__(self, n_head, d_model, d_k, d_v, dropout=0.1):
        super().__init__()
        self.n_head, self.d_k, self.d_v = n_head, d_k, d_v
        self.w_qs = nn.Linear(d_model, n_head * d_k)
        self.w_ks = nn.Linear(d_model, n_head * d_k)
        self.w_vs = nn.Linear(d_model, n_head * d_v)
        nn.init.normal_(self.w_qs.weight, mean=0, std=np.sqrt(2.0 / (d_model + d_k)))
        nn.init.normal_(self.w_ks.weight, mean=0, std=np.sqrt(2.0 / (d_model + d_k)))
        nn.init.normal_(self.w_vs.weight, mean=0, std=np.sqrt(2.0 / (d_model + d_v)))
        self.attention = ScaledDotProductAttention(temperature=np.power(d_k, 0.5), attn_dropout=dropout)
        self.layer_norm = nn.LayerNorm(d_model)
        self.fc = nn.Linear(n_head * d_v, d_model)
        nn.init.xavier_normal_(self.fc.weight)
        self.dropout = nn.Dropout(dropout)

    def forward(self, q, k, v, mask=None):
        d_k, d_v, n_head = self.d_k, self.d_v, self.n_head
        sz_b, len_q, _ = q.size()
        len_k, len_v = k.size(1), v.size(1)
        residual = q
        q = self.w_qs(q).view(sz_b, len_q, n_head, d_k)
        k = self.w_ks(k).view(sz_b, len_k, n_head, d_k)
        v = self.w_vs(v).view(sz_b, len_v, n_head, d_v)
        q = q.permute(2, 0, 1, 3).contiguous().view(-1, len_q, d_k)   # (n_head*b) x T x d_k, index h*b + i
        k = k.permute(2, 0, 1, 3).contiguous().view(-1, len_k, d_k)
        v = v.permute(2, 0, 1, 3).contiguous().view(-1, len_v, d_v)
        if mask is not None:
            mask = mask.repeat(n_head, 1, 1)
        output, attn = self.attention(q, k, v, mask=mask)
        output = output.view(n_head, sz_b, len_q, d_v)
        output = output.permute(1, 2, 0, 3).contiguous().view(sz_b, len_q, -1)
        output = self.dropout(self.fc(output))
        output = self.layer_norm(output + residual)
        return output, attn


class PositionwiseFeedForward(nn.Module):
    """module.py:35-52"""

    def __init__(self, d_model, d_ff, dropout=0.1):
        super().__init__()
        self.w_1 = nn.Linear(d_model, d_ff)
        self.w_2 = nn.Linear(d_ff, d_model)
        self.dropout = nn.Dropout(dropout)
        self.layer_norm = nn.LayerNorm(d_model)

    def forward(self, x):
        residual = x
        output = self.w_2(F.relu(self.w_1(x)))
        output = self.dropout(output)
        return self.layer_norm(output + residual)


class EncoderLayer(nn.Module):
    """encoder.py:70-91"""

    def __init__(self, d_model, d_inner, n_head, d_k, d_v, dropout=0.1):
        super().__init__()
        self.slf_attn = MultiHeadAttention(n_head, d_model, d_k, d_v, dropout=dropout)
        self.pos_ffn = PositionwiseFeedForward(d_model, d_inner, dropout=dropout)

    def forward(self, enc_input, non_pad_mask=None, slf_attn_mask=None):
        enc_output, enc_slf_attn = self.slf_attn(enc_input, enc_input, enc_input, mask=slf_attn_mask)
        enc_output = enc_output * non_pad_mask
        enc_output = self.pos_ffn(enc_output)
        enc_output = enc_output * non_pad_mask
        return enc_output, enc_slf_attn


class Encoder(nn.Module):
    """encoder.py:8-67.  Returns (enc_output,) or (enc_output, [attn per layer]) with return_attns=True."""

    def __init__(self, d_input, n_layers, n_head, d_k, d_v, d_model, d_inner, dropout=0.1, pe_maxlen=5000):
        super().__init__()
        self.linear_in = nn.Linear(d_input, d_model)
        self.layer_norm_in = nn.LayerNorm(d_model)
        self.positional_encoding = PositionalEncoding(d_model, max_len=pe_maxlen)
        self.dropout = nn.Dropout(dropout)
        self.layer_stack = nn.ModuleList([
            EncoderLayer(d_model, d_inner, n_head, d_k, d_v, dropout=dropout) for _ in range(n_layers)])

    def forward(self, padded_input, input_lengths, return_attns=False):
        enc_slf_attn_list = []
        non_pad_mask = get_non_pad_mask(padded_input, input_lengths=input_lengths)
        length = padded_input.size(1)
        slf_attn_mask = get_attn_pad_mask(padded_input, input_lengths, length)
        enc_output = self.dropout(self.layer_norm_in(self.linear_in(padded_input)) +
                                  self.positional_encoding(padded_input))
        for enc_layer in self.layer_stack:
            enc_output, enc_slf_attn = enc_layer(enc_output, non_pad_mask=non_pad_mask, slf_attn_mask=slf_attn_mask)
            if return_attns:
                enc_slf_attn_list += [enc_slf_attn]
        if return_attns:
            return enc_output, enc_slf_attn_list
        return (enc_output,)


# ----------------------------------------------------------------------------------------------
# stage-1 pre-training model  (the stage-1 sub-project's transformer/transformer.py:6-38)
# ----------------------------------------------------------------------------------------------
class Stage1Transformer(nn.Module):
    """Frontend + `encoder_v` + `fc_1500` word head + `fc_2` language head, with the reference's attribute names.  Its
    forward cannot run as published (SURVEY.md §0), so only the modules are restated; callers apply the heads."""

    def __init__(self, encoder):
        super().__init__()
        self.visual_frontend = Lipreading()
        self.encoder_v = encoder
        self.fc_1500 = nn.Linear(512, 1500)
        self.fc_2 = nn.Linear(512, 2)


def build_stage1(state_dict=None, n_layers_enc=3, seed=7):
    """The stage-1 model as the sub-project's train.py:37-41 builds it; `state_dict` is loaded non-strictly."""
    torch.manual_seed(seed)
    enc = Encoder(512, n_layers_enc, 8, 64, 64, 512, 2048, dropout=0.1, pe_maxlen=5000)
    model = Stage1Transformer(enc)
    if state_dict is not None:
        _, unexpected = model.load_state_dict(state_dict, strict=False)
        assert not unexpected, unexpected
    return model
