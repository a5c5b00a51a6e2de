"""fp32 functional restatement of the reference's IR-SE backbone (tests only), built on oracle/lfan_oracle.py.

The oracle covers bottleneck_IR (any get_blocks table, strided identity shortcut included); this adds the SE
unit of models/arcface_model.py: SEModule (:23-41) and bottleneck_IR_SE (:63-84), whose res_layer ends in
SEModule(depth, 16) as res_layer.5.  Works on a reference-layout state_dict, like the oracle.  Pinned against the
reference's own Backbone by tests/test_backbone_variants_host.py where oracle/_ref is staged.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from oracle import lfan_oracle as O


def se_module(sd, p, x):
    """SEModule.forward, arcface_model.py:23-41: x * sigmoid(fc2(relu(fc1(avg_pool(x)))))."""
    m = x.mean(dim=(2, 3), keepdim=True)                                                    # AdaptiveAvgPool2d(1)
    h = torch.relu(F.conv2d(m, sd[p + ".fc1.weight"]))
    return x * torch.sigmoid(F.conv2d(h, sd[p + ".fc2.weight"]))


def ir_se_unit(sd, p, x, cin, depth, stride):
    """bottleneck_IR_SE.forward, arcface_model.py:63-84 (shortcut_layer as in bottleneck_IR)."""
    if cin == depth:
        shortcut = x[:, :, ::stride, ::stride]                                              # MaxPool2d(1, stride)
    else:
        shortcut = O._bn_eval(sd, p + ".shortcut_layer.1", F.conv2d(x, sd[p + ".shortcut_layer.0.weight"], None, stride))
    r = O._bn_eval(sd, p + ".res_layer.0", x)
    r = O._prelu(F.conv2d(r, sd[p + ".res_layer.1.weight"], None, 1, 1), sd[p + ".res_layer.2.weight"])
    r = O._bn_eval(sd, p + ".res_layer.4", F.conv2d(r, sd[p + ".res_layer.3.weight"], None, stride, 1))
    return se_module(sd, p + ".res_layer.5", r) + shortcut


def ir_forward(sd, x, prefix="", units=O.IR50_UNITS, se=False):
    """Backbone.forward (arcface_model.py:147-151) for mode 'ir' (oracle.ir50_forward) or 'ir_se'."""
    if not se:
        return O.ir50_forward(sd, x, prefix, units=units)
    p = prefix
    h = F.conv2d(x, sd[p + "input_layer.0.weight"], None, 1, 1)
    h = O._prelu(O._bn_eval(sd, p + "input_layer.1", h), sd[p + "input_layer.2.weight"])
    for i, (cin, depth, stride) in enumerate(units):
        h = ir_se_unit(sd, f"{p}body.{i}", h, cin, depth, stride)
    h = O._bn_eval(sd, p + "output_layer.0", h).reshape(h.shape[0], -1)
    h = O._bn_eval(sd, p + "output_layer.4", F.linear(h, sd[p + "output_layer.3.weight"], sd[p + "output_layer.3.bias"]))
    return h / torch.norm(h, 2, 1, True)
