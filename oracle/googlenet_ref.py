"""ORACLE (test infrastructure only — never imported by the product path).

Functional fp32 PyTorch restatement of the reference's stage-2 classifier, operating on a reference-format
state_dict (344 tensors, keys prefixed `googlenet.`):

  分类/test.py:64-73 (== 分类/ROI_main.py:86-95)  GoogLeNetClassifier: torchvision googlenet(pretrained=True)
      with fc replaced by Linear(1024, num_classes).  pretrained=True implies transform_input=True and
      aux_logits=False in eval, so the aux heads never run and are absent from the state_dict.

The arithmetic lives in the third-party dependency torchvision (un-pinned by the reference; 0.26.0 in this
image), module torchvision/models/googlenet.py: GoogLeNet._transform_input, GoogLeNet._forward, Inception
(the "5x5" branch is a 3x3 conv), BasicConv2d (bias-free Conv2d + BatchNorm2d(eps=1e-3) + ReLU).  Pool
geometry: maxpool1-3 = MaxPool2d(3, stride 2, ceil_mode), maxpool4 = MaxPool2d(2, stride 2, ceil_mode),
Inception branch4 pool = MaxPool2d(3, stride 1, padding 1, ceil_mode).

Pinned by tests/test_oracle_nets.py against torchvision's own module (present in the image, also on the GPU
box) and against tests/golden/googlenet_golden.npz.
"""
import torch
import torch.nn.functional as F

BN_EPS = 1e-3
INCEPTIONS = ["inception3a", "inception3b", "inception4a", "inception4b", "inception4c", "inception4d",
              "inception4e", "inception5a", "inception5b"]


def basic_conv(x, sd, p, stride=1, padding=0, training=False):
    y = F.conv2d(x, sd[p + ".conv.weight"], None, stride=stride, padding=padding)
    if training:
        y = F.batch_norm(y, None, None, sd[p + ".bn.weight"], sd[p + ".bn.bias"], True, 0.0, BN_EPS)
    else:
        y = F.batch_norm(y, sd[p + ".bn.running_mean"], sd[p + ".bn.running_var"], sd[p + ".bn.weight"],
                         sd[p + ".bn.bias"], False, 0.0, BN_EPS)
    return F.relu(y)


def inception(x, sd, p, training=False):
    b1 = basic_conv(x, sd, p + ".branch1", training=training)
    b2 = basic_conv(basic_conv(x, sd, p + ".branch2.0", training=training), sd, p + ".branch2.1", padding=1,
                    training=training)
    b3 = basic_conv(basic_conv(x, sd, p + ".branch3.0", training=training), sd, p + ".branch3.1", padding=1,
                    training=training)
    b4 = basic_conv(F.max_pool2d(x, 3, stride=1, padding=1, ceil_mode=True), sd, p + ".branch4.1",
                    training=training)
    return torch.cat([b1, b2, b3, b4], dim=1)


def transform_input(x):
    """GoogLeNet._transform_input with transform_input=True."""
    c0 = x[:, 0:1] * (0.229 / 0.5) + (0.485 - 0.5) / 0.5
    c1 = x[:, 1:2] * (0.224 / 0.5) + (0.456 - 0.5) / 0.5
    c2 = x[:, 2:3] * (0.225 / 0.5) + (0.406 - 0.5) / 0.5
    return torch.cat((c0, c1, c2), 1)


def googlenet_forward(sd, x, prefix="googlenet.", training=False):
    """fp32 NCHW [B,3,224,224] in [0,1] -> logits [B, num_classes] (a float64 input is evaluated in float64)."""
    g = {k[len(prefix):]: v for k, v in sd.items() if k.startswith(prefix)}
    x = transform_input(x if x.dtype == torch.float64 else x.float())
    x = basic_conv(x, g, "conv1", stride=2, padding=3, training=training)
    x = F.max_pool2d(x, 3, stride=2, ceil_mode=True)
    x = basic_conv(x, g, "conv2", training=training)
    x = basic_conv(x, g, "conv3", padding=1, training=training)
    x = F.max_pool2d(x, 3, stride=2, ceil_mode=True)
    x = inception(x, g, "inception3a", training)
    x = inception(x, g, "inception3b", training)
    x = F.max_pool2d(x, 3, stride=2, ceil_mode=True)
    for name in ("inception4a", "inception4b", "inception4c", "inception4d", "inception4e"):
        x = inception(x, g, name, training)
    x = F.max_pool2d(x, 2, stride=2, ceil_mode=True)
    x = inception(x, g, "inception5a", training)
    x = inception(x, g, "inception5b", training)
    x = torch.flatten(F.adaptive_avg_pool2d(x, 1), 1)
    return F.linear(x, g["fc.weight"], g["fc.bias"])  # dropout is identity in eval
