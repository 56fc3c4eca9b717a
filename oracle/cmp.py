"""ORACLE (test infrastructure): CMP sparse-to-dense flow network, inference forward only.

Restates (module/parameter names identical, so reference checkpoints' `state_dict` loads after stripping the
`module.` prefix added by FixModule, models/cmp/models/modules/others.py:3-10):
  CMP.forward                /root/reference/MOFA-Video-Traj/models/cmp/models/modules/cmp.py:27-35
  ResNet (resnet50, layer3/4 dilated 2/4 and un-strided, conv5 1x1)   .../backbone/resnet.py:94-168
  ShallowNet (shallownet8x)  .../modules/shallownet.py:4-42
  MotionDecoderSkipLayer     .../modules/decoder.py:96-215
  Fuser.convert_flow         .../utils/visualize_utils.py:6-19   (nbins 99, fmax 50: config.yaml:22-23)
  CMP_demo.run               /root/reference/MOFA-Video-Traj/models/svdxt_featureflow_forward_controlnet_s2d_fixcmp_norefine.py:51-62

PINNED: tests/golden/cmp_small.pt is produced by running the reference's own module files on CPU
(oracle/make_goldens.py: make_cmp) with weights drawn by `seeded_state_dict` below; tests/test_oracle.py compares.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F


class Bottleneck(nn.Module):
    expansion = 4

    def __init__(self, inplanes, planes, stride=1, downsample=None):
        super().__init__()
        self.conv1 = nn.Conv2d(inplanes, planes, 1, bias=False)
        self.bn1 = nn.BatchNorm2d(planes)
        self.conv2 = nn.Conv2d(planes, planes, 3, stride=stride, padding=1, bias=False)
        self.bn2 = nn.BatchNorm2d(planes)
        self.conv3 = nn.Conv2d(planes, planes * 4, 1, bias=False)
        self.bn3 = nn.BatchNorm2d(planes * 4)
        self.downsample = downsample

    def forward(self, x):
        out = F.relu(self.bn1(self.conv1(x)))
        out = F.relu(self.bn2(self.conv2(out)))
        out = self.bn3(self.conv3(out))
        res = x if self.downsample is None else self.downsample(x)
        return F.relu(out + res)


class ResNet50Dilated(nn.Module):
    def __init__(self, output_dim):
        super().__init__()
        self.inplanes = 64
        self.conv1 = nn.Conv2d(3, 64, 7, stride=2, padding=3, bias=False)
        self.bn1 = nn.BatchNorm2d(64)
        self.maxpool = nn.MaxPool2d(3, stride=2, padding=1)
        self.layer1 = self._make_layer(64, 3)
        self.layer2 = self._make_layer(128, 4, stride=2)
        self.layer3 = self._make_layer(256, 6, stride=2)
        self.layer4 = self._make_layer(512, 3, stride=2)
        self.conv5 = nn.Conv2d(2048, output_dim, 1)
        for layer, d in ((self.layer3, 2), (self.layer4, 4)):   # resnet.py:118-127
            for n, m in layer.named_modules():
                if "conv2" in n:
                    m.dilation, m.padding, m.stride = (d, d), (d, d), (1, 1)
                elif "downsample.0" in n:
                    m.stride = (1, 1)

    def _make_layer(self, planes, blocks, stride=1):
        downsample = None
        if stride != 1 or self.inplanes != planes * 4:
            downsample = nn.Sequential(nn.Conv2d(self.inplanes, planes * 4, 1, stride=stride, bias=False),
                                       nn.BatchNorm2d(planes * 4))
        layers = [Bottleneck(self.inplanes, planes, stride, downsample)]
        self.inplanes = planes * 4
        layers += [Bottleneck(self.inplanes, planes) for _ in range(1, blocks)]
        return nn.Sequential(*layers)

    def forward(self, img):
        conv1 = F.relu(self.bn1(self.conv1(img)))
        layer1 = self.layer1(self.maxpool(conv1))
        out = self.conv5(self.layer4(self.layer3(self.layer2(layer1))))
        return out, [img, conv1, layer1]


class ShallowNet(nn.Module):
    def __init__(self, input_dim=4, output_dim=16):
        super().__init__()
        self.features = nn.Sequential(
            nn.Conv2d(input_dim, 16, 5, stride=2, padding=2), nn.BatchNorm2d(16), nn.ReLU(inplace=True),
            nn.MaxPool2d(2, stride=2),
            nn.Conv2d(16, output_dim, 3, padding=1), nn.BatchNorm2d(output_dim), nn.ReLU(inplace=True),
            nn.AvgPool2d(2, stride=2))

    def forward(self, x):
        return self.features(x)


def _cbr(cin, cout):
    return [nn.Conv2d(cin, cout, 3, padding=1), nn.BatchNorm2d(cout), nn.ReLU(inplace=True)]


class MotionDecoderSkipLayer(nn.Module):
    def __init__(self, input_dim=272, output_dim=198):
        super().__init__()
        self.decoder1 = nn.Sequential(*_cbr(input_dim, 128), *_cbr(128, 128), *_cbr(128, 128))
        for k in (2, 4, 8):
            setattr(self, f"decoder{k}", nn.Sequential(nn.MaxPool2d(k, stride=k), *_cbr(input_dim, 128),
                                                       *_cbr(128, 128), *_cbr(128, 128)))
        self.fusion8 = nn.Sequential(*_cbr(512, 256))
        self.skipconv4 = nn.Sequential(*_cbr(256, 128))
        self.fusion4 = nn.Sequential(*_cbr(256 + 128, 128))
        self.skipconv2 = nn.Sequential(*_cbr(64, 32))
        self.fusion2 = nn.Sequential(*_cbr(128 + 32, 64))
        self.head = nn.Conv2d(64, output_dim, 1)

    def forward(self, x, skip_feat):
        _, layer2, layer4 = skip_feat
        x1 = self.decoder1(x)
        up = lambda t, ref: F.interpolate(t, size=ref.shape[2:], mode="bilinear", align_corners=True)
        cat = torch.cat([x1, up(self.decoder2(x), x1), up(self.decoder4(x), x1), up(self.decoder8(x), x1)], dim=1)
        f8 = self.fusion8(cat)
        f4 = self.fusion4(torch.cat([up(f8, layer4), self.skipconv4(layer4)], dim=1))
        f2 = self.fusion2(torch.cat([up(f4, layer2), self.skipconv2(layer2)], dim=1))
        return self.head(f2)


class CMP(nn.Module):
    def __init__(self, img_enc_dim=256, sparse_enc_dim=16, output_dim=198):
        super().__init__()
        self.image_encoder = ResNet50Dilated(img_enc_dim)
        self.flow_encoder = ShallowNet(4, sparse_enc_dim)
        self.flow_decoder = MotionDecoderSkipLayer(img_enc_dim + sparse_enc_dim, output_dim)

    def forward(self, image, sparse):
        sparse_enc = self.flow_encoder(sparse)
        img_enc, skip = self.image_encoder(image)
        return self.flow_decoder(torch.cat((img_enc, sparse_enc), dim=1), skip)


def convert_flow(flow_prob, nbins=99, fmax=50):
    """Fuser.convert_flow (visualize_utils.py:6-19): expectation over nbins bin centres, per component."""
    step = 2 * fmax / float(nbins)
    mesh = torch.arange(nbins, device=flow_prob.device).view(1, -1, 1, 1).float() * step - fmax + step / 2
    px = torch.softmax(flow_prob[:, :nbins], dim=1) * mesh
    py = torch.softmax(flow_prob[:, nbins:], dim=1) * mesh
    return torch.cat([px.sum(1, keepdim=True), py.sum(1, keepdim=True)], dim=1)


def cmp_demo_run(model, image, sparse, mask):
    """CMP_demo.run (FCN.py:51-62): image in [0,1] -> *2-1; input = cat(sparse, mask); eval-mode BN; 192^2 logits ->
    expected flow -> bilinear(align_corners=True) back to the input size (no magnitude rescale, quirk Q15)."""
    dtype = image.dtype
    out = model((image * 2 - 1).float(), torch.cat([sparse, mask], dim=1).float())
    flow = convert_flow(out)
    if flow.shape[2] != image.shape[2]:
        flow = F.interpolate(flow, size=image.shape[2:4], mode="bilinear", align_corners=True)
    return flow.to(dtype)


def seeded_state_dict(model, seed=0):
    """Deterministic weights for any module with CMP-style key names (used for the reference-generated goldens of CMP
    and of the adapter encoders, and for the tests): N(0, 1/fan_in) convs, norm weight ~ U(0.3,0.7), bias/mean ~
    N(0,0.1), var ~ U(0.5,1.5)."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for k, v in sorted(model.state_dict().items()):
        if k.endswith("num_batches_tracked"):
            sd[k] = v.clone()
        elif k.endswith("running_var"):
            sd[k] = torch.rand(v.shape, generator=g) + 0.5
        elif k.endswith("weight") and v.ndim == 1:          # BN gamma: < 1 so 50 residual layers stay fp16-finite
            sd[k] = torch.rand(v.shape, generator=g) * 0.4 + 0.3
        elif v.ndim == 1:
            sd[k] = torch.randn(v.shape, generator=g) * 0.1
        else:
            fan_in = v[0].numel()
            sd[k] = torch.randn(v.shape, generator=g) * (1.0 / fan_in ** 0.5)
    return sd
