"""The consumer of the hot path: mirror of the reference's `models/resnet.py` (`class Model`, found by
`main_spectrogram.py` through `import_class('models.resnet.Model')`).

Reference forward (models/resnet.py:23-28): VirtualRadar -> unsqueeze(1) -> nearest interpolate to
image_size -> ResNet-18.  Here the first three steps are ONE fused launch (`VirtualRadar.forward_image`,
C ABI `vr_forward_image_f32`), optionally preceded by the data loader's temporal up-sampling on the device
(`num_pad_frames`, replaces `Dataset.pad_frames`, utils.py:134-140; fused too: `forward_upsampled`).  The classifier itself is not part of
the hot path: it is a plain PyTorch/cuDNN ResNet-18 with the reference's shape (1 input channel,
`num_filters` base width, models/resnet18.py:131-185), or any module passed as `base_model`.
"""
import torch
from torch import nn

from ..layers.virtual_radar import VirtualRadar


class BasicBlock(nn.Module):
    """Two 3x3 convolutions with an identity / 1x1-projection shortcut.  Sub-module names (`conv1`, `bn1`, `conv2`,
    `bn2`, `downsample.0/1`) are those of the reference's block (models/resnet18.py:36-76), so checkpoints interchange."""

    def __init__(self, cin, cout, stride):
        super().__init__()
        self.conv1 = nn.Conv2d(cin, cout, 3, stride, 1, bias=False)
        self.bn1 = nn.BatchNorm2d(cout)
        self.relu = nn.ReLU(inplace=True)
        self.conv2 = nn.Conv2d(cout, cout, 3, 1, 1, bias=False)
        self.bn2 = nn.BatchNorm2d(cout)
        self.downsample = None
        if stride != 1 or cin != cout:
            self.downsample = nn.Sequential(nn.Conv2d(cin, cout, 1, stride, bias=False), nn.BatchNorm2d(cout))

    def forward(self, x):
        y = self.bn2(self.conv2(self.relu(self.bn1(self.conv1(x)))))
        return self.relu(y + (x if self.downsample is None else self.downsample(x)))


class ResNet18(nn.Module):
    """ResNet-18 over single-channel images with the reference's layout and parameter names (models/resnet18.py:131-185,
    218-232: `conv1` 7x7/2 on 1 channel, `bn1`, 3x3/2 max-pool, `layer1..4` of two blocks with widths
    num_filters * (1, 2, 4, 8), global average pool, `fc`): `state_dict()` keys and shapes equal the reference's, so a
    checkpoint of the reference `Model` loads into `Model` here and vice versa (tests/test_feeder.py)."""

    def __init__(self, num_classes=60, num_filters=64):
        super().__init__()
        w = num_filters
        self.conv1 = nn.Conv2d(1, w, 7, 2, 3, bias=False)
        self.bn1 = nn.BatchNorm2d(w)
        self.relu = nn.ReLU(inplace=True)
        self.maxpool = nn.MaxPool2d(3, 2, 1)
        cin = w
        for i, cout in enumerate((w, 2 * w, 4 * w, 8 * w)):
            setattr(self, "layer%d" % (i + 1), nn.Sequential(BasicBlock(cin, cout, 1 if i == 0 else 2), BasicBlock(cout, cout, 1)))
            cin = cout
        self.avgpool = nn.AdaptiveAvgPool2d(1)
        self.fc = nn.Linear(cin, num_classes)
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")

    def forward(self, x):
        x = self.maxpool(self.relu(self.bn1(self.conv1(x))))
        x = self.layer4(self.layer3(self.layer2(self.layer1(x))))
        return self.fc(torch.flatten(self.avgpool(x), 1))


def resnet18(num_classes=60, num_filters=64):
    return ResNet18(num_classes, num_filters)


class Model(nn.Module):
    """Same constructor as the reference (`models/resnet.py:12-16`) plus two optional keywords:
    `base_model` (any classifier over (N,1,S,S) images; default: the ResNet-18 above) and
    `num_pad_frames` / `sigma` (up-sample raw sequences on the device before the radar; None = the
    input is already at the radar sampling rate, as in the reference)."""

    def __init__(self, num_classes=60, num_filters=64, image_size=256, device='cuda:0',
                 base_model=None, num_pad_frames=None, sigma=3):
        super().__init__()
        self.base_model = base_model if base_model is not None else resnet18(num_classes, num_filters)
        self.virtual_radar = VirtualRadar(wavelength=5e-4, device=device)
        self.image_size = image_size
        self.num_pad_frames = num_pad_frames
        self.sigma = sigma

    def spectrogram_image(self, x, radar_location=None, wavelength=None, noise_std=None, noise_seed=None):
        """radar_location / wavelength (optional): one radar placement per sequence; noise_std / noise_seed (optional):
        receiver noise (VirtualRadar.forward)."""
        kw = dict(radar_location=radar_location, wavelength=wavelength, noise_std=noise_std, noise_seed=noise_seed)
        if self.num_pad_frames:       # raw sequences: up-sampling, radar and resize in one fused pass
            return self.virtual_radar.forward_upsampled(x, self.num_pad_frames, self.sigma, self.image_size, **kw)
        return self.virtual_radar.forward_image(x, self.image_size, **kw)

    def forward(self, x, radar_location=None, wavelength=None, noise_std=None, noise_seed=None):
        return self.base_model(self.spectrogram_image(x, radar_location, wavelength, noise_std, noise_seed))
