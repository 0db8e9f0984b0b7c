"""Shared by make_golden_pseudogt.py (reference side) and tests/test_pseudo_gt_format.py (oracle / drop-in side)."""
import torch
import torch.nn as nn
import torch.nn.functional as F

RENDER, PSEUDO, PHOTO = 64, 16, 24        # render resolution, pseudo-GT (UV) resolution, photograph resolution


class TinyNet(nn.Module):
    """image [B,4,16,16] -> (texture [B,3,8,8] in [-1,1], displacement map [B,3,32,32])."""

    def __init__(self):
        super().__init__()
        self.t = nn.Conv2d(4, 3, 3, padding=1)
        self.m = nn.Conv2d(4, 3, 3, padding=1)

    def forward(self, x):
        tex = torch.tanh(F.avg_pool2d(self.t(x), 2))
        return tex, 0.05 * torch.tanh(F.interpolate(self.m(x), size=(32, 32), mode="bilinear", align_corners=False))


class Extractor(nn.Module):
    def forward(self, images):
        return [F.adaptive_avg_pool2d(images, 2).flatten(1).view(images.shape[0], -1, 1, 1)]


def build_net(seed=8):
    torch.manual_seed(seed)
    return TinyNet()


def record(make_record, seed=0, R=32):
    """One pseudo-GT record at texture resolution R from seeded inputs (make_record: data/pseudo_gt.py's)."""
    g = torch.Generator().manual_seed(seed)
    return make_record(torch.randn(3, 32, 32, generator=g) * 0.05, torch.rand(3, R, R, generator=g) * 2 - 1,
                       (torch.rand(1, R, R, generator=g) > 0.3).float(), torch.rand(4, 16, 16, generator=g) * 2 - 1)


def batches(n=2, B=2):
    g = torch.Generator().manual_seed(19)
    out = []
    for i in range(n):
        out.append((torch.rand(B, 4, 16, 16, generator=g) * 2 - 1, torch.rand(B, 3, 12, 12, generator=g) * 2 - 1,
                    torch.rand(B, 4, PHOTO, PHOTO, generator=g) * 2 - 1, 0.55 + 0.2 * torch.rand(B, 1, generator=g),
                    (torch.rand(B, 3, generator=g) - 0.5) * 0.2, F.normalize(torch.randn(B, 4, generator=g), dim=-1),
                    torch.tensor([[2 * i], [2 * i + 1 + 10 * (i % 2)]])))          # one mirrored index (>= dataset size 10)
    return out
