"""Random-init HigherHRNet in stock PyTorch -- ONLY a producer of synthetic network outputs.

BASELINE.json names its workloads "HigherHRNet-W32 / W48 ... random-init weights on synthetic images";
there is no checkpoint or dataset offline and the reference's model code does not exist on the GPU
box, so bench.py / smoke() build this network (default PyTorch init, eval mode) and run it on seeded
random images to get heatmap / tag tensors of the real shapes and statistics.  The convolutions are
out of scope of this library (north_star): everything here is plain torch.nn, nothing is optimised,
and the decode path never imports this module.

Architecture (HRNet, Sun et al. 2019; HigherHRNet, Cheng et al. 2020; interface of
/root/reference/src/keypoints/architectures/higher_hrnet.py:47-81): stem of two stride-2 3x3 convs,
one bottleneck stage, three multi-resolution stages (1 / 4 / 3 modules of 4 basic blocks per branch,
widths C, 2C, 4C, 8C) with full fusion, a 1x1 head giving 2K channels at 1/4 resolution (K heatmaps
+ K tags, returned as channel-slice VIEWS), and ``num_deconvs`` stride-2 transposed-conv modules with 4 basic blocks
each, every one giving K heatmaps at twice the resolution of the previous stage.  forward(x) -> ([hm_lo, hm_hi], tag)
for the default num_deconvs=1; ([hm], tag) for 0 (HRNet with the associative-embedding head); ([hm_lo, hm_hi, hm_full],
tag) for 2 (stages at S/4, S/2, S).
"""
import torch
from torch import nn


def _cbr(cin, cout, k=3, s=1, relu=True):
    layers = [nn.Conv2d(cin, cout, k, s, k // 2, bias=False), nn.BatchNorm2d(cout)]
    if relu:
        layers.append(nn.ReLU(inplace=True))
    return nn.Sequential(*layers)


class _Basic(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.a, self.b = _cbr(c, c), _cbr(c, c, relu=False)

    def forward(self, x):
        return torch.relu(self.b(self.a(x)) + x)


class _Bottleneck(nn.Module):
    def __init__(self, cin, mid):
        super().__init__()
        self.body = nn.Sequential(_cbr(cin, mid, 1), _cbr(mid, mid, 3), _cbr(mid, mid * 4, 1, relu=False))
        self.skip = None if cin == mid * 4 else _cbr(cin, mid * 4, 1, relu=False)

    def forward(self, x):
        return torch.relu(self.body(x) + (x if self.skip is None else self.skip(x)))


class _Module(nn.Module):
    """4 basic blocks per branch, then every output branch sums all (resampled) branches."""

    def __init__(self, widths, n_out=None):
        super().__init__()
        n = len(widths)
        self.n_out = n if n_out is None else n_out
        self.branches = nn.ModuleList([nn.Sequential(*[_Basic(w) for _ in range(4)]) for w in widths])
        fuse = []
        for i in range(self.n_out):
            row = []
            for j in range(n):
                if j == i:
                    row.append(nn.Identity())
                elif j > i:
                    row.append(nn.Sequential(_cbr(widths[j], widths[i], 1, relu=False),
                                             nn.Upsample(scale_factor=2 ** (j - i), mode="nearest")))
                else:
                    steps = [_cbr(widths[j], widths[j], 3, 2) for _ in range(i - j - 1)]
                    steps.append(_cbr(widths[j], widths[i], 3, 2, relu=False))
                    row.append(nn.Sequential(*steps))
            fuse.append(nn.ModuleList(row))
        self.fuse = nn.ModuleList(fuse)

    def forward(self, xs):
        ys = [b(x) for b, x in zip(self.branches, xs)]
        return [torch.relu(sum(f(y) for f, y in zip(row, ys))) for row in self.fuse]


class HigherHRNet(nn.Module):
    def __init__(self, num_kpts: int = 17, C: int = 32, num_deconvs: int = 1):
        super().__init__()
        if num_deconvs not in (0, 1, 2):
            raise ValueError(f"num_deconvs must be 0, 1 or 2 (got {num_deconvs})")
        self.num_kpts = num_kpts
        self.num_deconvs = num_deconvs
        self.stem = nn.Sequential(_cbr(3, 64, 3, 2), _cbr(64, 64, 3, 2))
        self.stage1 = nn.Sequential(_Bottleneck(64, 64), *[_Bottleneck(256, 64) for _ in range(3)])
        w = [C, 2 * C, 4 * C, 8 * C]
        self.trans = nn.ModuleList([
            nn.ModuleList([_cbr(256, w[0]), _cbr(256, w[1], 3, 2)]),
            _cbr(w[1], w[2], 3, 2),
            _cbr(w[2], w[3], 3, 2),
        ])
        self.stage2 = nn.ModuleList([_Module(w[:2])])
        self.stage3 = nn.ModuleList([_Module(w[:3]) for _ in range(4)])
        self.stage4 = nn.ModuleList([_Module(w[:4]) for _ in range(2)] + [_Module(w[:4], n_out=1)])
        self.head = nn.Conv2d(C, 2 * num_kpts, 1)
        self.deconv = nn.Sequential(nn.ConvTranspose2d(C + 2 * num_kpts, C, 4, 2, 1, bias=False), nn.BatchNorm2d(C),
                                    nn.ReLU(inplace=True))
        self.deconv_blocks = nn.Sequential(*[_Basic(C) for _ in range(4)])
        self.final = nn.Conv2d(C, num_kpts, 1)
        if num_deconvs == 2:   # the second module reads the first one's features and heatmaps
            self.deconv2 = nn.Sequential(nn.ConvTranspose2d(C + num_kpts, C, 4, 2, 1, bias=False), nn.BatchNorm2d(C),
                                         nn.ReLU(inplace=True))
            self.deconv2_blocks = nn.Sequential(*[_Basic(C) for _ in range(4)])
            self.final2 = nn.Conv2d(C, num_kpts, 1)

    def forward(self, x):
        x = self.stage1(self.stem(x))
        xs = [t(x) for t in self.trans[0]]
        for m in self.stage2:
            xs = m(xs)
        xs = xs + [self.trans[1](xs[-1])]
        for m in self.stage3:
            xs = m(xs)
        xs = xs + [self.trans[2](xs[-1])]
        for m in self.stage4:
            xs = m(xs)
        feats = xs[0]
        both = self.head(feats)                                   # [B, 2K, S/4, S/4]
        K = self.num_kpts
        if self.num_deconvs == 0:
            return [both[:, :K]], both[:, K:]
        f1 = self.deconv_blocks(self.deconv(torch.cat((feats, both), 1)))
        hm_hi = self.final(f1)
        if self.num_deconvs == 1:
            return [both[:, :K], hm_hi], both[:, K:]              # channel-slice views, like the reference
        hm_full = self.final2(self.deconv2_blocks(self.deconv2(torch.cat((f1, hm_hi), 1))))
        return [both[:, :K], hm_hi, hm_full], both[:, K:]


@torch.no_grad()
def network_outputs(batch: int, size: int = 512, flip: bool = True, seed: int = 0, C: int = 32, device="cuda:0",
                    chunk: int = 8, num_kpts: int = 17, image_seed=None, num_deconvs: int = 1):
    """One scale dict of CUDA tensors [B,K,h,w] produced by a default-init HigherHRNet-W{C} on seeded
    N(0,1) images (torch.manual_seed(seed) -> net -> images, the order SURVEY.md 8(d) fixes).
    ``image_seed`` (default seed + 1) seeds the images separately: several ranks then run ONE network
    (same ``seed``) on different images.  ``num_deconvs`` as in HigherHRNet: the default 1 gives the two-stage
    {hm_lo, hm_hi, tag[, hm_lo_f, hm_hi_f, tag_f]} dict, 0 and 2 the stage format {hm: [...], tag[, hm_f, tag_f]}."""
    torch.manual_seed(seed)
    net = HigherHRNet(num_kpts, C, num_deconvs).eval().to(device)
    g = torch.Generator(device="cpu").manual_seed(seed + 1 if image_seed is None else image_seed)
    n = max(num_deconvs, 0) + 1
    runs = ("", "_f") if flip else ("",)
    hms = {r: [[] for _ in range(n)] for r in runs}
    tags = {r: [] for r in runs}
    for b0 in range(0, batch, chunk):
        x = torch.randn(min(chunk, batch - b0), 3, size, size, generator=g).to(device)
        for r in runs:
            stages, tag = net(x if r == "" else torch.flip(x, [3]))
            for i, h in enumerate(stages):
                hms[r][i].append(h)
            tags[r].append(tag)
    # keep the first stage / tag as channel-slice views of one 2K-channel tensor per batch (strided, like the reference)
    out = {}
    for r in runs:
        both = torch.cat([torch.cat((a, t), 1) for a, t in zip(hms[r][0], tags[r])], 0)
        out["hm" + r] = [both[:, :num_kpts]] + [torch.cat(hs, 0) for hs in hms[r][1:]]
        out["tag" + r] = both[:, num_kpts:]
    if num_deconvs != 1:
        return out if flip else dict(out, hm_f=[], tag_f=None)
    res = {}
    for r in runs:
        res["hm_lo" + r], res["tag" + r], res["hm_hi" + r] = out["hm" + r][0], out["tag" + r], out["hm" + r][1]
    return res
