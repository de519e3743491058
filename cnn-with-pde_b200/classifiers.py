"""The classifiers the reference scripts wrap around their PDE layer, rebuilt on the B200 layers.

Only the PDE block is native code; everything after it is stock torch (dense layers, batch
norm, pooling: cuBLAS / ATen), exactly as in the reference.  The classes keep the reference's
attribute names so that a ``state_dict`` saved by a reference model loads here and vice versa
(tests/test_classifiers.py):

    mnist_test.PDEClassifier              mnist_test.py:223-237
    fashion_mnist.FashionPDEClassifier    fashion_mnist.py:200-224
    SVHN.PDEClassifier                    SVHN.py:234-270
    emotion_recognition.DiffusionClassifier   emotion_recognition.py:170-195
    cifar10.SpatialAttention / MultiScaleExtractor / EnhancedFC / CIFAR10PDENoConv   cifar10.py:215-361
    tiny_imagenet.BasicBlock / ImprovedTinyImageNetClassifier                       tiny_imagenet.py:237-327
    cifar_2version.SymmetricLayer / ParabolicBlock / HamiltonianBlock / HybridPDEExtractor /
        NonConvSpatialAttention / PDEClassifier / CIFAR10HybridPDEModel            cifar_2version.py:189-408

They are used by the data-parallel launcher (train.py); each is re-exported from the module
named after its script.
"""
from __future__ import annotations

import os

import torch
import torch.nn as nn
import torch.nn.functional as F

from .functional import _traced


# side streams of the branch-parallel extractors: per device, shared by all modules (kept out of the modules'
# __dict__ so that copy.deepcopy / pickling of a model that has already run keeps working)
_SIDE_STREAMS = {}


def _side_streams(device, n):
    pool = _SIDE_STREAMS.setdefault(device, [])
    while len(pool) < n:
        pool.append(torch.cuda.Stream(device=device))
    return pool[:n]


def _dense_stack(owner: nn.Module, widths, batch_norm: bool):
    """Register fc1..fcK (and bn1..bn{K-1}) on `owner` for the layer widths w0 -> w1 -> ... -> wK."""
    for k in range(1, len(widths)):
        setattr(owner, f"fc{k}", nn.Linear(widths[k - 1], widths[k]))
    if batch_norm:   # registered after the linears, as the reference does (parameter order matters to optimizers)
        for k in range(1, len(widths) - 1):
            setattr(owner, f"bn{k}", nn.BatchNorm1d(widths[k]))


class MnistPDEClassifier(nn.Module):
    """diff -> flatten -> dropout -> fc1 -> relu -> dropout -> fc2 (mnist_test.py:223-237)."""

    def __init__(self, dropout_rate=0.1, dx=1.0, dy=1.0):
        super().__init__()
        from .mnist_test import DiffusionLayer
        self.diff = DiffusionLayer(dx=dx, dy=dy)
        self.dropout = nn.Dropout(dropout_rate)
        _dense_stack(self, (28 * 28, 256, 10), batch_norm=False)

    def forward(self, x):
        h = self.diff(x).flatten(1)
        h = self.dropout(F.relu(self.fc1(self.dropout(h))))
        return self.fc2(h)


class FashionPDEClassifier(nn.Module):
    """diff -> 784-512-256-10 with batch norm (fashion_mnist.py:200-224)."""

    def __init__(self, dropout_rate=0.15):
        super().__init__()
        from .fashion_mnist import DiffusionLayer
        self.diff = DiffusionLayer()
        self.dropout = nn.Dropout(dropout_rate)
        _dense_stack(self, (28 * 28, 512, 256, 10), batch_norm=True)

    def forward(self, x):
        h = self.diff(x).flatten(1)
        h = self.dropout(F.relu(self.bn1(self.fc1(h))))
        h = self.dropout(F.relu(self.bn2(self.fc2(h))))
        return self.fc3(h)


class SvhnPDEClassifier(nn.Module):
    """diff(32, 3) -> 3072-2048-1024-512-256-10 with batch norm (SVHN.py:234-270).  The reference
    registers fc_k and bn_k interleaved; so does this class."""

    def __init__(self, dropout_rate=0.5):
        super().__init__()
        from .SVHN import DiffusionLayer
        self.diff = DiffusionLayer(size=32, channels=3)
        self.dropout = nn.Dropout(dropout_rate)
        widths = (32 * 32 * 3, 2048, 1024, 512, 256, 10)
        for k in range(1, len(widths)):
            setattr(self, f"fc{k}", nn.Linear(widths[k - 1], widths[k]))
            if k < len(widths) - 1:
                setattr(self, f"bn{k}", nn.BatchNorm1d(widths[k]))

    def forward(self, x):
        h = self.diff(x).flatten(1)
        for k in range(1, 5):
            h = self.dropout(F.relu(getattr(self, f"bn{k}")(getattr(self, f"fc{k}")(h))))
        return self.fc5(h)


class DiffusionClassifier(nn.Module):
    """pde -> Sequential(flatten, [linear, bn, relu, dropout] x 3, linear) (emotion_recognition.py:170-195)."""

    def __init__(self, img_size=48, num_classes=7, dropout_rate=0.3):
        super().__init__()
        from .emotion_recognition import PDELayer
        self.pde = PDELayer(Nx=img_size, Ny=img_size)
        mods = [nn.Flatten()]
        widths = (img_size * img_size, 512, 256, 128)
        for k in range(1, len(widths)):
            mods += [nn.Linear(widths[k - 1], widths[k]), nn.BatchNorm1d(widths[k]), nn.ReLU(), nn.Dropout(dropout_rate)]
        mods.append(nn.Linear(widths[-1], num_classes))
        self.classifier = nn.Sequential(*mods)

    def forward(self, x):
        return self.classifier(self.pde(x))


class SpatialAttention(nn.Module):
    """Channel gate from the spatial mean of (x + learned position embedding) (cifar10.py:215-244)."""

    def __init__(self, channels, size):
        super().__init__()
        self.channels = channels
        self.size = size
        self.pos_embed = nn.Parameter(torch.randn(1, channels, size, size) * 0.1)
        self.attention_fc = nn.Sequential(nn.Linear(channels, channels * 2), nn.ReLU(),
                                          nn.Linear(channels * 2, channels), nn.Sigmoid())

    def forward(self, x):
        gate = self.attention_fc((x + self.pos_embed).mean(dim=(2, 3)))
        return x * gate[:, :, None, None]


class MultiScaleExtractor(nn.Module):
    """Three PDE layers on the same input, each gated, softmax-combined (cifar10.py:248-282)."""

    def __init__(self, input_size=32, channels=3):
        super().__init__()
        from .cifar10 import EnhancedDiffusionLayer
        self.pde1 = EnhancedDiffusionLayer(input_size, channels, dt=0.001, num_steps=5, dx=1.0, dy=1.0)
        self.pde2 = EnhancedDiffusionLayer(input_size, channels, dt=0.002, num_steps=8, dx=2.0, dy=2.0)
        self.pde3 = EnhancedDiffusionLayer(input_size, channels, dt=0.005, num_steps=4, dx=1.5, dy=1.5)
        self.attention1 = SpatialAttention(channels, input_size)
        self.attention2 = SpatialAttention(channels, input_size)
        self.attention3 = SpatialAttention(channels, input_size)
        self.combine_weights = nn.Parameter(torch.ones(3) / 3)

    # The three branches read the same input and are independent until the combine (SURVEY section 8(f)
    # rank 1).  Two ways to exploit that, both built and parity-tested:
    #   concurrent_branches  each branch (PDE layer + its gate) on its own stream: fork / join around the
    #                        current stream, captured as parallel branches of a CUDA graph; a branch's gate and
    #                        its backward start as soon as that branch's PDE kernel is done;
    #   fused_branches       the three PDE layers through ONE launch per pass (blocks dealt to the layers in
    #                        proportion to their sweeps; cifar10.apply_to_same_input), gates on side streams.
    # Measured on one B200, batch 512, CUDA graph (DESIGN.md section 6): 1.18 - 1.20 ms per step with three
    # concurrent launches, 1.13 - 1.24 ms fused depending on the run -- one launch saves four launches but makes
    # every gate wait for the slowest layer and the PDE backward wait for all three gates.  No consistent winner,
    # so the streams stay the default and the fused call is opt-in (set fused_branches = True).
    fused_branches = False
    concurrent_branches = True

    def _side_streams(self, device):
        return _side_streams(device, 2)

    def forward(self, x):
        branches = ((self.pde1, self.attention1), (self.pde2, self.attention2), (self.pde3, self.attention3))
        # a traced call (torch.compile, torch.export, shape inference) takes the serial branch: the same values,
        # without side streams or an environment read
        serial = _traced(x) or bool(os.environ.get("PDE_B200_SERIAL_BRANCHES"))
        if x.is_cuda and self.fused_branches and not serial and torch.is_grad_enabled():
            from .cifar10 import apply_to_same_input
            ys = apply_to_same_input(x, [pde for pde, _ in branches])
            if self.concurrent_branches:
                # the gates (a dozen tiny kernels each, forward and backward) of branches 2 and 3 on side streams
                cur = torch.cuda.current_stream(x.device)
                sides = self._side_streams(x.device)
                feats = [None, None, None]
                for i, s in enumerate(sides, start=1):
                    s.wait_stream(cur)
                    ys[i].record_stream(s)
                    with torch.cuda.stream(s):
                        feats[i] = branches[i][1](ys[i])
                feats[0] = branches[0][1](ys[0])
                for i, s in enumerate(sides, start=1):
                    cur.wait_stream(s)
                    feats[i].record_stream(cur)
            else:
                feats = [att(y) for (_, att), y in zip(branches, ys)]
        elif x.is_cuda and self.concurrent_branches and not serial:
            cur = torch.cuda.current_stream(x.device)
            sides = self._side_streams(x.device)
            for s in sides:
                s.wait_stream(cur)          # fork: x is ready
            feats = [None, None, None]
            for i, (pde, att) in enumerate(branches[1:], start=1):
                with torch.cuda.stream(sides[i - 1]):
                    feats[i] = att(pde(x))
            feats[0] = branches[0][1](branches[0][0](x))
            for i, s in enumerate(sides, start=1):
                cur.wait_stream(s)          # join
                feats[i].record_stream(cur)
        else:
            feats = [att(pde(x)) for pde, att in branches]
        w = F.softmax(self.combine_weights, dim=0)
        combined = w[0] * feats[0] + w[1] * feats[1] + w[2] * feats[2]
        return (combined, *feats)


class EnhancedFC(nn.Module):
    """[linear, bn, relu, dropout] per hidden width, then a linear; Kaiming-normal weights (cifar10.py:286-314)."""

    def __init__(self, input_size, hidden_sizes, num_classes, dropout_rate=0.3):
        super().__init__()
        mods, prev = [], input_size
        for width in hidden_sizes:
            mods += [nn.Linear(prev, width), nn.BatchNorm1d(width), nn.ReLU(inplace=True), nn.Dropout(dropout_rate)]
            prev = width
        mods.append(nn.Linear(prev, num_classes))
        self.network = nn.Sequential(*mods)
        for m in self.modules():
            if isinstance(m, nn.Linear):
                nn.init.kaiming_normal_(m.weight)
                nn.init.constant_(m.bias, 0)

    def forward(self, x):
        return self.network(x)


class PlaneBatchNorm2d(nn.BatchNorm2d):
    """``nn.BatchNorm2d`` with the same parameters, buffers, ``state_dict`` and results.  In training
    mode on CUDA the batch statistics and the normalisation are ATen reductions / elementwise ops:
    cuDNN's spatial batch norm runs ONE block per channel, which for the 3-channel feature map of the
    CIFAR classifier (cifar10.py:329) means 3 blocks on 148 SMs -- 0.27 ms forward + 0.54 ms backward
    of a 1.9 ms training step at batch 512 (profiles/r01_launches_train_cifar10.csv)."""

    def forward(self, x):
        if not (self.training and x.is_cuda and self.affine and self.track_running_stats
                and self.momentum is not None and x.dim() == 4):
            return super().forward(x)
        n = x.numel() // x.shape[1]
        var, mean = torch.var_mean(x, dim=(0, 2, 3), unbiased=False)
        with torch.no_grad():
            self.num_batches_tracked.add_(1)
            self.running_mean.lerp_(mean, self.momentum)
            self.running_var.lerp_(var * (n / max(n - 1, 1)), self.momentum)
        inv = torch.rsqrt(var + self.eps)
        scale = self.weight * inv
        shift = self.bias - mean * scale
        return x * scale[None, :, None, None] + shift[None, :, None, None]


class CIFAR10PDENoConv(nn.Module):
    """Multi-scale PDE features -> BatchNorm2d -> 4x4 avg + max pooling -> EnhancedFC (cifar10.py:318-361)."""

    def __init__(self, dropout_rate=0.3):
        super().__init__()
        self.feature_extractor = MultiScaleExtractor(input_size=32, channels=3)
        self.adaptive_pool = nn.AdaptiveAvgPool2d((4, 4))
        self.max_pool = nn.AdaptiveMaxPool2d((4, 4))
        self.classifier = EnhancedFC(input_size=96, hidden_sizes=[512, 256, 128, 64], num_classes=10,
                                     dropout_rate=dropout_rate)
        self.feature_bn = PlaneBatchNorm2d(3)   # nn.BatchNorm2d(3) in the reference (cifar10.py:329)

    def forward(self, x):
        combined = self.feature_extractor(x)[0]
        f = self.feature_bn(combined)
        pooled = torch.cat([self.adaptive_pool(f), self.max_pool(f)], dim=1)
        return self.classifier(pooled.flatten(1))


# ------------------------------------------------------------------ cifar_2version.py:189-408
class SymmetricLayer(nn.Module):
    """F_sym(Y) = -K^T act(BN(K Y)) on the flattened feature map (cifar_2version.py:190-222); stock
    torch (two 3072 x 3072 GEMMs: cuBLAS)."""

    def __init__(self, channels, spatial_size, activation="relu"):
        super().__init__()
        self.channels = channels
        self.spatial_size = spatial_size
        self.feature_dim = channels * spatial_size * spatial_size
        self.K = nn.Linear(self.feature_dim, self.feature_dim, bias=False)
        self.norm = nn.BatchNorm1d(self.feature_dim)
        self.activation = nn.ReLU() if activation == "relu" else (nn.Tanh() if activation == "tanh" else nn.Identity())
        nn.init.eye_(self.K.weight)
        self.K.weight.data += torch.randn_like(self.K.weight) * 0.01

    def forward(self, Y):
        B, C, H, W = Y.shape
        s = self.activation(self.norm(self.K(Y.reshape(B, -1))))
        return (-torch.matmul(s, self.K.weight)).view(B, C, H, W)


class ParabolicBlock(nn.Module):
    """Y <- Y + dt F_sym(Y), num_steps times (cifar_2version.py:225-238)."""

    def __init__(self, channels, spatial_size, num_steps=3, dt=1.0):
        super().__init__()
        self.num_steps = num_steps
        self.dt = dt
        self.symmetric_layer = SymmetricLayer(channels, spatial_size)

    def forward(self, Y):
        for _ in range(self.num_steps):
            Y = Y + self.dt * self.symmetric_layer(Y)
        return Y


class HamiltonianBlock(nn.Module):
    """Symplectic pair Y <- Y - dt F_Y(Z); Z <- Z - dt F_Z(Y), Z0 = 0 (cifar_2version.py:241-258)."""

    def __init__(self, channels, spatial_size, num_steps=3, dt=1.0):
        super().__init__()
        self.num_steps = num_steps
        self.dt = dt
        self.F_Y = SymmetricLayer(channels, spatial_size)
        self.F_Z = SymmetricLayer(channels, spatial_size)

    def forward(self, Y):
        Z = torch.zeros_like(Y)
        for _ in range(self.num_steps):
            Y = Y + self.dt * (-self.F_Y(Z))
            Z = Z - self.dt * self.F_Z(Y)
        return Y


class HybridPDEExtractor(nn.Module):
    """Two learnable diffusion layers (the B200 kernels) + parabolic + Hamiltonian blocks on the same
    input, softmax-combined, BatchNorm2d (cifar_2version.py:261-307)."""

    concurrent_branches = True

    def __init__(self, input_size=32, channels=3):
        super().__init__()
        from .cifar_2version import LearnableDiffusionLayer
        self.diffusion1 = LearnableDiffusionLayer(input_size, channels, dt=0.001, num_steps=8)
        self.diffusion2 = LearnableDiffusionLayer(input_size, channels, dt=0.002, num_steps=5)
        self.parabolic = ParabolicBlock(channels, input_size, num_steps=4, dt=0.5)
        self.hamiltonian = HamiltonianBlock(channels, input_size, num_steps=3, dt=0.8)
        self.combination_weights = nn.Parameter(torch.ones(4) / 4)
        self.feature_norm = PlaneBatchNorm2d(channels)   # nn.BatchNorm2d in the reference (cifar_2version.py:276)

    fused_branches = False   # see MultiScaleExtractor

    def forward(self, x):
        serial = _traced(x) or bool(os.environ.get("PDE_B200_SERIAL_BRANCHES"))   # see MultiScaleExtractor
        if x.is_cuda and self.fused_branches and not serial and torch.is_grad_enabled():
            from .cifar10 import apply_to_same_input
            d1, d2 = apply_to_same_input(x, [self.diffusion1, self.diffusion2])   # one launch per pass for both
            par, ham = self.parabolic(x), self.hamiltonian(x)
        elif x.is_cuda and self.concurrent_branches and not serial:
            # the second diffusion layer on a side stream; the dense blocks keep the GPU busy on the main one
            cur = torch.cuda.current_stream(x.device)
            side = _side_streams(x.device, 1)[0]
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                d2 = self.diffusion2(x)
            d1 = self.diffusion1(x)
            par = self.parabolic(x)
            ham = self.hamiltonian(x)
            cur.wait_stream(side)
            d2.record_stream(cur)
        else:
            d1, d2 = self.diffusion1(x), self.diffusion2(x)
            par, ham = self.parabolic(x), self.hamiltonian(x)
        w = F.softmax(self.combination_weights, dim=0)
        combined = self.feature_norm(w[0] * d1 + w[1] * d2 + w[2] * par + w[3] * ham)
        return combined, d1, d2, par, ham


class NonConvSpatialAttention(nn.Module):
    """Per-pixel sigmoid gate from an MLP on (x + position embedding) (cifar_2version.py:310-333)."""

    def __init__(self, channels, spatial_size):
        super().__init__()
        self.channels = channels
        self.spatial_size = spatial_size
        self.feature_dim = channels * spatial_size * spatial_size
        self.pos_embed = nn.Parameter(torch.randn(1, channels, spatial_size, spatial_size) * 0.02)
        fd = self.feature_dim
        self.attention_net = nn.Sequential(nn.Linear(fd, fd // 4), nn.ReLU(), nn.Linear(fd // 4, fd // 8), nn.ReLU(),
                                           nn.Linear(fd // 8, fd), nn.Sigmoid())

    def forward(self, x):
        B, C, H, W = x.shape
        gate = self.attention_net((x + self.pos_embed).reshape(B, -1)).view(B, C, H, W)
        return x * gate


class HybridFC(nn.Module):
    """cifar_2version.PDEClassifier (cifar_2version.py:336-372): 1024-512-256-128 with batch norm,
    dropout p, p, p, p // 2 (sic), Kaiming-normal weights."""

    def __init__(self, input_dim, num_classes=10, dropout_rate=0.4):
        super().__init__()
        mods, prev = [], input_dim
        for width, p in ((1024, dropout_rate), (512, dropout_rate), (256, dropout_rate), (128, dropout_rate // 2)):
            mods += [nn.Linear(prev, width), nn.BatchNorm1d(width), nn.ReLU(inplace=True), nn.Dropout(p)]
            prev = width
        mods.append(nn.Linear(prev, num_classes))
        self.classifier = nn.Sequential(*mods)
        for m in self.modules():
            if isinstance(m, nn.Linear):
                nn.init.kaiming_normal_(m.weight)
                if m.bias is not None:
                    nn.init.constant_(m.bias, 0)

    def forward(self, x):
        return self.classifier(x)


class CIFAR10HybridPDEModel(nn.Module):
    """HybridPDEExtractor -> NonConvSpatialAttention -> BatchNorm2d -> 8x8 avg + max pooling ->
    PDEClassifier (cifar_2version.py:375-408)."""

    def __init__(self, dropout_rate=0.4):
        super().__init__()
        self.feature_extractor = HybridPDEExtractor(input_size=32, channels=3)
        self.attention = NonConvSpatialAttention(channels=3, spatial_size=32)
        self.adaptive_avg_pool = nn.AdaptiveAvgPool2d((8, 8))
        self.adaptive_max_pool = nn.AdaptiveMaxPool2d((8, 8))
        self.feature_bn = PlaneBatchNorm2d(3)   # nn.BatchNorm2d(3) in the reference (cifar_2version.py:392)
        self.classifier = HybridFC(input_dim=384, num_classes=10, dropout_rate=dropout_rate)

    def forward(self, x):
        combined = self.feature_extractor(x)[0]
        f = self.feature_bn(self.attention(combined))
        pooled = torch.cat([self.adaptive_avg_pool(f), self.adaptive_max_pool(f)], dim=1)
        return self.classifier(pooled.reshape(pooled.size(0), -1))


# ------------------------------------------------------------------ tiny_imagenet.py:237-327
class BasicBlock(nn.Module):
    """ResNet basic block (tiny_imagenet.py:306-327); stock torch (cuDNN convolutions)."""

    def __init__(self, in_planes, planes, stride=1):
        super().__init__()
        self.conv1 = nn.Conv2d(in_planes, planes, kernel_size=3, stride=stride, padding=1, bias=False)
        self.bn1 = nn.BatchNorm2d(planes)
        self.conv2 = nn.Conv2d(planes, planes, kernel_size=3, stride=1, padding=1, bias=False)
        self.bn2 = nn.BatchNorm2d(planes)
        self.shortcut = nn.Sequential()
        if stride != 1 or in_planes != planes:
            self.shortcut = nn.Sequential(nn.Conv2d(in_planes, planes, kernel_size=1, stride=stride, bias=False),
                                          nn.BatchNorm2d(planes))

    def forward(self, x):
        out = F.relu(self.bn1(self.conv1(x)))
        out = self.bn2(self.conv2(out))
        out = out + self.shortcut(x)
        return F.relu(out)


class ImprovedTinyImageNetClassifier(nn.Module):
    """diff (the B200 explicit layer, 3 x 64 x 64) -> ResNet-18-style backbone -> 200 classes
    (tiny_imagenet.py:237-303)."""

    def __init__(self, num_classes=200, use_pde=True, dropout_rate=0.3):
        super().__init__()
        self.use_pde = use_pde
        if use_pde:
            from .tiny_imagenet import ImprovedDiffusionLayer
            self.diff = ImprovedDiffusionLayer(size=64, channels=3, num_steps=1, use_implicit=False)
        self.conv1 = nn.Conv2d(3, 64, kernel_size=7, stride=2, padding=3, bias=False)
        self.bn1 = nn.BatchNorm2d(64)
        self.maxpool = nn.MaxPool2d(kernel_size=3, stride=2, padding=1)
        self.layer1 = self._make_layer(64, 64, 2, stride=1)
        self.layer2 = self._make_layer(64, 128, 2, stride=2)
        self.layer3 = self._make_layer(128, 256, 2, stride=2)
        self.layer4 = self._make_layer(256, 512, 2, stride=2)
        self.avgpool = nn.AdaptiveAvgPool2d((1, 1))
        self.dropout = nn.Dropout(dropout_rate)
        self.fc = nn.Linear(512, num_classes)
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
            elif isinstance(m, nn.BatchNorm2d):
                nn.init.constant_(m.weight, 1)
                nn.init.constant_(m.bias, 0)
            elif isinstance(m, nn.Linear):
                nn.init.normal_(m.weight, 0, 0.01)
                nn.init.constant_(m.bias, 0)

    @staticmethod
    def _make_layer(in_planes, planes, num_blocks, stride):
        return nn.Sequential(BasicBlock(in_planes, planes, stride), *[BasicBlock(planes, planes, 1) for _ in range(1, num_blocks)])

    def forward(self, x):
        if self.use_pde:
            x = self.diff(x)
        x = self.maxpool(F.relu(self.bn1(self.conv1(x))))
        x = self.layer4(self.layer3(self.layer2(self.layer1(x))))
        x = torch.flatten(self.avgpool(x), 1)
        return self.fc(self.dropout(x))
