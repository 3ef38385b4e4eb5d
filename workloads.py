"""The benchmark / parity workloads: the models of the reference's training scripts, written once
against an abstract `df` namespace (anything with `.nn`, `.tensor`, `.Tensor`) so the *same* model
code builds on the reference package (oracle/make_golden.py, run in the build container) and on
deepflows_b200's host package (tests, bench.py).

  mlp_mnist       test/MLP_MNIST.py:72-83          784-100-20-10, ReLU
  cnn_mnist       test/CNN_MNIST_cuda.py:72-96     Conv(1,32,k5,p2)-ReLU-Pool, Conv(32,64,k5,p2)-ReLU-Pool, FC
  cnn_cifar10     test/CNN_CIFAR10_cuda.py:61-110  3 x (Conv-BN-ReLU-Pool), Dropout(.5), FC
  resnet_cifar    test/ResNet_CIFAR10_cuda.py:20-100  stem Conv3x3-BN-ReLU-MaxPool, 4 stages of basic
                  blocks (conv-bn-conv-bn + optional 1x1/s2 conv-bn shortcut, no ReLU inside the block),
                  mean(2), mean(2), FC
  dcgan_generator (new, no reference script)  Linear, 3 x (ConvTranspose2d-BN-ReLU), Upsample(x2, bilinear), Conv
  unet            (new, no reference script)  encoder levels of 2 x (Conv-BN-ReLU) with MaxPool between them, decoder
                  levels of ConvTranspose2d(k2, s2), cat with the skip, 2 x (Conv-BN-ReLU); 1x1 Conv head
"""
import types


def namespace(package):
    """df namespace from an imported DeepFlows package (reference or deepflows_b200's mirror)."""
    import importlib
    ns = types.SimpleNamespace()
    ns.nn = importlib.import_module(package.__name__ + ".nn")
    ns.tensor = importlib.import_module(package.__name__ + ".tensor")
    ns.Tensor = ns.tensor.Tensor
    ns.optim = importlib.import_module(package.__name__ + ".optim")
    ns.backend_api = package.backend_api
    return ns


def mlp_mnist(df, device, sizes=(784, 100, 20, 10)):
    nn = df.nn

    class MLP(nn.Module):
        def __init__(self):
            super().__init__()
            self.fc1 = nn.Linear(sizes[0], sizes[1], device=device)
            self.fc2 = nn.Linear(sizes[1], sizes[2], device=device)
            self.fc3 = nn.Linear(sizes[2], sizes[3], device=device)
            self.relu = nn.ReLU()

        def forward(self, x):
            return self.fc3(self.relu(self.fc2(self.relu(self.fc1(x)))))

    return MLP()


def cnn_mnist(df, device, widths=(32, 64), num_classes=10, in_hw=28):
    nn = df.nn

    class MNIST_CNN(nn.Module):
        def __init__(self):
            super().__init__()
            self.conv1 = nn.Conv2d(1, widths[0], kernel_size=5, padding=2, device=device)
            self.relu1 = nn.ReLU()
            self.pool1 = nn.MaxPool2d(kernel_size=2, stride=2)
            self.conv2 = nn.Conv2d(widths[0], widths[1], kernel_size=5, padding=2, device=device)
            self.relu2 = nn.ReLU()
            self.pool2 = nn.MaxPool2d(kernel_size=2, stride=2)
            self.fc = nn.Linear(widths[1] * (in_hw // 4) ** 2, num_classes, device=device)

        def forward(self, x):
            x = self.pool1(self.relu1(self.conv1(x)))
            x = self.pool2(self.relu2(self.conv2(x)))
            return self.fc(x.reshape(x.shape[0], -1))

    return MNIST_CNN()


def cnn_cifar10(df, device, widths=(32, 64, 128), num_classes=10, in_hw=32, dropout=0.5):
    nn = df.nn

    class CIFAR10_CNN(nn.Module):
        def __init__(self):
            super().__init__()
            self.conv1 = nn.Conv2d(3, widths[0], kernel_size=5, padding=2, device=device)
            self.bn1 = nn.BatchNorm2d(widths[0], device=device)
            self.relu1 = nn.ReLU()
            self.pool1 = nn.MaxPool2d(kernel_size=2, stride=2)
            self.conv2 = nn.Conv2d(widths[0], widths[1], kernel_size=5, padding=2, device=device)
            self.bn2 = nn.BatchNorm2d(widths[1], device=device)
            self.relu2 = nn.ReLU()
            self.pool2 = nn.MaxPool2d(kernel_size=2, stride=2)
            self.conv3 = nn.Conv2d(widths[1], widths[2], kernel_size=3, padding=1, device=device)
            self.bn3 = nn.BatchNorm2d(widths[2], device=device)
            self.relu3 = nn.ReLU()
            self.pool3 = nn.MaxPool2d(kernel_size=2, stride=2)
            self.drop = nn.Dropout(dropout)
            self.fc = nn.Linear(widths[2] * (in_hw // 8) ** 2, num_classes, device=device)

        def forward(self, x):
            x = self.pool1(self.relu1(self.bn1(self.conv1(x))))
            x = self.pool2(self.relu2(self.bn2(self.conv2(x))))
            x = self.pool3(self.relu3(self.bn3(self.conv3(x))))
            x = x.reshape(x.shape[0], -1)
            return self.fc(self.drop(x))

    return CIFAR10_CNN()


def resnet_cifar(df, device, widths=(32, 64, 128, 256), layers=(2, 2, 2, 2), num_classes=10, registered=True):
    """`registered=False` reproduces the script as written: blocks and shortcuts live in Python lists, so
    only conv1 / bn1 / fc are registered parameters (SURVEY Q5). `registered=True` additionally sets every
    block (and shortcut layer) as an attribute so that all of them train - the variant a user means."""
    nn, tensor = df.nn, df.tensor

    class ResidualBlock(nn.Module):
        def __init__(self, cin, cout, stride=1, downsample=None):
            super().__init__()
            self.conv1 = nn.Conv2d(cin, cout, kernel_size=3, stride=stride, padding=1, bias=False, device=device)
            self.bn1 = nn.BatchNorm2d(cout, device=device)
            self.conv2 = nn.Conv2d(cout, cout, kernel_size=3, stride=1, padding=1, bias=False, device=device)
            self.bn2 = nn.BatchNorm2d(cout, device=device)
            self.downsample = downsample
            if registered and downsample is not None:
                self.ds_conv, self.ds_bn = downsample

        def forward(self, x):
            identity = x
            out = self.bn2(self.conv2(self.bn1(self.conv1(x))))
            if self.downsample is not None:
                for layer in self.downsample:
                    identity = layer(identity)
            return out + identity

    class ResNet(nn.Module):
        def __init__(self):
            super().__init__()
            self.in_channels = widths[0]
            self.conv1 = nn.Conv2d(3, widths[0], kernel_size=3, stride=1, padding=1, bias=False, device=device)
            self.bn1 = nn.BatchNorm2d(widths[0], device=device)
            self.relu = nn.ReLU()
            self.pool1 = nn.MaxPool2d(kernel_size=2, stride=2)
            self.stages = []
            for si, (wd, nb) in enumerate(zip(widths, layers)):
                stage = self._make_layer(wd, nb, stride=1 if si == 0 else 2)
                self.stages.append(stage)
                if registered:
                    for bi, block in enumerate(stage):
                        setattr(self, "layer%d_%d" % (si + 1, bi), block)
            self.fc = nn.Linear(widths[-1], num_classes, device=device)

        def _make_layer(self, cout, blocks, stride):
            downsample = None
            if stride != 1 or self.in_channels != cout:
                downsample = [nn.Conv2d(self.in_channels, cout, kernel_size=1, stride=stride, bias=False, device=device),
                              nn.BatchNorm2d(cout, device=device)]
            out = [ResidualBlock(self.in_channels, cout, stride, downsample)]
            self.in_channels = cout
            for _ in range(1, blocks):
                out.append(ResidualBlock(cout, cout))
            return out

        def forward(self, x):
            x = self.pool1(self.relu(self.bn1(self.conv1(x))))
            for stage in self.stages:
                for block in stage:
                    x = block(x)
            x = tensor.mean(x, axis=2)
            x = tensor.mean(x, axis=2)
            return self.fc(x)

    return ResNet()


def all_parameters(model):
    """(name, tensor) for every parameter reachable from `model`, registered or not (for parity checks
    of the `registered=False` variant, where most weights never reach `named_parameters()`)."""
    seen, out = set(), []

    def visit(obj, prefix):
        if id(obj) in seen:
            return
        seen.add(id(obj))
        params = getattr(obj, "_parameters", None)
        if params is not None:
            for k, p in params.items():
                if p is not None:
                    out.append((prefix + k, p))
            for k, m in obj._modules.items():
                if m is not None:
                    visit(m, prefix + k + ".")
            for k, v in vars(obj).items():
                if isinstance(v, (list, tuple)):
                    for i, item in enumerate(v):
                        if isinstance(item, (list, tuple)):
                            for j, sub in enumerate(item):
                                if hasattr(sub, "_parameters"):
                                    visit(sub, "%s%s.%d.%d." % (prefix, k, i, j))
                        elif hasattr(item, "_parameters"):
                            visit(item, "%s%s.%d." % (prefix, k, i))

    visit(model, "")
    return out


def vgg16_bn(df, device, img=224, num_classes=10, widths=(64, 128, 256, 512, 512), fc=4096, dropout=0.5):
    """test/VGG.py:7-138: 13 bias-free 3x3 convs (2-2-3-3-3 per stage), each followed by BatchNorm and ReLU, a 2x2
    max-pool after every stage, then Linear(512 * (img/32)^2, 4096) - ReLU - Dropout - Linear(4096, 4096) - ReLU -
    Dropout - Linear(4096, classes)."""
    nn = df.nn
    depth = (2, 2, 3, 3, 3)

    class VGG16Model(nn.Module):
        def __init__(self):
            super().__init__()
            cin = 3
            self.plan = []
            for si, (wd, nconv) in enumerate(zip(widths, depth)):
                for ci in range(nconv):
                    cname, bname = "conv%d_%d" % (si + 1, ci + 1), "bn%d_%d" % (si + 1, ci + 1)
                    setattr(self, cname, nn.Conv2d(cin, wd, kernel_size=3, stride=1, padding=1, bias=False, device=device))
                    setattr(self, bname, nn.BatchNorm2d(wd, device=device))
                    self.plan.append((cname, bname))
                    cin = wd
                setattr(self, "pool%d" % (si + 1), nn.MaxPool2d(kernel_size=2, stride=2))
                self.plan.append(("pool%d" % (si + 1), None))
            side = img // 32
            self.fc1 = nn.Linear(widths[-1] * side * side, fc, device=device)
            self.fc2 = nn.Linear(fc, fc, device=device)
            self.fc3 = nn.Linear(fc, num_classes, device=device)
            self.relu = nn.ReLU()
            self.dropout = nn.Dropout(dropout)

        def forward(self, x):
            for a, b in self.plan:
                if b is None:
                    x = getattr(self, a)(x)
                else:
                    x = self.relu(getattr(self, b)(getattr(self, a)(x)))
            x = x.reshape(x.shape[0], -1)
            x = self.dropout(self.relu(self.fc1(x)))
            x = self.dropout(self.relu(self.fc2(x)))
            return self.fc3(x)

    return VGG16Model()


def resnet_imagenet(df, device, layers=(3, 4, 6, 3), widths=(64, 128, 256, 512), num_classes=10, registered=True):
    """test/ResNet.py:24-150 (the model `pretrained_models.py:455-460` falls back to for "ResNet-50": basic blocks,
    [3,4,6,3]): stem conv3x3(3->64, stride 1)-BN-ReLU with NO max-pool, basic blocks conv-bn-conv-bn (+ 1x1 conv-bn
    shortcut) + identity followed by ReLU, mean(2), mean(2), Linear(512, classes). As in the CIFAR script the blocks
    live in Python lists (SURVEY Q5); `registered=True` also sets them as attributes so that all of them train."""
    nn, tensor = df.nn, df.tensor

    class ResidualBlock(nn.Module):
        def __init__(self, cin, cout, stride=1, downsample=None):
            super().__init__()
            self.conv1 = nn.Conv2d(cin, cout, kernel_size=3, stride=stride, padding=1, bias=False, device=device)
            self.bn1 = nn.BatchNorm2d(cout, device=device)
            self.conv2 = nn.Conv2d(cout, cout, kernel_size=3, stride=1, padding=1, bias=False, device=device)
            self.bn2 = nn.BatchNorm2d(cout, device=device)
            self.downsample = downsample
            self.relu = nn.ReLU()
            if registered and downsample is not None:
                self.ds_conv, self.ds_bn = downsample

        def forward(self, x):
            identity = x
            out = self.bn2(self.conv2(self.bn1(self.conv1(x))))
            if self.downsample is not None:
                for layer in self.downsample:
                    identity = layer(identity)
            return self.relu(out + identity)

    class ResNet(nn.Module):
        def __init__(self):
            super().__init__()
            self.in_channels = widths[0]
            self.conv1 = nn.Conv2d(3, widths[0], kernel_size=3, stride=1, padding=1, bias=False, device=device)
            self.bn1 = nn.BatchNorm2d(widths[0], device=device)
            self.relu = nn.ReLU()
            self.stages = []
            for si, (wd, nb) in enumerate(zip(widths, layers)):
                stage = self._make_layer(wd, nb, stride=1 if si == 0 else 2)
                self.stages.append(stage)
                if registered:
                    for bi, block in enumerate(stage):
                        setattr(self, "layer%d_%d" % (si + 1, bi), block)
            self.fc = nn.Linear(widths[-1], num_classes, device=device)

        def _make_layer(self, cout, blocks, stride):
            downsample = None
            if stride != 1 or self.in_channels != cout:
                downsample = [nn.Conv2d(self.in_channels, cout, kernel_size=1, stride=stride, bias=False, device=device),
                              nn.BatchNorm2d(cout, device=device)]
            out = [ResidualBlock(self.in_channels, cout, stride, downsample)]
            self.in_channels = cout
            for _ in range(1, blocks):
                out.append(ResidualBlock(cout, cout))
            return out

        def forward(self, x):
            x = self.relu(self.bn1(self.conv1(x)))
            for stage in self.stages:
                for block in stage:
                    x = block(x)
            x = tensor.mean(x, axis=2)
            x = tensor.mean(x, axis=2)
            return self.fc(x)

    return ResNet()


def dcgan_generator(df, device, nz=64, widths=(256, 128, 64, 32), channels=3):
    """A small DCGAN-style generator (a decoder: every layer makes the image larger): z (N, nz) -> Linear -> reshape to
    (N, widths[0], 4, 4) -> 3 x [ConvTranspose2d(k4, s2, p1) -> BatchNorm2d -> ReLU] (4 -> 8 -> 16 -> 32 px) ->
    Upsample(x2, bilinear) -> Conv2d(k3, p1) to `channels` -> (N, channels, 64, 64)."""
    nn = df.nn

    class Generator(nn.Module):
        def __init__(self):
            super().__init__()
            self.fc = nn.Linear(nz, widths[0] * 16, device=device)
            self.ups = []
            for i, (cin, cout) in enumerate(zip(widths[:-1], widths[1:])):
                up = (nn.ConvTranspose2d(cin, cout, kernel_size=4, padding=1, stride=2, bias=False, device=device),
                      nn.BatchNorm2d(cout, device=device))
                setattr(self, "up%d" % (i + 1), up[0])
                setattr(self, "bn%d" % (i + 1), up[1])
                self.ups.append(up)
            self.relu = nn.ReLU()
            self.upsample = nn.Upsample(scale_factor=2, mode="bilinear")
            self.out = nn.Conv2d(widths[-1], channels, kernel_size=3, padding=1, device=device)

        def forward(self, z):
            x = self.fc(z).reshape(z.shape[0], widths[0], 4, 4)
            for conv, bn in self.ups:
                x = self.relu(bn(conv(x)))
            return self.out(self.upsample(x))

    return Generator()


def unet(df, device, in_channels=3, out_channels=3, widths=(32, 64, 128, 256)):
    """A U-Net (encoder-decoder with skip connections): len(widths) levels. Each encoder level is
    [Conv3x3(p1, bias-free) -> BatchNorm2d -> ReLU] x 2, with MaxPool2d(2) between levels. Each decoder level is
    ConvTranspose2d(k2, s2, bias-free) from widths[i+1] to widths[i], `cat([up, skip], dim=1)` with the encoder output of the
    same level, then [Conv3x3 -> BN -> ReLU] x 2 from 2 * widths[i] to widths[i]. A 1x1 Conv2d maps to `out_channels`.
    H and W must be divisible by 2 ** (len(widths) - 1); the output has the input's size."""
    nn, tensor = df.nn, df.tensor

    class DoubleConv(nn.Module):
        def __init__(self, cin, cout):
            super().__init__()
            self.conv1 = nn.Conv2d(cin, cout, kernel_size=3, padding=1, bias=False, device=device)
            self.bn1 = nn.BatchNorm2d(cout, device=device)
            self.conv2 = nn.Conv2d(cout, cout, kernel_size=3, padding=1, bias=False, device=device)
            self.bn2 = nn.BatchNorm2d(cout, device=device)
            self.relu = nn.ReLU()

        def forward(self, x):
            return self.relu(self.bn2(self.conv2(self.relu(self.bn1(self.conv1(x))))))

    class UNet(nn.Module):
        def __init__(self):
            super().__init__()
            self.down = []
            for i, (cin, cout) in enumerate(zip((in_channels,) + tuple(widths[:-1]), widths)):
                self.down.append(DoubleConv(cin, cout))
                setattr(self, "down%d" % i, self.down[-1])
            self.pool = nn.MaxPool2d(kernel_size=2, stride=2)
            self.up = []
            for i in reversed(range(len(widths) - 1)):
                up = (nn.ConvTranspose2d(widths[i + 1], widths[i], kernel_size=2, stride=2, bias=False, device=device),
                      DoubleConv(2 * widths[i], widths[i]))
                setattr(self, "up%d" % i, up[0])
                setattr(self, "dec%d" % i, up[1])
                self.up.append(up)
            self.head = nn.Conv2d(widths[0], out_channels, kernel_size=1, device=device)

        def forward(self, x):
            levels = len(widths)
            if x.shape[2] % 2 ** (levels - 1) or x.shape[3] % 2 ** (levels - 1):
                raise ValueError("unet: H and W (%d, %d) must be divisible by %d" % (x.shape[2], x.shape[3], 2 ** (levels - 1)))
            skips = []
            for i, block in enumerate(self.down):
                x = block(x if i == 0 else self.pool(x))
                skips.append(x)
            x = skips.pop()
            for upconv, block in self.up:
                x = block(tensor.cat([upconv(x), skips.pop()], dim=1))
            return self.head(x)

    return UNet()
