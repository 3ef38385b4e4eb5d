from .activation import Sigmoid, Tanh, ReLU, LeakyReLU, Softmax, LogSoftmax  # noqa: F401
from .conv import Conv1d, Conv2d, ConvTranspose2d  # noqa: F401
from .pool import MaxPool1d, MaxPool2d, AvgPool1d, AvgPool2d  # noqa: F401
from .upsampling import Upsample  # noqa: F401
from .dropout import Dropout  # noqa: F401
from .batchnorm import BatchNorm2d  # noqa: F401
from .linear import Linear  # noqa: F401
from .loss import L1Loss, MSELoss, NLLLoss, BCELoss, CrossEntropyLoss  # noqa: F401
from .module import Module  # noqa: F401
from .container import Sequential, ModuleList, ModuleDict  # noqa: F401
