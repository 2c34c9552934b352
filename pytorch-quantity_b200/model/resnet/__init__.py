from .resnet_fabu import resnet18_fabu, resnet50_fabu, resnet50d_fabu, resnext50_32x4d_fabu, FabuResNet  # noqa: F401
