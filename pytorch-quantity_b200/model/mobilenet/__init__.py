from .mobilenetv2_fabu import mobilenetv2_fabu, MobileNetV2Fabu  # noqa: F401
