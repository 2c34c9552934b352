"""Model / data selection shared by the two example drivers."""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
if PKG not in sys.path:
    sys.path.insert(0, PKG)          # the reference's scripts do sys.path.insert(0, '../')

MODELS = {
    # name: (builder, calibration input shape)
    "lenet": (lambda: __import__("model.lenet", fromlist=["Cnn"]).Cnn(1, 10), (1, 28, 28)),
    "resnet18_cifar": (lambda: __import__("model.resnet.resnet18_cifar_fabu", fromlist=["ResNet18"]).ResNet18(),
                       (3, 32, 32)),
    "resnet18": (lambda: __import__("model.resnet.resnet_fabu", fromlist=["resnet18_fabu"]).resnet18_fabu(),
                 (3, 224, 224)),
    "resnet50": (lambda: __import__("model.resnet.resnet_fabu", fromlist=["resnet50_fabu"]).resnet50_fabu(),
                 (3, 224, 224)),
    "resnet50d": (lambda: __import__("model.resnet.resnet_fabu", fromlist=["resnet50d_fabu"]).resnet50d_fabu(),
                  (3, 224, 224)),
    "resnext50_32x4d": (lambda: __import__("model.resnet.resnet_fabu",
                                           fromlist=["resnext50_32x4d_fabu"]).resnext50_32x4d_fabu(), (3, 224, 224)),
    "mobilenetv2": (lambda: __import__("model.mobilenet.mobilenetv2_fabu",
                                       fromlist=["mobilenetv2_fabu"]).mobilenetv2_fabu(), (3, 224, 224)),
    "fpn_r50": (lambda: __import__("model.fpn.fpn_fabu", fromlist=["fpn_r50_fabu"]).fpn_r50_fabu(), (3, 512, 512)),
}


def build(name, checkpoint=None, seed=0):
    """The architecture `name`, with `checkpoint` loaded (a state_dict saved by the reference's training scripts)
    or, without one, seeded default initialisation and randomised BatchNorm statistics (there is no network
    here to fetch trained weights)."""
    from model.resnet.resnet_fabu import randomize_bn_
    builder, shape = MODELS[name]
    torch.manual_seed(seed)
    net = builder().eval()
    if checkpoint:
        net.load_state_dict(torch.load(checkpoint, map_location="cpu"))
    else:
        with torch.no_grad():
            randomize_bn_(net, seed)
    return net, shape


def batches(shape, n_batches, batch, images_npy=None, labels_npy=None, seed=1):
    """(images, labels) tuples, the loader form PRE_PROCESS.IMG = 1 expects.  From .npy files when given,
    else synthetic (normal for the ResNets, which expect normalised images; uniform [0, 1) for LeNet)."""
    if images_npy:
        import numpy as np
        x = torch.from_numpy(np.load(images_npy)).float()
        y = torch.from_numpy(np.load(labels_npy)).long() if labels_npy else None
        return [(x[i:i + batch], None if y is None else y[i:i + batch])
                for i in range(0, min(len(x), n_batches * batch), batch)]
    out = []
    for i in range(n_batches):
        g = torch.Generator().manual_seed(seed + i)
        x = torch.rand(batch, *shape, generator=g) if shape[0] == 1 else torch.randn(batch, *shape, generator=g)
        out.append((x, None))
    return out


def configs(workdir, shape, n_batches):
    import tools._config as tc
    cfg = tc.load_tool_config(os.path.join(PKG, "tools", "configs.yml"))
    cfg["OUTPUT"] = {"WORK_DIR": workdir, "WEIGHT_BIT_TABLE": workdir + "/weight.table",
                     "FEAT_BIT_TABLE": workdir + "/feat.table", "WEIGHT_DIR": workdir + "/weight",
                     "BIAS_DIR": workdir + "/bias", "FINAL_WEIGHT_DIR": workdir + "/new_weight",
                     "FINAL_BIAS_DIR": workdir + "/new_bias"}
    cfg["SETTINGS"]["MAX_CALI_IMG_NUM"] = n_batches - 1
    user = tc.load_user_config({"PATH": {"QUANTITY_MODEL_PATH": workdir + "/quantity_model.pth"},
                                "MODEL": {"INPUT_SHAPE": ",".join(map(str, (1,) + tuple(shape)))},
                                "PRE_PROCESS": {"IMG": 1}, "SETTINGS": {"DEVICE": "gpu", "GPU": 0}})
    return cfg, user
