"""3-D ResNet family behind the reference's factory API (reference: pretorched/models/resnet3D.py).

The classes here are parameter containers: they create exactly the tensors of the reference's
``state_dict`` (same names, shapes, registration and RNG order, so a seeded random init is
bit-identical and zoo checkpoints load unchanged), while every ``forward`` body delegates to
``pretorched_x_b200.engine`` -- fused sm_100a kernels, fp16 NDHWC activations.

Drop-in surface kept (SURVEY.md section 8b): ``resnet3d10..200`` / ``resneti3d50`` factories with the
reference signatures, ``features / logits / forward``, a swappable ``last_linear`` (``fc`` is None as
after ``modify_resnets``, torchvision_models.py:443-481), ``pretrained_settings``.
"""
from collections import defaultdict

import torch
import torch.nn as nn

from .. import engine, ops
from ..ops import Act

__all__ = [
    'ResNet3D', 'resnet3d10', 'resnet3d18', 'resnet3d34',
    'resnet3d50', 'resnet3d101', 'resnet3d152', 'resnet3d200', 'resneti3d50',
]

_URL_ROOT = 'http://pretorched-x.csail.mit.edu/models/'
_CHECKPOINTS = {
    'kinetics-400': {
        'resnet3d18': 'resnet3d18_kinetics-e9f44270.pth',
        'resnet3d34': 'resnet3d34_kinetics-7fed38dd.pth',
        'resnet3d50': 'resnet3d50_kinetics-aad059c9.pth',
        'resnet3d101': 'resnet3d101_kinetics-8d4c9d63.pth',
        'resnet3d152': 'resnet3d152_kinetics-575c47e2.pth',
    },
    'moments': {'resnet3d50': 'resnet3d50_16seg_moments-6eb53860.pth'},
}
_NUM_CLASSES = {'kinetics-400': 400, 'moments': 339}


def _make_settings(names, checkpoints=_CHECKPOINTS):
    """Registry rows in the reference's schema (resnet3D.py:33-55)."""
    table = defaultdict(dict)
    for name in names:
        for dataset, files in checkpoints.items():
            fname = files.get(name)
            table[name][dataset] = {
                'input_space': 'RGB',
                'input_range': [0, 1],
                'url': (_URL_ROOT + fname) if fname else None,
                'std': [0.229, 0.224, 0.225],
                'mean': [0.485, 0.456, 0.406],
                'num_classes': _NUM_CLASSES[dataset],
                'input_size': [3, 224, 224],
            }
    return table


pretrained_settings = _make_settings([n for n in __all__ if n not in ('ResNet3D', 'resneti3d50')])


# ---------------------------------------------------------------------------------------------
# shared behaviour of every engine-backed module
# ---------------------------------------------------------------------------------------------
class EngineModule(engine.CacheOwner, nn.Module):
    """Accepts either an engine ``Act`` (inside a network) or a plain NCDHW tensor (standalone use, as the
    reference's blocks allow) and returns the same kind."""

    def _run(self, a):
        raise NotImplementedError

    def forward(self, x):
        if isinstance(x, Act):
            return self._run(x)
        return ops.to_ncdhw(self._run(ops.from_ncdhw(x, pitch=ops._round_up(x.shape[1], 8))))

    def backward(self, *a, **k):  # pragma: no cover - documentation of scope
        raise NotImplementedError("pretorched_x_b200 is a forward-pass engine")


class ShortcutA:
    """Parameter-free shortcut (resnet3D.py:65-74): stride-subsample, then zero-pad channels to ``planes``."""

    def __init__(self, planes, stride):
        self.planes, self.stride = planes, stride

    def __call__(self, x):
        if isinstance(x, Act):
            return ops.shortcut_a(x, self.stride, self.planes)
        return ops.to_ncdhw(ops.shortcut_a(ops.from_ncdhw(x, pitch=ops._round_up(x.shape[1], 8)), self.stride, self.planes))


def conv3x3x3(in_planes, out_planes, stride=1):
    return nn.Conv3d(in_planes, out_planes, kernel_size=3, stride=stride, padding=1, bias=False)


class BasicBlock(EngineModule):
    expansion = 1
    Conv3d = staticmethod(conv3x3x3)

    def __init__(self, inplanes, planes, stride=1, downsample=None):
        super().__init__()
        mk = self.Conv3d
        self.conv1, self.bn1 = mk(inplanes, planes, stride), nn.BatchNorm3d(planes)
        self.relu = nn.ReLU(inplace=True)
        self.conv2, self.bn2 = mk(planes, planes), nn.BatchNorm3d(planes)
        self.downsample = downsample
        self.stride = stride

    def _run(self, a):
        return engine.run_basic(self, a)


class Bottleneck(EngineModule):
    expansion = 4
    Conv3d = nn.Conv3d

    def __init__(self, inplanes, planes, stride=1, downsample=None):
        super().__init__()
        mk = self.Conv3d
        self.conv1, self.bn1 = mk(inplanes, planes, kernel_size=1, bias=False), nn.BatchNorm3d(planes)
        self.conv2 = mk(planes, planes, kernel_size=3, stride=stride, padding=1, bias=False)
        self.bn2 = nn.BatchNorm3d(planes)
        self.conv3, self.bn3 = mk(planes, planes * 4, kernel_size=1, bias=False), nn.BatchNorm3d(planes * 4)
        self.relu = nn.ReLU(inplace=True)
        self.downsample = downsample
        self.stride = stride

    def _run(self, a):
        return engine.run_bottleneck(self, a)


Bottleneck3D = Bottleneck   # the name BASELINE.json's north_star uses


class ResNet3D(engine.CacheOwner, nn.Module):
    """conv1(7x7x7, s(1,2,2)) - bn - relu - maxpool - layer1..4 - avgpool - last_linear."""

    Conv3d = nn.Conv3d
    head_name = 'last_linear'       # R2Plus1D keeps the reference's `fc`

    def __init__(self, block, layers, shortcut_type='B', num_classes=339):
        super().__init__()
        self.inplanes = 64
        self.conv1 = self.Conv3d(3, 64, kernel_size=7, stride=(1, 2, 2), padding=(3, 3, 3), bias=False)
        self.bn1 = nn.BatchNorm3d(64)
        self.relu = nn.ReLU(inplace=True)
        self.maxpool = nn.MaxPool3d(kernel_size=(3, 3, 3), stride=2, padding=1)
        for i, (planes, nblocks) in enumerate(zip((64, 128, 256, 512), layers)):
            setattr(self, 'layer%d' % (i + 1),
                    self._make_layer(block, planes, nblocks, shortcut_type, stride=1 if i == 0 else 2))
        self.avgpool = nn.AdaptiveAvgPool3d(1)
        setattr(self, self.head_name, nn.Linear(512 * block.expansion, num_classes))
        if self.head_name == 'last_linear':
            self.fc = None           # what modify_resnets leaves behind (torchvision_models.py:445-446)
        self.init_weights()
        self._register_load_state_dict_pre_hook(self._accept_zoo_head_keys)

    # -- construction (same tensor/RNG order as resnet3D.py:166-193) --------------------------------
    def _make_layer(self, block, planes, blocks, shortcut_type, stride=1):
        out_planes = planes * block.expansion
        downsample = None
        if stride != 1 or self.inplanes != out_planes:
            if shortcut_type == 'A':
                downsample = ShortcutA(out_planes, stride)
            else:
                downsample = nn.Sequential(
                    self.Conv3d(self.inplanes, out_planes, kernel_size=1, stride=stride, bias=False),
                    nn.BatchNorm3d(out_planes))
        seq = [block(self.inplanes, planes, stride, downsample)]
        self.inplanes = out_planes
        seq += [block(self.inplanes, planes) for _ in range(1, blocks)]
        return nn.Sequential(*seq)

    def init_weights(self):
        for m in self.modules():
            if isinstance(m, self.Conv3d):
                nn.init.kaiming_normal_(m.weight, mode='fan_out')
            elif isinstance(m, nn.BatchNorm3d):
                m.weight.data.fill_(1)
                m.bias.data.zero_()

    def _accept_zoo_head_keys(self, state_dict, prefix, *args):
        # zoo checkpoints were saved before modify_resnets renamed fc -> last_linear (resnet3D.py:276-277)
        other = 'fc' if self.head_name == 'last_linear' else 'last_linear'
        for leaf in ('weight', 'bias'):
            src, dst = '%s%s.%s' % (prefix, other, leaf), '%s%s.%s' % (prefix, self.head_name, leaf)
            if src in state_dict and dst not in state_dict:
                state_dict[dst] = state_dict.pop(src)

    # -- fine-tuning -----------------------------------------------------------------------------
    def enable_fine_tuning(self, ft_begin_index):
        """Give ``layer{ft_begin_index}..layer4`` a backward (opt-in; returns the model).  While grad mode is on, their blocks run
        through ``functions.TrainableBlockFunction``: conv weights and BatchNorm weight / bias receive ``.grad``, with the
        BatchNorm running statistics frozen (the model stays in ``eval()``; ``train()`` still refuses to run).  Earlier stages
        stay frozen.  5: head only (the default behaviour); ``None``: off.  Only ``resnet3d.BasicBlock`` / ``Bottleneck`` with
        plain ``nn.Conv3d`` convolutions have a backward; the stem (0) has none."""
        if ft_begin_index is None or ft_begin_index == 5:
            self._b2_ft_begin = None
            return self
        if ft_begin_index == 0:
            raise NotImplementedError("the stem (conv1 / bn1) has no backward: fine-tuning starts at layer1 or later")
        if ft_begin_index not in (1, 2, 3, 4):
            raise ValueError("ft_begin_index must be 0..5 or None, got %r" % (ft_begin_index,))
        for i in range(ft_begin_index, 5):
            for blk in getattr(self, "layer%d" % i):
                _check_trainable(blk, "layer%d" % i)
        self._b2_ft_begin = int(ft_begin_index)
        return self

    # -- reference API ------------------------------------------------------------------------
    def features_act(self, x):
        """Trunk on the engine's native layout (fp16 NDHWC ``Act``)."""
        if self.training:
            raise RuntimeError("the forward engine is inference-only: call model.eval() first")
        ft = self.__dict__.get("_b2_ft_begin")
        return engine.run_trunk(self, x, trainable_from=ft if torch.is_grad_enabled() else None)

    def features(self, input):
        return ops.to_ncdhw(self.features_act(input))

    def logits(self, features):
        a = features if isinstance(features, Act) else ops.from_ncdhw(features, pitch=ops._round_up(features.shape[1], 8))
        return engine.run_head(self, a, getattr(self, self.head_name))

    def forward(self, input):
        return self.logits(self.features_act(input))


def _check_trainable(blk, where):
    """Raise NotImplementedError unless ``blk`` is a block the fine-tuning backward covers (exact types: the R(2+1)D blocks
    subclass these)."""
    ok = type(blk) in (BasicBlock, Bottleneck) and getattr(blk, "nonlocalblock", None) is None
    convs = [blk.conv1, blk.conv2] + ([blk.conv3] if hasattr(blk, "conv3") else [])
    ds = blk.downsample
    if isinstance(ds, nn.Sequential):
        ok = ok and len(ds) == 2 and isinstance(ds[1], nn.BatchNorm3d)
        convs.append(ds[0])
    else:
        ok = ok and (ds is None or isinstance(ds, ShortcutA))
    ok = ok and all(type(c) is nn.Conv3d and c.bias is None and c.groups == 1 and tuple(c.dilation) == (1, 1, 1)
                    and len(set(c.stride)) == 1 for c in convs)
    if not ok:
        raise NotImplementedError("%s: %s blocks have no backward (fine-tuning covers resnet3d BasicBlock / Bottleneck with "
                                  "plain Conv3d convolutions)" % (where, type(blk).__name__))


def get_fine_tuning_parameters(model, ft_begin_index):
    """Optimizer parameter groups that train ``layer{ft_begin_index}..layer4`` and the head, with lr 0 for everything else
    (resnet3D.py:221-239).  ``ft_begin_index == 0``: ``model.parameters()``.  The head is matched by the model's
    ``head_name`` (``last_linear``, or ``fc``).  Changes no model state; pair it with ``model.enable_fine_tuning``."""
    if ft_begin_index == 0:
        return model.parameters()
    ft_module_names = ['layer{}'.format(i) for i in range(ft_begin_index, 5)]
    ft_module_names.append(getattr(model, 'head_name', 'fc'))
    parameters = []
    for k, v in model.named_parameters():
        if any(name in k for name in ft_module_names):
            parameters.append({'params': v})
        else:
            parameters.append({'params': v, 'lr': 0.0})
    return parameters


def _attach_settings(model, settings):
    for key in ('input_space', 'input_size', 'input_range', 'mean', 'std'):
        setattr(model, key, settings[key])
    return model


def load_pretrained(model, num_classes, settings):
    """torchvision_models.py:158-167: assert class count, fetch the checkpoint, attach preprocessing attrs."""
    assert num_classes == settings['num_classes'], \
        "num_classes should be {}, but is {}".format(settings['num_classes'], num_classes)
    import torch.utils.model_zoo as model_zoo
    model.load_state_dict(model_zoo.load_url(settings['url']))
    return _attach_settings(model, settings)


def inflate_pretrained(model, num_classes, settings):
    """torchvision_models.py:170-191: 2-D checkpoint tensors are repeated along T (no 1/T rescale)."""
    assert num_classes == settings['num_classes'], \
        "num_classes should be {}, but is {}".format(settings['num_classes'], num_classes)
    import torch.utils.model_zoo as model_zoo
    target = model.state_dict()
    weights = model_zoo.load_url(settings['url'])
    for key in list(weights):
        head_alias = key.replace('fc.', 'last_linear.') if key.startswith('fc.') else key
        ref = target.get(key, target.get(head_alias))
        if ref is not None and weights[key].shape != ref.shape:
            weights[key] = weights[key].unsqueeze(2).expand_as(ref)
    model.load_state_dict(weights)
    return _attach_settings(model, settings)


def _build(name, block, layers, num_classes, pretrained, **kwargs):
    model = ResNet3D(block, layers, num_classes=num_classes, **kwargs)
    if pretrained is not None:
        model = load_pretrained(model, num_classes, pretrained_settings[name][pretrained])
    return model


def resnet3d10(**kwargs):
    return ResNet3D(BasicBlock, [1, 1, 1, 1], **kwargs)


def resnet3d18(num_classes=400, pretrained='kinetics-400', shortcut_type='A', **kwargs):
    return _build('resnet3d18', BasicBlock, [2, 2, 2, 2], num_classes, pretrained, shortcut_type=shortcut_type, **kwargs)


def resnet3d34(num_classes=400, pretrained='kinetics-400', shortcut_type='A', **kwargs):
    return _build('resnet3d34', BasicBlock, [3, 4, 6, 3], num_classes, pretrained, shortcut_type=shortcut_type, **kwargs)


def resnet3d50(num_classes=400, pretrained='kinetics-400', **kwargs):
    return _build('resnet3d50', Bottleneck, [3, 4, 6, 3], num_classes, pretrained, **kwargs)


def resnet3d101(num_classes=400, pretrained='kinetics-400', **kwargs):
    return _build('resnet3d101', Bottleneck, [3, 4, 23, 3], num_classes, pretrained, **kwargs)


def resnet3d152(num_classes=400, pretrained='kinetics-400', **kwargs):
    return _build('resnet3d152', Bottleneck, [3, 8, 36, 3], num_classes, pretrained, **kwargs)


def resnet3d200(num_classes=400, pretrained='kinetics-400', **kwargs):
    # the reference ignores num_classes here (resnet3D.py:301-308): the net is built with the class default
    model = ResNet3D(Bottleneck, [3, 24, 36, 3], **kwargs)
    if pretrained is not None:
        model = load_pretrained(model, num_classes, pretrained_settings['resnet3d200'][pretrained])
    return model


def resneti3d50(num_classes=400, pretrained='moments', **kwargs):
    model = ResNet3D(Bottleneck, [3, 4, 6, 3], num_classes=num_classes, **kwargs)
    if pretrained is not None:
        from .resnet2d import pretrained_settings as settings2d
        model = inflate_pretrained(model, num_classes, settings2d['resnet50'][pretrained])
    return model
