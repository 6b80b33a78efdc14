"""CPU restatement of the reference's hot-path forward passes -- TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference`` legs may
import this package.  The product path (``pretorched_x_b200``) never does.

Every function restates, in plain functional PyTorch on CPU fp32 tensors, what one reference ``forward`` body
computes from a ``state_dict`` (citations: file:line under /root/reference).  The reference's arithmetic itself
lives in third-party torch (unpinned in requirements.txt:1; installed here: 2.11.0+cu128, oneDNN CPU backend),
which is why the restatement also calls torch.nn.functional: it is the same library the reference calls, minus
the reference's nn.Module graph.

Pinning: the reference ships no golden vectors and no tests for this path (SURVEY.md section 4), so the oracle is
pinned against *outputs of the reference itself run in the build container*: ``oracle/make_golden.py`` imports
the unmodified reference from /root/reference, checks these functions against it bit-for-bit on seeded inputs,
and stores the reference's outputs under ``tests/golden/``.  ``tests/test_oracle_golden.py`` re-checks the
restatement against those fixtures wherever the test-suite runs.
"""
import hashlib
import itertools

import numpy as np
import torch
import torch.nn.functional as F

BN_EPS = 1e-5  # nn.BatchNorm3d default, used by every BN on the path (resnet3D.py:84)


# ---------------------------------------------------------------------------------------------
# architecture table (what the reference's factories instantiate)
# ---------------------------------------------------------------------------------------------
ARCHS = {
    # resnet3D.py:242-308
    'resnet3d10': dict(family='resnet3d', block='basic', layers=[1, 1, 1, 1], shortcut='B'),
    'resnet3d18': dict(family='resnet3d', block='basic', layers=[2, 2, 2, 2], shortcut='A'),
    'resnet3d34': dict(family='resnet3d', block='basic', layers=[3, 4, 6, 3], shortcut='A'),
    'resnet3d50': dict(family='resnet3d', block='bottleneck', layers=[3, 4, 6, 3], shortcut='B'),
    'resnet3d101': dict(family='resnet3d', block='bottleneck', layers=[3, 4, 23, 3], shortcut='B'),
    # r2plus1d.py:113-152
    'r2plus1d10': dict(family='r2plus1d', block='basic', layers=[1, 1, 1, 1], shortcut='B'),
    'r2plus1d18': dict(family='r2plus1d', block='basic', layers=[2, 2, 2, 2], shortcut='B'),
    'r2plus1d34': dict(family='r2plus1d', block='basic', layers=[3, 4, 6, 3], shortcut='B'),
    'r2plus1d50': dict(family='r2plus1d', block='bottleneck', layers=[3, 4, 6, 3], shortcut='B'),
    # nonlocalnet.py:553-570 (5 non-local blocks: nonlocal_blocks=[0,2,3,0], shortcut A)
    'nonlocalresnet3d50': dict(family='nonlocal', block='bottleneck', layers=[3, 4, 6, 3], shortcut='A',
                               nonlocal_blocks=[0, 2, 3, 0]),
    # torchvision_models.py:484-492 (torchvision BasicBlock body)
    'resnet18': dict(family='resnet2d', block='basic', layers=[2, 2, 2, 2], shortcut='B'),
    # torchvision Bottleneck body (stride on the 3x3 conv, v1.5) behind `resnet50` torchvision_models.py:494-532: the TRN backbone
    'resnet50': dict(family='resnet2d', block='bottleneck', layers=[3, 4, 6, 3], shortcut='B'),
    # pre_act_resnet3D.py:100-139 (ResNet3D subclass: default shortcut 'B', head `fc`)
    'preact_resnet3d18': dict(family='resnet3d', block='preact_basic', layers=[2, 2, 2, 2], shortcut='B'),
    'preact_resnet3d50': dict(family='resnet3d', block='preact_bottleneck', layers=[3, 4, 6, 3], shortcut='B'),
    # resnext3D.py:224-252 (ResNeXtBottleneck: grouped 3x3x3 conv, expansion 2, planes 128..1024, head `fc`)
    'resnext3d50': dict(family='resnext3d', block='resnext', layers=[3, 4, 6, 3], shortcut='B', cardinality=32),
    'resnext3d101': dict(family='resnext3d', block='resnext', layers=[3, 4, 23, 3], shortcut='B', cardinality=32),
}


def arch_spec(arch, kwargs=None):
    """Architecture row for a factory call: ``shortcut_type=`` in the factory kwargs overrides the table's default."""
    spec = ARCHS[arch]
    st = (kwargs or {}).get('shortcut_type')
    return dict(spec, shortcut=st) if st and st != spec['shortcut'] else spec


def build_package_model(pkg, fx):
    """The package-under-test's model for a ``kind == 'model'`` fixture: same factory call, seeds and BN / non-local
    conditioning as oracle/make_golden.py applied to the reference."""
    torch.manual_seed(fx["seeds"]["init"])
    arch = fx["arch"]
    if arch.startswith(("r2plus1d", "preact_")):             # plain **kwargs factories upstream (no `pretrained`)
        m = getattr(pkg, arch)(**fx["kwargs"])
    else:
        m = getattr(pkg, arch)(pretrained=None, **fx["kwargs"])
    randomize_bn_(m, fx["seeds"]["bn"])
    if fx.get("nl_factors"):
        apply_nonlocal_factors_(m, fx["nl_factors"])
    return m.eval()


def nonlocal_positions(layers, nonlocal_blocks):
    """Blocks that carry a non-local block: i % (blocks // n) == 0 (nonlocalnet.py:474-479)."""
    out = []
    for li, (nb, nn_) in enumerate(zip(layers, nonlocal_blocks)):
        freq = nb // nn_ if nn_ != 0 else -1
        out.append([i for i in range(nb) if freq > 0 and i % freq == 0])
    return out


# ---------------------------------------------------------------------------------------------
# primitives
# ---------------------------------------------------------------------------------------------
def _bn(x, sd, p):
    """Eval-mode BatchNorm: (x - mean) / sqrt(var + eps) * gamma + beta."""
    return F.batch_norm(x, sd[p + '.running_mean'], sd[p + '.running_var'], sd[p + '.weight'], sd[p + '.bias'],
                        False, 0.0, BN_EPS)


def _conv(x, sd, p, stride=1, padding=0):
    w = sd[p + '.weight']
    fn = F.conv2d if w.dim() == 4 else F.conv3d
    return fn(x, w, sd.get(p + '.bias'), stride, padding)


def spatio_temporal_conv(x, sd, p, kernel, stride, padding):
    """SpatioTemporalConv.forward (r2plus1d.py:85-88): (1,k,k) conv -> BN -> ReLU -> (k,1,1) conv."""
    kt, kh, kw = kernel
    st, sh, sw = stride
    pt, ph, pw = padding
    x = _conv(x, sd, p + '.spatial_conv', (1, sh, sw), (0, ph, pw))
    x = F.relu(_bn(x, sd, p + '.bn'))
    return _conv(x, sd, p + '.temporal_conv', (st, 1, 1), (pt, 0, 0))


def _block_conv(x, sd, p, family, k, stride, padding):
    """A block-level "Conv3d": plain nn.Conv3d, or SpatioTemporalConv for R(2+1)D (r2plus1d.py:91-96)."""
    if family == 'r2plus1d':
        return spatio_temporal_conv(x, sd, p, (k, k, k), (stride,) * 3, (padding,) * 3)
    return _conv(x, sd, p, stride, padding)


def shortcut_a(x, planes, stride):
    """downsample_basic_block (resnet3D.py:65-74 / nonlocalnet.py:322-332)."""
    out = F.avg_pool3d(x, kernel_size=1, stride=stride)
    pad = torch.zeros(out.size(0), planes - out.size(1), out.size(2), out.size(3), out.size(4), dtype=out.dtype)
    return torch.cat([out, pad], dim=1)


def _residual(x, sd, p, family, shortcut, planes_out, stride, has_downsample):
    if not has_downsample:
        return x
    if shortcut == 'A':
        return shortcut_a(x, planes_out, stride)
    # type B: 1x1x1 conv (stride s) + BN (resnet3D.py:176-185)
    y = _block_conv(x, sd, p + '.downsample.0', family, 1, stride, 0)
    return _bn(y, sd, p + '.downsample.1')


def basic_block(x, sd, p, family, shortcut, planes, stride, has_downsample):
    """BasicBlock.forward (resnet3D.py:91-106; torchvision resnet.py BasicBlock for the 2-D net)."""
    out = F.relu(_bn(_block_conv(x, sd, p + '.conv1', family, 3, stride, 1), sd, p + '.bn1'))
    out = _bn(_block_conv(out, sd, p + '.conv2', family, 3, 1, 1), sd, p + '.bn2')
    out = out + _residual(x, sd, p, family, shortcut, planes, stride, has_downsample)
    return F.relu(out)


def bottleneck(x, sd, p, family, shortcut, planes, stride, has_downsample):
    """Bottleneck.forward (resnet3D.py:125-143)."""
    out = F.relu(_bn(_block_conv(x, sd, p + '.conv1', family, 1, 1, 0), sd, p + '.bn1'))
    out = F.relu(_bn(_block_conv(out, sd, p + '.conv2', family, 3, stride, 1), sd, p + '.bn2'))
    out = _bn(_block_conv(out, sd, p + '.conv3', family, 1, 1, 0), sd, p + '.bn3')
    out = out + _residual(x, sd, p, family, shortcut, planes * 4, stride, has_downsample)
    return F.relu(out)


def preact_basic_block(x, sd, p, family, shortcut, planes, stride, has_downsample):
    """PreActivationBasicBlock.forward (pre_act_resnet3D.py:41-57): BN-ReLU-conv twice, + shortcut(x), no final ReLU."""
    out = _conv(F.relu(_bn(x, sd, p + '.bn1')), sd, p + '.conv1', stride, 1)
    out = _conv(F.relu(_bn(out, sd, p + '.bn2')), sd, p + '.conv2', 1, 1)
    return out + _residual(x, sd, p, family, shortcut, planes, stride, has_downsample)


def preact_bottleneck(x, sd, p, family, shortcut, planes, stride, has_downsample):
    """PreActivationBottleneck.forward (pre_act_resnet3D.py:76-96)."""
    out = _conv(F.relu(_bn(x, sd, p + '.bn1')), sd, p + '.conv1')
    out = _conv(F.relu(_bn(out, sd, p + '.bn2')), sd, p + '.conv2', stride, 1)
    out = _conv(F.relu(_bn(out, sd, p + '.bn3')), sd, p + '.conv3')
    return out + _residual(x, sd, p, family, shortcut, planes * 4, stride, has_downsample)


def resnext_bottleneck(x, sd, p, shortcut, planes, cardinality, stride, has_downsample):
    """ResNeXtBottleneck.forward (resnext3D.py:101-122): 1x1x1 -> grouped 3x3x3 (groups = cardinality, stride s) -> 1x1x1
    to planes * 2, BN after each, residual (type A / B as in resnet3D), ReLU."""
    out = F.relu(_bn(_conv(x, sd, p + '.conv1'), sd, p + '.bn1'))
    out = F.conv3d(out, sd[p + '.conv2.weight'], None, stride, 1, 1, cardinality)
    out = F.relu(_bn(out, sd, p + '.bn2'))
    out = _bn(_conv(out, sd, p + '.conv3'), sd, p + '.bn3')
    out = out + _residual(x, sd, p, 'resnext3d', shortcut, planes * 2, stride, has_downsample)
    return F.relu(out)


def nonlocal_block(x, sd, p):
    """_NonLocalBlockND._embedded_gaussian (nonlocalnet.py:143-166), 3-D, no sub-sampling."""
    b, c = x.shape[0], x.shape[1]
    d = sd[p + '.g.weight'].shape[0]
    g_x = _conv(x, sd, p + '.g').view(b, d, -1).permute(0, 2, 1)
    theta_x = _conv(x, sd, p + '.theta').view(b, d, -1).permute(0, 2, 1)
    phi_x = _conv(x, sd, p + '.phi').view(b, d, -1)
    f = torch.matmul(theta_x, phi_x)                 # unscaled logits
    f_div_c = F.softmax(f, dim=-1)                   # over keys
    y = torch.matmul(f_div_c, g_x).permute(0, 2, 1).contiguous().view(b, d, *x.shape[2:])
    w_y = _bn(_conv(y, sd, p + '.W.0'), sd, p + '.W.1')
    return w_y + x


def nonlocal_block_nd(x, sd, p, dimension, mode, sub_sample, bn_layer=True):
    """_NonLocalBlockND.forward for the softmax / dot-product / concatenation modes (nonlocalnet.py:143-243), any of 1/2/3
    position axes, with optional max-pooled phi / g (:126-131).  ``p`` is the key prefix ('' for a bare block)."""
    key = (lambda k: p + '.' + k) if p else (lambda k: k)
    conv = (None, F.conv1d, F.conv2d, F.conv3d)[dimension]
    pool = (None, F.max_pool1d, F.max_pool2d, F.max_pool3d)[dimension]
    cw = lambda name: conv(x, sd[key(name + '.weight')], sd[key(name + '.bias')])
    b = x.size(0)
    gk, pk = ('g.0', 'phi.0') if sub_sample else ('g', 'phi')
    g_x = cw(gk)
    if sub_sample:
        g_x = pool(g_x, 2)
    d = g_x.shape[1]
    g_x = g_x.reshape(b, d, -1).permute(0, 2, 1)
    if mode == 'gaussian':
        theta_x = x.reshape(b, x.shape[1], -1).permute(0, 2, 1)
        phi_x = (pool(x, 2) if sub_sample else x).reshape(b, x.shape[1], -1)
    else:
        theta_x = cw('theta').reshape(b, d, -1).permute(0, 2, 1)
        phi_x = cw(pk)
        if sub_sample:
            phi_x = pool(phi_x, 2)
        phi_x = phi_x.reshape(b, d, -1)
    if mode == 'concatenation':
        # _concatenation (nonlocalnet.py:213-243): [theta_i ; phi_j] on an N x N grid -> bias-free 1x1 Conv2d to one
        # channel -> ReLU -> / N.  Same tensor ops as the reference (repeat + cat + conv2d) so the result is bit-identical.
        th = cw('theta').reshape(b, d, -1, 1)
        ph = phi_x.reshape(b, d, 1, -1)
        h, w = th.size(2), ph.size(3)
        feat = torch.cat([th.repeat(1, 1, 1, w), ph.repeat(1, 1, h, 1)], dim=1)
        f = F.relu(F.conv2d(feat, sd[key('concat_project.0.weight')])).view(b, h, w)
        f_div_c = f / f.size(-1)
    else:
        f = torch.matmul(theta_x, phi_x)
        f_div_c = f / f.size(-1) if mode == 'dot_product' else F.softmax(f, dim=-1)
    y = torch.matmul(f_div_c, g_x).permute(0, 2, 1).contiguous().view(b, d, *x.shape[2:])
    if bn_layer:
        w_y = conv(y, sd[key('W.0.weight')], sd[key('W.0.bias')])
        w_y = F.batch_norm(w_y, sd[key('W.1.running_mean')], sd[key('W.1.running_var')], sd[key('W.1.weight')],
                           sd[key('W.1.bias')], False, 0.0, BN_EPS)
    else:
        w_y = conv(y, sd[key('W.weight')], sd[key('W.bias')])
    return w_y + x


# ---------------------------------------------------------------------------------------------
# whole networks
# ---------------------------------------------------------------------------------------------
def stem(x, sd, family):
    """conv1 -> bn1 -> relu -> maxpool (torchvision_models.py:449-452; modules resnet3D.py:153-156)."""
    if family == 'resnet2d':
        x = F.relu(_bn(_conv(x, sd, 'conv1', 2, 3), sd, 'bn1'))
        return F.max_pool2d(x, 3, 2, 1)
    if family == 'r2plus1d':
        x = spatio_temporal_conv(x, sd, 'conv1', (7, 7, 7), (1, 2, 2), (3, 3, 3))
    else:
        x = _conv(x, sd, 'conv1', (1, 2, 2), (3, 3, 3))
    x = F.relu(_bn(x, sd, 'bn1'))
    return F.max_pool3d(x, kernel_size=(3, 3, 3), stride=2, padding=1)


def trunk(x, sd, arch, stages=None):
    """``features`` (torchvision_models.py:448-458).  If ``stages`` is a dict it receives every stage output."""
    spec = ARCHS[arch] if isinstance(arch, str) else arch
    family, shortcut = spec['family'], spec['shortcut']
    block_fn = {'bottleneck': bottleneck, 'preact_basic': preact_basic_block,
                'preact_bottleneck': preact_bottleneck}.get(spec['block'], basic_block)
    expansion = {'bottleneck': 4, 'preact_bottleneck': 4, 'resnext': 2}.get(spec['block'], 1)
    widths = (128, 256, 512, 1024) if spec['block'] == 'resnext' else (64, 128, 256, 512)     # resnext3D.py:134-137
    nl = nonlocal_positions(spec['layers'], spec['nonlocal_blocks']) if 'nonlocal_blocks' in spec else [[]] * 4
    x = stem(x, sd, family)
    if stages is not None:
        stages['maxpool'] = x
    inplanes = 64
    for li, (planes, nblocks) in enumerate(zip(widths, spec['layers'])):
        for bi in range(nblocks):
            stride = 2 if (li > 0 and bi == 0) else 1
            has_ds = bi == 0 and (stride != 1 or inplanes != planes * expansion)
            p = 'layer%d.%d' % (li + 1, bi)
            if spec['block'] == 'resnext':
                x = resnext_bottleneck(x, sd, p, shortcut, planes, spec['cardinality'], stride, has_ds)
                inplanes = planes * expansion
                continue
            x = block_fn(x, sd, p, 'resnet3d' if family in ('nonlocal', 'resnet2d') else family, shortcut, planes,
                         stride, has_ds)
            if bi in nl[li]:
                x = nonlocal_block(x, sd, p + '.nonlocalblock')
            inplanes = planes * expansion
        if stages is not None:
            stages['layer%d' % (li + 1)] = x
    return x


def head(feat, sd, name=None):
    """avgpool -> view -> last_linear / fc (torchvision_models.py:460-464)."""
    if name is None:
        name = 'last_linear' if 'last_linear.weight' in sd else 'fc'
    pooled = feat.mean(dim=tuple(range(2, feat.dim())))
    return F.linear(pooled, sd[name + '.weight'], sd[name + '.bias'])


def forward(x, sd, arch, stages=None):
    """``model(x)`` = logits(features(x)) (torchvision_models.py:466-469)."""
    feat = trunk(x, sd, arch, stages)
    out = head(feat, sd)
    if stages is not None:
        stages['logits'] = out
    return out


# ---------------------------------------------------------------------------------------------
# SlowFast (slowfast.py) -- SURVEY.md section 8f row n2
# ---------------------------------------------------------------------------------------------
def _sf_block(x, sd, p, bottleneck, stride, head_conv, has_ds):
    """slowfast.py BasicBlock.forward (:38-54) / Bottleneck.forward (:83-101)."""
    if bottleneck:
        c1 = _conv(x, sd, p + '.conv1', 1, (1, 0, 0) if head_conv == 3 else 0)
        out = F.relu(_bn(c1, sd, p + '.bn1'))
        out = F.relu(_bn(_conv(out, sd, p + '.conv2', (1, stride, stride), (0, 1, 1)), sd, p + '.bn2'))
        out = _bn(_conv(out, sd, p + '.conv3'), sd, p + '.bn3')
    else:
        if head_conv == 1:
            c1 = _conv(x, sd, p + '.conv1', (1, stride, stride), (0, 1, 1))
        else:
            c1 = _conv(x, sd, p + '.conv1', 1, (1, 0, 0))
        out = F.relu(_bn(c1, sd, p + '.bn1'))
        out = _bn(_conv(out, sd, p + '.conv2', (1, stride, stride), (0, 1, 1)), sd, p + '.bn2')
    res = x
    if has_ds:
        res = _bn(_conv(x, sd, p + '.downsample.0', (1, stride, stride), 0), sd, p + '.downsample.1')
    return F.relu(out + res)


def _sf_stage(x, sd, p, bottleneck, nblocks, stride, head_conv, inplanes, planes):
    exp = 4 if bottleneck else 1
    for i in range(nblocks):
        s = stride if i == 0 else 1
        has_ds = i == 0 and (stride != 1 or inplanes != planes * exp)
        x = _sf_block(x, sd, '%s.%d' % (p, i), bottleneck, s, head_conv, has_ds)
    return x


def slowfast_forward(x, sd, layers, bottleneck=True, mode='sf', slow_stride=16, fast_stride=2):
    """SlowFast.forward (slowfast.py:390-396), SlowOnly.forward (:217-231), FastOnly.forward (:362-374)."""
    exp = 4 if bottleneck else 1
    res3_stride = 2 if bottleneck else 1
    pool = lambda t: F.max_pool3d(t, (1, 3, 3), (1, 2, 2), (0, 1, 1))
    gap = lambda t: t.mean(dim=(2, 3, 4))
    fp = 'fast.' if mode == 'sf' else ''
    sp = 'slow.' if mode == 'sf' else ''
    lateral = None
    fast = None
    if mode in ('sf', 'f'):
        xf = x[:, :, ::fast_stride]
        a = pool(F.relu(_bn(_conv(xf, sd, fp + 'conv1', (1, 2, 2), (2, 3, 3)), sd, fp + 'bn1')))
        lateral = [] if mode == 'sf' else None
        if lateral is not None:
            lateral.append(_conv(a, sd, fp + 'lateral_p1', (8, 1, 1), (2, 0, 0)))
        inpl = 8
        for name, planes, n, stride in (('res2', 8, layers[0], 1), ('res3', 16, layers[1], res3_stride),
                                        ('res4', 32, layers[2], 2), ('res5', 64, layers[3], 2)):
            a = _sf_stage(a, sd, fp + name, bottleneck, n, stride, 3, inpl, planes)
            inpl = planes * exp
            if lateral is not None and name != 'res5':
                lateral.append(_conv(a, sd, fp + 'lateral_' + name, (8, 1, 1), (2, 0, 0)))
        fast = gap(a)
        if mode == 'f':
            return F.linear(fast, sd['last_linear.weight'], sd['last_linear.bias'])
    xs = x[:, :, ::slow_stride]
    a = pool(F.relu(_bn(_conv(xs, sd, sp + 'conv1', (1, 2, 2), (0, 3, 3)), sd, sp + 'bn1')))
    inpl = 64 + (16 if mode == 'sf' else 0)
    for i, (name, planes, n, stride, head) in enumerate((('res2', 64, layers[0], 1, 1), ('res3', 128, layers[1], res3_stride, 1),
                                                         ('res4', 256, layers[2], 2, 3), ('res5', 512, layers[3], 2, 3))):
        if mode == 'sf':
            a = torch.cat([a, lateral[i]], dim=1)
        a = _sf_stage(a, sd, sp + name, bottleneck, n, stride, head, inpl, planes)
        inpl = planes * exp + (planes * exp // 8 * 2 if mode == 'sf' else 0)
    slow = gap(a)
    if mode == 's':
        return F.linear(slow, sd['last_linear.weight'], sd['last_linear.bias'])
    return F.linear(torch.cat([slow, fast], dim=1), sd['last_linear.weight'], sd.get('last_linear.bias'))


# ---------------------------------------------------------------------------------------------
# TRN relation heads
# ---------------------------------------------------------------------------------------------
def relation(x, sd, p, num_inputs, in_features):
    """Relation.func (trn.py:47-49): view(-1, T*F) -> ReLU -> Linear -> ReLU -> Linear -> view(B, -1, out)."""
    flat = x.contiguous().view(-1, num_inputs * in_features)
    h = F.relu(F.linear(F.relu(flat), sd[p + 'relate.1.weight'], sd[p + 'relate.1.bias']))
    out = F.linear(h, sd[p + 'relate.3.weight'], sd[p + 'relate.3.bias'])
    return out.view(x.size(0), -1, out.shape[-1])


def multiscale_relation(x, sd, num_input, in_features, num_relations=3, tuples=None, p=''):
    """MultiScaleRelation.forward (trn.py:100-110).  ``tuples`` (per scale) overrides the np.random.choice draw;
    when None the draw is made exactly as the reference does, from NumPy's global RNG.  ``p``: state_dict key prefix."""
    scales = list(range(num_input, 1, -1))
    sets = [list(itertools.combinations(range(num_input), s)) for s in scales]
    outs = []
    for si, s in enumerate(scales):
        if tuples is None:
            idx = np.random.choice(len(sets[si]), min(num_relations, len(sets[si])), replace=False)
            chosen = [sets[si][i] for i in idx]
        else:
            chosen = tuples[si]
        for tup in chosen:
            outs.append(relation(x[..., list(tup), :], sd, p + 'relations.%d.' % si, s, in_features))
    total = torch.stack(outs).sum(0)
    return total.view(x.size(0), -1, total.shape[-1])


def trn_forward(x, sd, arch, consensus, num_segments, stages=None):
    """TRN.forward (trn.py:246-263) in eval mode: frames folded into the batch of the 2-D backbone (``base_model.*`` keys, whose
    ``last_linear`` is a Dropout == identity, :211-212), pooled frame features regrouped [B, 1, T, F] (:249-254), consensus
    module (``Relation`` for 'TRN', the degenerate depth-0 ``HierarchicalRelation`` == its ``final_relation`` for 'HTRN'
    (:155-158 with no hierarchy levels), ``MultiScaleRelation`` for 'MSTRN'), ``.squeeze()``, final Linear (:257-258)."""
    base = {k[len('base_model.'):]: v for k, v in sd.items() if k.startswith('base_model.')}
    b = x.size(0)
    frames = x.view((-1, 3) + tuple(x.shape[-2:]))
    feat = trunk(frames, base, arch)
    rep = feat.mean(dim=(2, 3))                                   # avgpool + view; Dropout (eval) is the identity
    fdim = rep.size(-1)
    rep = rep.view(b, -1, num_segments, fdim)
    t_in = rep.view(-1, rep.size(1), num_segments, fdim)
    if consensus == 'TRN':
        v = relation(t_in, sd, 'temporal_relation.', num_segments, fdim)
    elif consensus == 'HTRN':
        v = relation(t_in.view(-1, num_segments, fdim), sd, 'temporal_relation.final_relation.', num_segments, fdim)
    elif consensus == 'MSTRN':
        v = multiscale_relation(t_in, sd, num_segments, fdim, p='temporal_relation.')
    else:
        raise ValueError(consensus)
    v = v.squeeze()
    if stages is not None:
        stages['features'] = v
    return F.linear(v, sd['last_linear.weight'], sd['last_linear.bias'])


# ---------------------------------------------------------------------------------------------
# deterministic test conditioning shared by the golden generator and the tests
# ---------------------------------------------------------------------------------------------
def randomize_bn_(module, seed):
    """Give every BatchNorm non-trivial affine + running stats (SURVEY.md section 8c) so that BN folding bugs
    cannot hide behind identity statistics.  Walks ``named_modules()`` in order; works on the reference's
    modules and on pretorched_x_b200's alike (same tree => same values)."""
    g = torch.Generator().manual_seed(seed)
    for _, m in module.named_modules():
        if isinstance(m, torch.nn.modules.batchnorm._BatchNorm):
            n = m.num_features
            m.running_mean.copy_(torch.randn(n, generator=g) * 0.1)
            m.running_var.copy_(torch.rand(n, generator=g) + 0.5)
            m.weight.data.copy_(torch.rand(n, generator=g) + 0.5)
            m.bias.data.copy_(torch.randn(n, generator=g) * 0.1)
    return module


def seeded_input(shape, seed):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


def state_digest(sd):
    """Per-tensor (sum, abs-sum) in float64 -- a cheap fingerprint to prove two inits are identical."""
    return {k: (float(v.double().sum()), float(v.double().abs().sum())) for k, v in sd.items()}


def digests_match(a, b, rtol=1e-9):
    """Compare two ``state_digest`` results.  The float64 sums are reduced by the host CPU's vector units, whose
    summation order differs between machines, so equality is up to a few ulps rather than bit-exact."""
    if list(a) != list(b):
        return False
    for k in a:
        for u, v in zip(a[k], b[k]):
            if abs(u - v) > rtol * max(abs(u), abs(v), 1e-30):
                return False
    return True


def state_hashes(sd):
    """Per-tensor (shape, dtype, SHA-256 of the raw bytes): equal hashes mean ``torch.equal`` tensors, so a stored copy
    can stand in for a state_dict that is too large to keep."""
    return {k: (tuple(v.shape), str(v.dtype), hashlib.sha256(v.detach().contiguous().cpu().numpy().tobytes()).hexdigest())
            for k, v in sd.items()}


def calibrate_nonlocal_(model, x, target_std=3.0):
    """Rescale theta/phi of every non-local block, in execution order, so that the std of its logits
    f = theta^T phi on input ``x`` equals ``target_std``; returns {block name: factor}.

    At raw random init the reference's unscaled logits reach 1e4..1e8: the softmax is an arg-max whose top-2 gaps can
    fall below fp16 (even fp32 re-association) resolution, and one flipped row is amplified by every later block --
    end-to-end comparison of the whole network is then chaotic rather than informative.  Trained checkpoints live in
    a benign regime; this data-dependent rescale (a one-pass LSUV on the logits) emulates one.  It runs on the
    REFERENCE model when fixtures are generated; tests re-apply the recorded factors with
    ``apply_nonlocal_factors_`` so both sides hold identical weights."""
    factors = {}
    blocks = [(n, m) for n, m in model.named_modules() if n.endswith("nonlocalblock")]
    for name, blk in blocks:
        seen = {}
        handle = blk.register_forward_hook(lambda m, i, o: seen.__setitem__("x", i[0].detach()))
        with torch.no_grad():
            model(x)
        handle.remove()
        xin = seen["x"]
        with torch.no_grad():
            th = blk.theta(xin).flatten(2)
            ph = blk.phi(xin).flatten(2)
            f = th.transpose(1, 2) @ ph
            s = float((target_std / f.std().item()) ** 0.5)
        apply_nonlocal_factors_(model, {name: s})
        factors[name] = s
    return factors


def apply_nonlocal_factors_(module, factors):
    """Multiply theta/phi (weights and biases) of the named non-local blocks by the given factors."""
    mods = dict(module.named_modules())
    with torch.no_grad():
        for name, s in factors.items():
            for proj in (mods[name].theta, mods[name].phi):
                proj.weight.mul_(s)
                proj.bias.mul_(s)
    return module
