"""Generate the golden fixtures in this directory from the REAL reference.

Runs only in the authoring container (needs /root/reference, which does not exist on the GPU
box).  It imports toandaominh1997/EfficientDet.Pytorch with the three shims of SURVEY.md 8(c):
  1. models.efficientnet.load_pretrained_weights -> no-op   (no network)
  2. torch.Tensor.cuda -> identity                          (losses.py hard-codes .cuda())
  3. BiFPNModule.relu1/relu2 -> relu(x).clone()             (in-place `/=` on a ReLU output
                                                             breaks autograd on torch>=1.5)
then, for each case, loads oracle-generated weights into the reference, runs the reference
and the oracle on identical inputs, REQUIRES bit-exact agreement (torch.equal) of every
intermediate, and stores sampled reference outputs (+ float64 norms) as small .npz files.
tests/test_oracle_golden.py re-checks the oracle against these files anywhere.

usage:  python tests/golden/make_golden.py
"""
import hashlib
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get('EFFDET_REFERENCE', '/root/reference')
sys.path.insert(0, REF)
sys.path.insert(0, os.path.join(REPO, 'oracle'))

import effdet_oracle as O  # noqa: E402

import models.efficientnet as ref_effnet  # noqa: E402  (the reference)
ref_effnet.load_pretrained_weights = lambda *a, **k: None
torch.Tensor.cuda = lambda self, *a, **k: self
import models.bifpn as ref_bifpn  # noqa: E402
from models.efficientdet import EfficientDet as RefEfficientDet  # noqa: E402


class _ReluClone(torch.nn.Module):
    def forward(self, x):
        return torch.relu(x).clone()


def build_reference(cfg, sd, is_training, threshold=0.01, iou_threshold=0.5):
    torch.manual_seed(0)
    m = RefEfficientDet(num_classes=cfg['num_classes'], network=cfg['network'], D_bifpn=cfg['D'],
                        W_bifpn=cfg['W'], is_training=is_training, threshold=threshold,
                        iou_threshold=iou_threshold)
    for mod in m.modules():
        if isinstance(mod, ref_bifpn.BiFPNModule):
            mod.relu1, mod.relu2 = _ReluClone(), _ReluClone()
    ref_keys = list(m.state_dict().keys())
    assert ref_keys == list(sd.keys()), 'state-dict schema differs from the reference'
    for k, v in m.state_dict().items():
        assert tuple(v.shape) == tuple(sd[k].shape), (k, v.shape, sd[k].shape)
    m.load_state_dict(sd)
    return m


def sample(t, n=257):
    a = t.detach().cpu().contiguous().view(-1)
    idx = np.unique(np.linspace(0, a.numel() - 1, n).astype(np.int64))
    return a[torch.from_numpy(idx)].numpy().copy(), idx


def put(store, name, t):
    v, idx = sample(t)
    store[name + '/s'] = v
    store[name + '/i'] = idx
    store[name + '/n'] = np.array([float(torch.linalg.vector_norm(t.detach().double())),
                                   float(t.detach().double().sum())])
    store[name + '/shape'] = np.array(t.shape, dtype=np.int64)


def must_equal(name, a, b):
    if not torch.equal(a, b):
        raise SystemExit('oracle != reference at %s (max abs %g)' % (name, float((a - b).abs().max())))


def run_forward_case(tag, cfg, mode, size, B, seed, threshold=None):
    sd = O.init_state_dict(cfg, seed=seed, mode=mode)
    if threshold is None:
        threshold = 0.3 if mode == 'wellcond' else 0.01
    ref = build_reference(cfg, sd, is_training=False, threshold=threshold)
    ref.eval()
    images, _ = O.synthetic_batch(B, size=size, seed=100 + seed)
    cap = {}
    hooks = []
    hooks.append(ref.backbone.register_forward_hook(lambda m, i, o: cap.__setitem__('P', list(o))))
    for i, lc in enumerate(ref.neck.lateral_convs):
        hooks.append(lc.register_forward_hook(lambda m, i_, o, i=i: cap.__setitem__('lat%d' % i, o)))
    for d, layer in enumerate(ref.neck.stack_bifpn_convs):
        hooks.append(layer.register_forward_hook(lambda m, i_, o, d=d: cap.__setitem__('bifpn%d' % d, list(o))))
    hooks.append(ref.bbox_head.register_forward_hook(lambda m, i, o: cap.__setitem__('head', o)))
    with torch.no_grad():
        det_ref = ref(images[:1].clone()) if B == 1 else None
        cap1 = dict(cap)
        coll = {}
        det_orc = O.detect(sd, images[:1], cfg, threshold=ref.threshold, iou_threshold=ref.iou_threshold,
                           collect=coll) if B == 1 else None
    for h in hooks:
        h.remove()
    store = {}
    for li in range(7):
        must_equal('P%d' % li, cap1['P'][li], coll['P'][li])
        put(store, 'P%d' % li, cap1['P'][li])
    for li in range(5):
        must_equal('lat%d' % li, cap1['lat%d' % li], coll['laterals'][li])
        put(store, 'lat%d' % li, cap1['lat%d' % li])
    for d in range(cfg['D']):
        for li in range(5):
            must_equal('bifpn%d_%d' % (d, li), cap1['bifpn%d' % d][li], coll['bifpn%d' % d][li])
            put(store, 'bifpn%d_%d' % (d, li), cap1['bifpn%d' % d][li])
    cls_ref = torch.cat(cap1['head'][0], dim=1)
    reg_ref = torch.cat(cap1['head'][1], dim=1)
    must_equal('cls', cls_ref, coll['cls'])
    must_equal('reg', reg_ref, coll['reg'])
    put(store, 'cls', cls_ref)
    put(store, 'reg', reg_ref)
    anc_ref = ref.anchors(images[:1])
    must_equal('anchors', anc_ref, coll['anchors'])
    store['anchors/sha256'] = np.frombuffer(hashlib.sha256(anc_ref.numpy().tobytes()).digest(), dtype=np.uint8)
    store['anchors/head'] = anc_ref[0, :18].numpy()
    store['anchors/tail'] = anc_ref[0, -18:].numpy()
    store['anchors/shape'] = np.array(anc_ref.shape)
    # detection outputs of the reference (torchvision NMS inside) vs oracle (nms_greedy)
    assert len(det_ref) == 3
    for k, (a, b) in enumerate(zip(det_ref, det_orc)):
        must_equal('det%d' % k, a, b)
    store['det/scores'] = det_ref[0].numpy()
    store['det/classes'] = det_ref[1].numpy()
    store['det/boxes'] = det_ref[2].numpy()
    store['det/threshold'] = np.array([ref.threshold, ref.iou_threshold])
    store['meta/seed'] = np.array([seed, size, B])
    np.savez_compressed(os.path.join(HERE, tag + '.npz'), **store)
    print('%-28s ok: %d tensors pinned, %d detections' % (tag, len(store), det_ref[0].numel()))


def run_train_case(tag, cfg, size, B, seed, empty_first, samples=True):
    """samples=False leaves out the sampled large gradients (gsamp/), which only the D0 GPU test reads: the D4 file
    stays under 1 MB with every full gradient and every norm kept"""
    sd = O.init_state_dict(cfg, seed=seed, mode='wellcond')
    ref = build_reference(cfg, sd, is_training=True)
    ref.eval()                 # no drop-connect; BN is frozen in either mode
    ref.is_training = True
    images, ann = O.synthetic_batch(B, size=size, num_classes=cfg['num_classes'], seed=200 + seed,
                                    empty_first=empty_first)
    cl, rl = ref([images.clone(), ann.clone()])
    (cl.mean() + rl.mean()).backward()
    # oracle
    sdg = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and 'running' not in k else v)
           for k, v in sd.items()}
    ocl, orl = O.train_forward(sdg, images, ann, cfg)
    (ocl.mean() + orl.mean()).backward()
    must_equal('cls_loss', cl.detach(), ocl.detach())
    must_equal('reg_loss', rl.detach(), orl.detach())
    store = {'loss/cls': cl.detach().numpy(), 'loss/reg': rl.detach().numpy()}
    names, norms = [], []
    worst = 0.0
    for k, p in ref.named_parameters():
        g = p.grad
        og = sdg[k].grad
        if g is None:
            assert og is None or float(og.abs().max()) == 0.0, k
            continue
        # autograd accumulation order may differ between module graph and functional graph:
        # require agreement to fp32 round-off, not bit equality
        e = O.rel_err(og, g)
        worst = max(worst, e)
        assert e < 2e-5, (k, e)
        names.append(k)
        norms.append(float(torch.linalg.vector_norm(g.double())))
        if g.numel() <= 4096 or k.endswith('w1') or k.endswith('w2'):
            store['grad/' + k] = g.numpy().copy()
        elif samples:
            v, idx = sample(g, 129)
            store['gsamp/' + k + '/s'] = v
            store['gsamp/' + k + '/i'] = idx
    store['grad_names'] = np.array(names)
    store['grad_norms'] = np.array(norms)
    store['meta/seed'] = np.array([seed, size, B, int(empty_first)])
    np.savez_compressed(os.path.join(HERE, tag + '.npz'), **store)
    print('%-28s ok: losses %.6f %.6f, %d grads pinned (oracle-vs-reference worst rel %.2e)'
          % (tag, float(cl), float(rl), len(names), worst))


def run_nms_case():
    """torchvision.ops.nms (CPU) vs oracle.nms_greedy on adversarial inputs (ties, IoU == thr)."""
    from torchvision.ops import nms
    g = torch.Generator().manual_seed(7)
    store = {}
    for case in range(4):
        n = [200, 1500, 64, 3000][case]
        xy = torch.rand(n, 2, generator=g) * 300
        wh = torch.rand(n, 2, generator=g) * 80 + 2
        boxes = torch.cat([xy, xy + wh], dim=1)
        scores = torch.rand(n, generator=g)
        if case == 1:
            scores = (scores * 20).floor() / 20          # many ties
        if case == 2:
            boxes = torch.tensor([[0, 0, 10, 10.]]).repeat(n, 1)
            boxes[1::2] = torch.tensor([0, 0, 10, 5.])   # IoU exactly 0.5 against evens
        keep_tv = nms(boxes, scores, 0.5)
        keep_or = O.nms_greedy(boxes, scores, 0.5)
        must_equal('nms%d' % case, keep_tv, keep_or)
        store['c%d/boxes' % case] = boxes.numpy()
        store['c%d/scores' % case] = scores.numpy()
        store['c%d/keep' % case] = keep_tv.numpy()
    np.savez_compressed(os.path.join(HERE, 'nms_torchvision.npz'), **store)
    print('nms_torchvision             ok')


if __name__ == '__main__':
    # usage: make_golden.py [substring]   -- regenerate only the fixtures whose tag contains the substring
    only = sys.argv[1] if len(sys.argv) > 1 else ''
    torch.set_num_threads(8)
    d0 = O.make_config('efficientdet-d0', num_classes=80, W_bifpn=64, D_bifpn=2)
    d0s = O.make_config('efficientdet-d0', num_classes=20, W_bifpn=64, D_bifpn=2)
    d1 = O.make_config('efficientdet-d1', num_classes=20, W_bifpn=88, D_bifpn=3)
    # the deep / wide family members whose GPU tests (D4 1024^2 train step, D7 1536^2 inference) compare against the
    # ORACLE: pin the oracle to the reference on the same architectures at a CPU-sized resolution
    d4 = O.make_config('efficientdet-d4', num_classes=20, W_bifpn=224, D_bifpn=6)
    d7 = O.make_config('efficientdet-d7', num_classes=20, W_bifpn=384, D_bifpn=8)
    cases = [
        ('nms_torchvision', run_nms_case, ()),
        ('d0_512_fwd_wellcond', run_forward_case, (d0, 'wellcond', 512, 1, 1)),
        ('d0_512_fwd_asbuilt', run_forward_case, (d0, 'asbuilt', 512, 1, 2)),
        ('d0_256_train_b2', run_train_case, (d0s, 256, 2, 3, False)),
        ('d0_256_train_b2_empty', run_train_case, (d0s, 256, 2, 4, True)),
        ('d1_384_fwd_wellcond', run_forward_case, (d1, 'wellcond', 384, 1, 5)),
        ('d4_256_fwd_wellcond', run_forward_case, (d4, 'wellcond', 256, 1, 6, 0.05)),
        ('d4_128_train_b2', run_train_case, (d4, 128, 2, 7, False, False)),
        ('d7_256_fwd_wellcond', run_forward_case, (d7, 'wellcond', 256, 1, 8, 0.05)),
    ]
    for tag, fn, a in cases:
        if only in tag:
            fn(*((tag,) + a)) if fn is not run_nms_case else fn()
