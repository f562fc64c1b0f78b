"""The oracle against the golden vectors captured from the real reference
(tests/golden/make_golden.py).  CPU only; no /root/reference needed."""
import hashlib
import os

import numpy as np
import pytest
import torch

import effdet_oracle as O

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


@pytest.fixture(autouse=True)
def golden_threads():
    """torch's CPU convolutions split their work by thread count and the bits depend on the split: run at the 8 threads
    the goldens were captured with (make_golden.py), whatever the host's core count or an earlier test set"""
    n = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(n)


def _check(store, name, t):
    s, i = store[name + '/s'], store[name + '/i']
    assert tuple(store[name + '/shape']) == tuple(t.shape), name
    got = t.detach().contiguous().view(-1)[torch.from_numpy(i)].numpy()
    assert np.array_equal(got, s), '%s: sampled values differ from the reference' % name
    n = float(torch.linalg.vector_norm(t.detach().double()))
    assert abs(n - store[name + '/n'][0]) <= 1e-9 * max(1.0, n), name


@pytest.mark.parametrize('tag,net,W,D,K,mode', [
    ('d0_512_fwd_wellcond', 'efficientdet-d0', 64, 2, 80, 'wellcond'),
    ('d0_512_fwd_asbuilt', 'efficientdet-d0', 64, 2, 80, 'asbuilt'),
    ('d1_384_fwd_wellcond', 'efficientdet-d1', 88, 3, 20, 'wellcond'),
    # the architectures whose GPU tests (D4 1024^2 train step, D7 1536^2 inference) use the oracle as the checker
    ('d4_256_fwd_wellcond', 'efficientdet-d4', 224, 6, 20, 'wellcond'),
    ('d7_256_fwd_wellcond', 'efficientdet-d7', 384, 8, 20, 'wellcond'),
])
def test_forward_matches_reference_golden(tag, net, W, D, K, mode):
    st = np.load(os.path.join(G, tag + '.npz'))
    seed, size, B = [int(v) for v in st['meta/seed']]
    cfg = O.make_config(net, num_classes=K, W_bifpn=W, D_bifpn=D)
    sd = O.init_state_dict(cfg, seed=seed, mode=mode)
    images, _ = O.synthetic_batch(B, size=size, seed=100 + seed)
    coll = {}
    thr, iou = [float(v) for v in st['det/threshold']]
    with torch.no_grad():
        det = O.detect(sd, images[:1], cfg, threshold=thr, iou_threshold=iou, collect=coll)
    for li in range(7):
        _check(st, 'P%d' % li, coll['P'][li])
    for li in range(5):
        _check(st, 'lat%d' % li, coll['laterals'][li])
        for d in range(D):
            _check(st, 'bifpn%d_%d' % (d, li), coll['bifpn%d' % d][li])
    _check(st, 'cls', coll['cls'])
    _check(st, 'reg', coll['reg'])
    anc = coll['anchors'].numpy()
    assert hashlib.sha256(anc.tobytes()).digest() == bytes(st['anchors/sha256'])
    assert np.array_equal(anc[0, :18], st['anchors/head']) and np.array_equal(anc[0, -18:], st['anchors/tail'])
    assert np.array_equal(det[0].numpy(), st['det/scores'])
    assert np.array_equal(det[1].numpy(), st['det/classes'])
    assert np.array_equal(det[2].numpy(), st['det/boxes'])


@pytest.mark.parametrize('tag,net,W,D,nlive', [('d0_256_train_b2', 'efficientdet-d0', 64, 2, 274),
                                               ('d0_256_train_b2_empty', 'efficientdet-d0', 64, 2, 274),
                                               ('d4_128_train_b2', 'efficientdet-d4', 224, 6, 551)])
def test_train_step_matches_reference_golden(tag, net, W, D, nlive):
    st = np.load(os.path.join(G, tag + '.npz'))
    seed, size, B, empty = [int(v) for v in st['meta/seed']]
    cfg = O.make_config(net, num_classes=20, W_bifpn=W, D_bifpn=D)
    sd = O.init_state_dict(cfg, seed=seed, mode='wellcond')
    images, ann = O.synthetic_batch(B, size=size, num_classes=20, seed=200 + seed, empty_first=bool(empty))
    sdg = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and 'running' not in k else v)
           for k, v in sd.items()}
    cl, rl = O.train_forward(sdg, images, ann, cfg)
    (cl.mean() + rl.mean()).backward()
    assert np.array_equal(cl.detach().numpy(), st['loss/cls'])
    assert np.array_equal(rl.detach().numpy(), st['loss/reg'])
    names, norms = list(st['grad_names']), st['grad_norms']
    assert len(names) == nlive
    for k, n in zip(names, norms):
        g = sdg[str(k)].grad
        gn = float(torch.linalg.vector_norm(g.double()))
        assert abs(gn - n) <= 2e-5 * max(n, 1e-30), (k, gn, n)
        key = 'grad/' + str(k)
        if key in st.files:
            ref = torch.from_numpy(st[key])
            assert O.rel_err(g, ref) < 2e-5, k
    # the 5 dead backbone params get no gradient (SURVEY 2.1)
    dead = [k for k, v in sdg.items() if v.is_floating_point() and v.requires_grad and
            (v.grad is None or float(v.grad.abs().max()) == 0.0)]
    # (signed fusion weights can additionally kill a lateral branch through the ReLU)
    assert set(['backbone._conv_head.weight', 'backbone._bn1.weight', 'backbone._bn1.bias',
                'backbone._fc.weight', 'backbone._fc.bias']) <= set(dead)
    assert all(k.startswith('backbone._') and 'blocks' not in k or k.startswith('neck.') for k in dead), dead


def test_nms_greedy_matches_torchvision_golden():
    st = np.load(os.path.join(G, 'nms_torchvision.npz'))
    for c in range(4):
        keep = O.nms_greedy(torch.from_numpy(st['c%d/boxes' % c]), torch.from_numpy(st['c%d/scores' % c]), 0.5)
        assert np.array_equal(keep.numpy(), st['c%d/keep' % c])


def test_state_dict_schema_counts():
    cfg = O.make_config('efficientdet-d0', 80, 64, 2)
    spec = O.state_dict_spec(cfg)
    assert len(spec) == 426                      # SURVEY section 5
    sd = O.init_state_dict(cfg, 0)
    nparam = sum(v.numel() for k, v in sd.items() if v.is_floating_point() and 'running' not in k)
    assert nparam == 11505854                    # BASELINE.md section 2
    assert O.anchors_for(512, 512).shape == (1, 49104, 4)
