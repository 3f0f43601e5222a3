"""Generate tests/golden/*.npz by EXECUTING THE REFERENCE (build container only).

    python tests/golden/make_golden.py [/root/reference]

The reference has no tests or golden vectors of its own (SURVEY.md section 4), so the
pin for every parity claim is the reference code itself, run here on seeded inputs.
The reference tree does not exist on the GPU box; only the small .npz files
written by this script travel.  Import recipe: SURVEY.md Appendix B (three stub
modules, none on the arithmetic path).  Nothing is copied from the reference; its
functions are called and their outputs recorded.
"""
import os
import sys
import types
from types import SimpleNamespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = sys.argv[1] if len(sys.argv) > 1 else '/root/reference'
sys.dont_write_bytecode = True
sys.path.insert(0, REF)
sys.path.insert(1, ROOT)


def _install_stubs():
    import torch.nn as nn
    for name in ['matplotlib', 'matplotlib.pyplot', 'skimage', 'skimage.filters', 'kornia', 'kornia.augmentation']:
        sys.modules[name] = types.ModuleType(name)
    sys.modules['skimage.filters'].gaussian = lambda *a, **k: None

    class Identity(nn.Module):
        def __init__(self, *a, **k):
            super().__init__()

        def forward(self, x):
            return x
    for n in ['RandomResizedCrop', 'RandomHorizontalFlip', 'ColorJitter', 'RandomGrayscale']:
        setattr(sys.modules['kornia.augmentation'], n, Identity)


_install_stubs()
import warnings
warnings.filterwarnings('ignore')

from utils.buffer import aser_utils, aser_retrieve, aser_update, buffer_utils, mir_retrieve, reservoir_update  # noqa: E402
from utils.loss import SupConLoss                                    # noqa: E402
from utils.setup_elements import setup_architecture                  # noqa: E402
from oracle import resnet as oresnet                                 # noqa: E402  (only for the seeded weight stream)

torch.set_num_threads(8)


def relu_feats(rs, n, d):
    return np.maximum(rs.standard_normal((n, d)), 0).astype(np.float32)


# ----------------------------------------------------------------------------- kNN-SV
def gen_knn_sv():
    out = {}
    cases = [(10, 100, 160, 3, 100), (100, 100, 160, 3, 100), (110, 160, 160, 3, 100),
             (7, 1, 16, 3, 2), (5, 2, 16, 3, 2), (5, 3, 16, 3, 2), (6, 4, 16, 3, 3),
             (12, 37, 32, 5, 4), (9, 64, 24, 1, 3), (33, 257, 40, 3, 10), (3, 600, 64, 3, 20)]
    orig = aser_utils.deep_features
    aser_utils.deep_features = lambda model, ex, ne, cx, nc: (ex, cx)
    rs = np.random.RandomState(1234)
    for i, (E, C, d, k, ncls) in enumerate(cases):
        ef, cf = relu_feats(rs, E, d), relu_feats(rs, C, d)
        ey, cy = rs.randint(0, ncls, E), rs.randint(0, ncls, C)
        sv = aser_utils.compute_knn_sv(None, torch.tensor(ef), torch.tensor(ey), torch.tensor(cf),
                                       torch.tensor(cy), k)
        order = aser_utils.sorted_cand_ind(torch.tensor(ef), torch.tensor(cf), E, C)
        out.update({'c%d_ef' % i: ef, 'c%d_cf' % i: cf, 'c%d_ey' % i: ey, 'c%d_cy' % i: cy,
                    'c%d_k' % i: np.int64(k), 'c%d_sv' % i: sv.numpy(), 'c%d_order' % i: order.numpy()})
    out['n_cases'] = np.int64(len(cases))
    aser_utils.deep_features = orig
    np.savez_compressed(os.path.join(HERE, 'knn_sv.npz'), **out)


# ----------------------------------------------------------------------------- SupCon
def gen_supcon():
    out = {}
    rs = np.random.RandomState(77)
    cases = [(8, 2, 16, 0.07, 3, True), (110, 2, 128, 0.07, 100, True), (16, 3, 32, 0.1, 4, True),
             (12, 1, 8, 0.5, 2, False), (20, 2, 24, 0.07, 20, True)]
    for i, (B, V, d, T, ncls, norm) in enumerate(cases):
        f = rs.standard_normal((B, V, d)).astype(np.float32)
        if norm:
            f /= np.linalg.norm(f, axis=2, keepdims=True)
        y = rs.randint(0, ncls, B)
        ft = torch.tensor(f, requires_grad=True)
        loss = SupConLoss(temperature=T)(ft, torch.tensor(y))
        loss.backward()
        out.update({'c%d_f' % i: f, 'c%d_y' % i: y, 'c%d_T' % i: np.float64(T),
                    'c%d_loss' % i: loss.detach().numpy(), 'c%d_grad' % i: ft.grad.numpy()})
    out['n_cases'] = np.int64(len(cases))
    np.savez_compressed(os.path.join(HERE, 'supcon.npz'), **out)


# ----------------------------------------------------------------------------- ResNet
def _ref_model(data, agent, head, spec, seed):
    params = SimpleNamespace(data=data, agent=agent, head=head)
    model = setup_architecture(params)
    p, bn = oresnet.seeded_state(spec, seed)
    sd = dict(p)
    sd.update(bn)
    missing = model.load_state_dict(sd, strict=True)
    return model, p, bn


def _grad_summary(model, out, tag):
    names, norms = [], []
    for name, prm in model.named_parameters():
        names.append(name)
        norms.append(0.0 if prm.grad is None else float(prm.grad.double().norm()))
    out[tag + '_grad_norms'] = np.array(norms)
    out[tag + '_grad_names'] = np.array(names)
    keep = ['conv1.weight', 'bn1.weight', 'bn1.bias', 'layer1.0.conv1.weight', 'layer2.0.shortcut.0.weight',
            'layer2.0.shortcut.1.weight', 'layer3.1.bn2.bias', 'layer4.0.conv1.weight', 'linear.weight',
            'linear.bias', 'head.0.weight', 'head.2.bias']
    for name, prm in model.named_parameters():
        short = name.replace('encoder.', '')
        if short in keep and prm.grad is not None:
            g = prm.grad.numpy()
            if g.size > 30000:
                g = g.reshape(g.shape[0], -1)[:8]
            out[tag + '_grad__' + name] = g


def gen_resnet():
    out = {}
    rs = np.random.RandomState(5)
    # ---- CIFAR-100 classifier (Reduced_ResNet18(100), setup_elements.py:55-56)
    spec = oresnet.Spec(32, 20, 100)
    model, p, bn = _ref_model('cifar100', 'ER', None, spec, seed=11)
    x = rs.uniform(0, 1, (6, 3, 32, 32)).astype(np.float32)
    y = rs.randint(0, 100, 6)
    out['cifar_x'], out['cifar_y'] = x, y
    model.eval()
    with torch.no_grad():
        out['cifar_feat_eval'] = model.features(torch.tensor(x)).numpy()
        out['cifar_logits_eval'] = model(torch.tensor(x)).numpy()
    model.train()
    logits = model(torch.tensor(x))
    loss = torch.nn.functional.cross_entropy(logits, torch.tensor(y))
    model.zero_grad()
    loss.backward()
    out['cifar_logits_train'] = logits.detach().numpy()
    out['cifar_loss'] = loss.detach().numpy()
    _grad_summary(model, out, 'cifar')
    sd = model.state_dict()
    for k in ['bn1', 'layer1.0.bn2', 'layer2.0.shortcut.1', 'layer4.1.bn2']:
        out['cifar_rm__' + k] = sd[k + '.running_mean'].numpy().copy()
        out['cifar_rv__' + k] = sd[k + '.running_var'].numpy().copy()
    # MIR scores on the same model state (grads present, stats already moved once)
    sub_x = rs.uniform(0, 1, (12, 3, 32, 32)).astype(np.float32)
    sub_y = rs.randint(0, 100, 12)
    buf = SimpleNamespace(model=model, buffer_img=torch.tensor(sub_x), buffer_label=torch.tensor(sub_y),
                          current_index=12)
    mp = SimpleNamespace(subsample=12, eps_mem_batch=4, learning_rate=0.1)
    np.random.seed(3)
    retr = mir_retrieve.MIR_retrieve(mp)
    rec = {}
    orig_rr = mir_retrieve.random_retrieve

    def rec_rr(buffer, n, *a, **k):
        xs, ys, idx = orig_rr(buffer, n, return_indices=True)
        rec['idx'] = idx.numpy()
        return xs, ys
    mir_retrieve.random_retrieve = rec_rr
    # re-run pieces by hand to also record the scores (mir_retrieve.py:23-29)
    grad_dims = [q.data.numel() for q in model.parameters()]
    gv = buffer_utils.get_grad_vector(model.parameters, grad_dims)
    sx, sy = rec_rr(buf, 12)
    mt = retr.get_future_step_parameters(model, gv, grad_dims)
    with torch.no_grad():
        pre = torch.nn.functional.cross_entropy(model(sx), sy, reduction='none')
        post = torch.nn.functional.cross_entropy(mt(sx), sy, reduction='none')
    mir_retrieve.random_retrieve = orig_rr
    out['mir_sub_x'], out['mir_sub_y'], out['mir_perm'] = sub_x, sub_y, rec['idx']
    out['mir_scores'] = (post - pre).numpy()
    out['mir_top'] = (post - pre).sort(descending=True)[1][:4].numpy()
    out['mir_rm_after__bn1'] = model.state_dict()['bn1.running_mean'].numpy().copy()

    # ---- Mini-ImageNet classifier (linear 640->100, setup_elements.py:63-66)
    spec = oresnet.Spec(84, 20, 100)
    model, p, bn = _ref_model('mini_imagenet', 'ER', None, spec, seed=12)
    x = rs.uniform(0, 1, (2, 3, 84, 84)).astype(np.float32)
    out['mini_x'] = x
    model.eval()
    with torch.no_grad():
        out['mini_feat_eval'] = model.features(torch.tensor(x)).numpy()
        out['mini_logits_eval'] = model(torch.tensor(x)).numpy()
    model.train()
    ym = rs.randint(0, 100, 2)
    logits = model(torch.tensor(x))
    loss = torch.nn.functional.cross_entropy(logits, torch.tensor(ym))
    model.zero_grad()
    loss.backward()
    out['mini_y'] = ym
    out['mini_logits_train'] = logits.detach().numpy()
    out['mini_loss'] = loss.detach().numpy()
    _grad_summary(model, out, 'mini')

    # ---- SupConResNet(head=mlp), two views, SupCon loss (scr.py:52-60)
    spec = oresnet.Spec(32, 20, 100, head='mlp')
    model, p, bn = _ref_model('cifar100', 'SCR', 'mlp', spec, seed=13)
    x1 = rs.uniform(0, 1, (8, 3, 32, 32)).astype(np.float32)
    x2 = np.clip(x1[:, :, :, ::-1] * 0.9 + 0.05, 0, 1).astype(np.float32).copy()
    ys = rs.randint(0, 4, 8)
    model.train()
    feats = torch.cat([model(torch.tensor(x1)).unsqueeze(1), model(torch.tensor(x2)).unsqueeze(1)], dim=1)
    loss = SupConLoss(temperature=0.07)(feats, torch.tensor(ys))
    model.zero_grad()
    loss.backward()
    out['scr_x1'], out['scr_x2'], out['scr_y'] = x1, x2, ys
    out['scr_feats'] = feats.detach().numpy()
    out['scr_loss'] = loss.detach().numpy()
    _grad_summary(model, out, 'scr')
    out['scr_rm__encoder.bn1'] = model.state_dict()['encoder.bn1.running_mean'].numpy().copy()
    out['scr_rv__encoder.bn1'] = model.state_dict()['encoder.bn1.running_var'].numpy().copy()
    model.eval()
    with torch.no_grad():
        out['scr_enc_feat_eval'] = model.features(torch.tensor(x1)).numpy()
    np.savez_compressed(os.path.join(HERE, 'resnet.npz'), **out)


# ----------------------------------------------------------------------------- ASER plugins
def gen_aser():
    """Run the reference ASER retrieve / update on feature-space 'images' (the network is
    bypassed: deep_features := identity) and record every sampled set and every decision."""
    out = {}
    orig = aser_utils.deep_features
    aser_utils.deep_features = lambda model, ex, ne, cx, nc: (ex, cx)
    rs = np.random.RandomState(99)
    CB = buffer_utils.ClassBalancedRandomSampling
    n_case = 0
    for (mem, ncls, d, n_smp, aser_type, skew, data) in [
            (400, 100, 160, 1.5, 'asvm', False, 'cifar100'), (400, 100, 96, 1.5, 'asv', False, 'cifar100'),
            (400, 100, 96, 1.5, 'neg_sv', False, 'cifar100'), (300, 10, 48, 4.0, 'asvm', True, 'cifar10'),
            (400, 100, 96, 2.0, 'asvm', True, 'cifar100')]:
        for rep in range(2):
            torch.manual_seed(1000 + n_case)
            np.random.seed(2000 + n_case)
            if skew:
                pcls = np.ones(ncls)
                pcls[:max(1, ncls // 10)] = 30.0
                pcls /= pcls.sum()
                by = rs.choice(ncls, mem, p=pcls)
            else:
                by = rs.randint(0, ncls, mem)
            bx = relu_feats(rs, mem, d) + 0.05 * by[:, None].astype(np.float32) / ncls
            cur_y = rs.randint(0, ncls, 10)
            cur_x = relu_feats(rs, 10, d)
            params = SimpleNamespace(eps_mem_batch=10, k=3, mem_size=mem, aser_type=aser_type, n_smp_cls=n_smp,
                                     data=data, update='ASER', num_tasks=10, buffer_tracker=False)
            tag = 'a%d_' % n_case
            # ---------------- retrieve (aser_retrieve.py:34-92)
            ret = aser_retrieve.ASER_retrieve(params)
            CB.class_index_cache = None
            CB.update_cache(torch.tensor(by), ncls, new_y=torch.tensor(by), ind=torch.arange(mem))
            rec = []
            orig_sample = CB.sample.__func__

            def rec_sample(cls, bxx, byy, n, excl_indices=None, device='cpu'):
                r = orig_sample(cls, bxx, byy, n, excl_indices=excl_indices, device=device)
                rec.append(r[2].numpy().copy())
                return r
            CB.sample = classmethod(rec_sample)
            rx, ry = ret._retrieve_by_knn_sv(None, torch.tensor(bx), torch.tensor(by), torch.tensor(cur_x),
                                             torch.tensor(cur_y), 10)
            out.update({tag + 'bx': bx, tag + 'by': by, tag + 'cur_x': cur_x, tag + 'cur_y': cur_y,
                        tag + 'k': np.int64(3), tag + 'type': np.array(aser_type), tag + 'mem': np.int64(mem),
                        tag + 'ncls': np.int64(ncls), tag + 'n_smp': np.float64(n_smp),
                        tag + 'ret_cand_ind': rec[0],
                        tag + 'ret_coop_ind': rec[1] if len(rec) > 1 else np.zeros(0, np.int64),
                        tag + 'ret_x': rx.numpy(), tag + 'ret_y': ry.numpy()})
            # which candidate positions were returned (rows are unique in this data)
            cand_x = bx[rec[0]]
            pos = [int(np.nonzero((cand_x == r).all(1))[0][0]) for r in rx.numpy()]
            out[tag + 'ret_pos'] = np.array(pos)
            # ---------------- update (aser_update.py:43-112)
            rec.clear()
            rr = {}
            orig_rr = aser_update.random_retrieve

            def rec_rr(buffer, n, excl=None, return_indices=False):
                r = orig_rr(buffer, n, excl, return_indices=True)
                rr['ind'] = r[2].numpy().copy()
                return r
            aser_update.random_retrieve = rec_rr
            thr = {}
            orig_min = aser_update.add_minority_class_input

            def rec_min(cx, cy, mem_size, num_class):
                st = torch.get_rng_state()
                thr['t'] = torch.tensor(1).float().uniform_(0, 1 / num_class).item()
                torch.set_rng_state(st)
                r = orig_min(cx, cy, mem_size, num_class)
                thr['n'] = r[0].shape[0]
                return r
            aser_update.add_minority_class_input = rec_min
            upd = aser_update.ASER_update(params)
            CB.class_index_cache = None
            CB.update_cache(torch.tensor(by), ncls, new_y=torch.tensor(by), ind=torch.arange(mem))
            CB.sample = classmethod(rec_sample)
            buf = SimpleNamespace(buffer_img=torch.tensor(bx).clone(), buffer_label=torch.tensor(by).clone(),
                                  current_index=mem, n_seen_so_far=mem + 10, model=None)
            counts_before = CB.class_num_cache.numpy().copy()
            upd._update_by_knn_sv(None, buf, torch.tensor(cur_x), torch.tensor(cur_y))
            changed = np.nonzero((buf.buffer_img.numpy() != bx).any(1))[0]
            out.update({tag + 'upd_eval_ind': rec[0], tag + 'upd_cand_ind': rr['ind'],
                        tag + 'upd_threshold': np.float64(thr['t']), tag + 'upd_n_minority': np.int64(thr['n']),
                        tag + 'upd_counts_before': counts_before,
                        tag + 'upd_changed_slots': changed,
                        tag + 'upd_new_labels': buf.buffer_label.numpy()[changed],
                        tag + 'upd_new_rows': buf.buffer_img.numpy()[changed]})
            CB.sample = classmethod(orig_sample)
            aser_update.random_retrieve = orig_rr
            aser_update.add_minority_class_input = orig_min
            n_case += 1
    out['n_cases'] = np.int64(n_case)
    aser_utils.deep_features = orig
    np.savez_compressed(os.path.join(HERE, 'aser.npz'), **out)


# ----------------------------------------------------------------------------- reservoir
def gen_reservoir():
    """Reference Reservoir_update on a tiny buffer with the uniform draws recorded
    (reservoir_update.py:8-60)."""
    out = {}
    torch.manual_seed(4)
    mem, steps = 37, 30
    params = SimpleNamespace(buffer_tracker=False)
    buf = SimpleNamespace(buffer_img=torch.zeros(mem, 5), buffer_label=torch.zeros(mem, dtype=torch.long),
                          current_index=0, n_seen_so_far=0, params=params)
    upd = reservoir_update.Reservoir_update(params)
    xs, ys, draws, rets = [], [], [], []
    for s in range(steps):
        x = torch.randn(10, 5)
        y = torch.randint(0, 9, (10,))
        place_left = max(0, mem - buf.current_index)
        st = torch.get_rng_state()
        n_after = buf.n_seen_so_far + min(place_left, 10)
        n_draw = 10 - place_left if place_left < 10 else 0
        d = torch.FloatTensor(max(n_draw, 0)).uniform_(0, n_after).long() if n_draw > 0 else torch.zeros(0).long()
        torch.set_rng_state(st)
        r = upd.update(buf, x, y)
        xs.append(x.numpy()); ys.append(y.numpy())
        draws.append(np.pad(d.numpy(), (0, 10 - len(d)), constant_values=-1))
        rets.append(np.pad(np.array(r, dtype=np.int64), (0, 10 - len(r)), constant_values=-1))
    out.update(x=np.stack(xs), y=np.stack(ys), draws=np.stack(draws), rets=np.stack(rets),
               final_img=buf.buffer_img.numpy(), final_label=buf.buffer_label.numpy(),
               n_seen=np.int64(buf.n_seen_so_far), mem=np.int64(mem))
    np.savez_compressed(os.path.join(HERE, 'reservoir.npz'), **out)



# ----------------------------------------------------------------------------- whole replay steps
def gen_steps():
    """Run the reference AGENTS (agents/exp_replay.py, agents/scr.py) for a few minibatches on a tiny
    synthetic task and record every batch, every random choice and the resulting state, so that
    oracle/replay_step.py can be replayed decision by decision."""
    from utils.name_match import agents
    from utils.setup_elements import setup_opt
    from utils.buffer import random_retrieve as rr_mod
    from utils.buffer import buffer_utils as bu
    out = {}
    CB = buffer_utils.ClassBalancedRandomSampling
    cfgs = [('er', 'ER', 'random', 'random', 'cifar10', 10), ('mir', 'ER', 'MIR', 'random', 'cifar10', 10),
            ('aser', 'ER', 'ASER', 'ASER', 'cifar10', 10), ('scr', 'SCR', 'random', 'random', 'cifar100', 20)]
    for tag, agent_name, retrieve, update, data, eps in cfgs:
        seed = {'er': 1, 'mir': 2, 'aser': 3, 'scr': 4}[tag]
        np.random.seed(seed); torch.manual_seed(seed)
        ncls = 10 if data == 'cifar10' else 100
        mem = 40
        params = SimpleNamespace(
            data=data, cuda=False, epoch=1, batch=10, verbose=False, mem_size=mem, eps_mem_batch=eps, mem_iters=1,
            update=update, retrieve=retrieve, agent=agent_name, k=3, aser_type='asvm', n_smp_cls=1.5, num_tasks=5,
            buffer_tracker=False, optimizer='SGD', learning_rate=0.01, weight_decay=0, temp=0.07, head='mlp',
            subsample=20, error_analysis=False,
            trick={'labels_trick': False, 'kd_trick': False, 'separated_softmax': False, 'review_trick': False,
                   'ncm_trick': False, 'kd_trick_star': False})
        spec = oresnet.Spec(32, 20, ncls, head='mlp' if agent_name == 'SCR' else None)
        model = setup_architecture(params)
        p0, bn0 = oresnet.seeded_state(spec, 100 + seed)
        sd = dict(p0); sd.update(bn0)
        model.load_state_dict(sd, strict=True)
        opt = setup_opt('SGD', model, 0.01, 0)     # lr 0.1 on random pixels is chaotic: 1e-7 -> 1e-1 in 6 steps
        agent = agents[agent_name](model, opt, params)
        rs = np.random.RandomState(50 + seed)
        n_steps = 7
        x_u8 = rs.randint(0, 256, (10 * n_steps, 32, 32, 3)).astype(np.uint8)
        y = rs.randint(0, 4, 10 * n_steps).astype(np.int64)     # four classes: matches exist among neighbours
        rec = {'bx': [], 'by': [], 'ret_idx': [], 'draws': [], 'cbrs': [], 'upd_cand': [], 'thr': [], 'mir_idx': []}
        # hooks -------------------------------------------------------------
        orig_update = agent.buffer.update
        def hook_update(x, y_, **kw):
            rec['bx'].append((x.numpy() * 255).round().astype(np.uint8)); rec['by'].append(y_.numpy().copy())
            place_left = max(0, mem - agent.buffer.current_index)
            n_draw = x.shape[0] - place_left if place_left < x.shape[0] else 0
            if update == 'random':
                st = torch.get_rng_state()
                n_after = agent.buffer.n_seen_so_far + min(place_left, x.shape[0])
                d = torch.FloatTensor(n_draw).uniform_(0, n_after).long().numpy() if n_draw > 0 else np.zeros(0, np.int64)
                torch.set_rng_state(st)
                rec['draws'].append(np.pad(d, (0, 10 - len(d)), constant_values=-1))
            return orig_update(x, y_, **kw)
        agent.buffer.update = hook_update
        orig_rr = bu.random_retrieve
        def hook_rr(buffer, n, excl=None, return_indices=False):
            r = orig_rr(buffer, n, excl, return_indices=True)
            rec['last_rr'] = r[2].numpy().copy()
            return r if return_indices else r[:2]
        rr_mod.random_retrieve = lambda buffer, n, *a, **k: _rec_ret(hook_rr(buffer, n, *a, **k), rec, eps)
        def _rec_ret(r, rec_, eps_):
            idx = rec_['last_rr']
            rec_['ret_idx'].append(np.pad(idx, (0, eps_ - len(idx)), constant_values=-1))
            return r
        mir_retrieve.random_retrieve = lambda buffer, n, *a, **k: _rec_mir(hook_rr(buffer, n, *a, **k), rec)
        def _rec_mir(r, rec_):
            idx = rec_['last_rr']
            rec_['mir_idx'].append(np.pad(idx, (0, 20 - len(idx)), constant_values=-1))
            return r
        aser_retrieve.random_retrieve = lambda buffer, n, *a, **k: _rec_ret(hook_rr(buffer, n, *a, **k), rec, eps)
        def hook_upd_rr(buffer, n, excl=None, return_indices=False):
            r = orig_rr(buffer, n, excl, return_indices=True)
            rec['upd_cand'].append(r[2].numpy().copy())
            return r
        aser_update.random_retrieve = hook_upd_rr
        orig_sample = CB.sample.__func__
        def rec_sample(cls, bxx, byy, n, excl_indices=None, device='cpu'):
            r = orig_sample(cls, bxx, byy, n, excl_indices=excl_indices, device=device)
            rec['cbrs'].append(r[2].numpy().copy())
            return r
        CB.sample = classmethod(rec_sample)
        orig_min = aser_update.add_minority_class_input
        def rec_min(cx, cy, mem_size, num_class):
            st = torch.get_rng_state()
            rec['thr'].append(torch.tensor(1).float().uniform_(0, 1 / num_class).item())
            torch.set_rng_state(st)
            return orig_min(cx, cy, mem_size, num_class)
        aser_update.add_minority_class_input = rec_min
        # run ---------------------------------------------------------------
        agent.train_learner(x_u8, y)
        # unhook
        rr_mod.random_retrieve = orig_rr; mir_retrieve.random_retrieve = orig_rr
        aser_retrieve.random_retrieve = orig_rr; aser_update.random_retrieve = orig_rr
        CB.sample = classmethod(orig_sample); aser_update.add_minority_class_input = orig_min
        out[tag + '_bx'] = np.stack(rec['bx']); out[tag + '_by'] = np.stack(rec['by'])
        if rec['ret_idx']:
            out[tag + '_ret_idx'] = np.stack(rec['ret_idx'])
        if rec['draws']:
            out[tag + '_draws'] = np.stack(rec['draws'])
        if rec['mir_idx']:
            out[tag + '_mir_idx'] = np.stack(rec['mir_idx'])
        for j, c in enumerate(rec['cbrs']):
            out['%s_cbrs%d' % (tag, j)] = c
        out[tag + '_n_cbrs'] = np.int64(len(rec['cbrs']))
        for j, c in enumerate(rec['upd_cand']):
            out['%s_updcand%d' % (tag, j)] = c
        out[tag + '_n_updcand'] = np.int64(len(rec['upd_cand']))
        out[tag + '_thr'] = np.array(rec['thr'], dtype=np.float64)
        out[tag + '_final_labels'] = agent.buffer.buffer_label.numpy().copy()
        out[tag + '_final_img_sum'] = agent.buffer.buffer_img.numpy().reshape(mem, -1).sum(1)
        out[tag + '_n_seen'] = np.int64(agent.buffer.n_seen_so_far)
        names, norms = [], []
        for name, prm in model.named_parameters():
            names.append(name); norms.append(float(prm.detach().double().norm()))
        out[tag + '_param_names'] = np.array(names); out[tag + '_param_norms'] = np.array(norms)
        out[tag + '_rm_bn1'] = [v for k_, v in model.state_dict().items() if k_.endswith('bn1.running_mean')][0].numpy().copy()
        out[tag + '_lin_w'] = [prm for n_, prm in model.named_parameters() if n_.endswith('linear.weight') or n_ == 'head.2.weight'][-1].detach().numpy().copy()
    np.savez_compressed(os.path.join(HERE, 'steps.npz'), **out)

# ----------------------------------------------------------------------------- GSS-greedy
def gen_gss():
    """Reference GSSGreedyUpdate (gss_greedy_update.py:7-124) driven through the reference Buffer on a seeded
    Reduced_ResNet18 (CPU): three fill batches, then full-memory updates with unseen classes (batch_sim < 0: the
    replacement lottery) and seen classes.  The inputs come from a numpy stream the test regenerates; the file
    records the torch seed before every update, the scores, labels and the source of every slot afterwards."""
    from utils import name_match  # noqa: F401  (resolves the reference's circular import first)
    from utils.buffer.buffer import Buffer
    from utils.buffer import gss_greedy_update
    out = {}
    spec = oresnet.Spec(32, 20, 10)
    model, p, bn = _ref_model('cifar10', 'ER', None, spec, 77)
    with torch.no_grad():          # a small classifier: softmax outputs near uniform, so the sign of a gradient cosine
        model.linear.weight.mul_(0.02)   # follows the label overlap (the test applies the same two lines to the oracle state)
        model.linear.bias.zero_()
    mem, batch, n_upd = 30, 10, 8
    params = SimpleNamespace(data='cifar10', cuda=False, mem_size=mem, update='GSS', retrieve='random',
                             gss_mem_strength=10, gss_batch_size=10, buffer_tracker=False, eps_mem_batch=10)
    buf = Buffer(model, params)
    upd = buf.update_method
    assert isinstance(upd, gss_greedy_update.GSSGreedyUpdate)
    sims = []
    orig = upd.get_batch_sim

    def hook(*a, **k):
        s, m = orig(*a, **k)
        sims.append(float(s))
        return s, m
    upd.get_batch_sim = hook
    rs = np.random.RandomState(770)
    # slot -> (update number, position in that batch) of the sample it holds: the memory contents without the pixels
    src = np.full((mem, 2), -1, dtype=np.int64)
    labels, scores, srcs, batch_sim, ys = [], [], [], [], []
    for u in range(n_upd):
        x = torch.from_numpy(rs.rand(batch, 3, 32, 32).astype(np.float32))
        lab = rs.randint(0, 3, batch)
        y = torch.from_numpy(lab.astype(np.int64))
        if u >= 3 and u % 2 == 1:
            lab = lab + 3 + 3 * ((u // 2) % 2)   # classes the memory does not hold: with near-uniform softmax outputs the batch gradient
            y = torch.from_numpy(lab.astype(np.int64))   # points away from the memory gradients (batch_sim < 0)
        torch.manual_seed(1000 + u)
        before_img = buf.buffer_img.clone()
        n_sims = len(sims)
        buf.update(x, y)
        changed = (buf.buffer_img != before_img).flatten(1).any(1).nonzero().flatten().tolist()
        for sl in changed:
            pos = [i for i in range(batch) if torch.equal(buf.buffer_img[sl], x[i])]
            assert len(pos) == 1
            src[sl] = (u, pos[0])
        ys.append(lab.astype(np.int64))
        labels.append(buf.buffer_label.numpy().copy())
        scores.append(upd.buffer_score.numpy().copy())
        srcs.append(src.copy())
        batch_sim.append(sims[-1] if len(sims) > n_sims else np.nan)
    assert model.training                                   # the rule leaves the model in train mode (:64)
    print('gss batch_sim', batch_sim)
    assert any(b < 0 for b in batch_sim if b == b) and any(b >= 0 for b in batch_sim if b == b)
    out.update(y=np.stack(ys), labels=np.stack(labels), scores=np.stack(scores), src=np.stack(srcs),
               batch_sim=np.array(batch_sim), mem=np.int64(mem), batch=np.int64(batch), model_seed=np.int64(77),
               data_seed=np.int64(770), torch_seed0=np.int64(1000))
    np.savez_compressed(os.path.join(HERE, 'gss.npz'), **out)


# ----------------------------------------------------------------------------- parity-mode random streams
def _digest(t):
    import hashlib
    return np.frombuffer(hashlib.sha256(t.contiguous().numpy().tobytes()).digest(), np.uint8)


def gen_parity():
    """The reference's host-side random decisions on the inputs of tests/test_parity_mode.py: class-balanced
    sampler draws (buffer_utils.py:60-140), reservoir updates (reservoir_update.py:8-60) and the stream
    DataLoader order (continuum/data_utils.py).  Image tensors are recorded as sha256 digests of their bytes."""
    from continuum.data_utils import dataset_transform
    from utils.setup_elements import transforms_match
    from torch.utils import data
    Ref = buffer_utils.ClassBalancedRandomSampling
    out = {}

    def sample(n, excl, seed):
        torch.manual_seed(seed)
        return Ref.sample(buf_x, buf_y, n, excl_indices=None if excl is None else set(excl), device='cpu')[2].numpy()
    for n_cls, mem in [(10, 200), (100, 1000)]:
        Ref.class_index_cache = Ref.class_num_cache = None
        tag = 'inc%d' % n_cls
        rs = np.random.RandomState(3)
        labels = rs.randint(0, n_cls, mem).astype(np.int64)
        buf_y = torch.zeros(mem, dtype=torch.int64)
        buf_x = torch.zeros(mem, 1)
        for s in range(0, mem, 10):
            ny = torch.from_numpy(labels[s:s + 10])
            Ref.update_cache(buf_y, n_cls, new_y=ny, ind=torch.arange(s, s + 10), device='cpu')
            buf_y[s:s + 10] = ny
        out[tag + '_keys'] = np.array(list(Ref.class_index_cache.keys()))
        for step in range(25):
            r1 = sample(1, None, 100 + step)
            r2 = sample(2, r1.tolist(), 200 + step)
            out['%s_r1_%d' % (tag, step)], out['%s_r2_%d' % (tag, step)] = r1, r2
            slots = rs.choice(mem, 4, replace=False)
            ny = rs.randint(0, n_cls, 4).astype(np.int64)
            Ref.update_cache(buf_y, n_cls, new_y=torch.from_numpy(ny), ind=torch.from_numpy(slots), device='cpu')
            buf_y[torch.from_numpy(slots)] = torch.from_numpy(ny)
            out['%s_num_%d' % (tag, step)] = Ref.class_num_cache.numpy().copy()
    Ref.class_index_cache = Ref.class_num_cache = None
    rs = np.random.RandomState(4)
    buf_y = torch.from_numpy(rs.randint(0, 20, 300).astype(np.int64))
    buf_x = torch.zeros(300, 1)
    Ref.update_cache(buf_y, 20)
    out['rebuild_keys'] = np.array(list(Ref.class_index_cache.keys()))
    for step in range(10):
        r = sample(3, None, step)
        out['rebuild_r_%d' % step], out['rebuild_r2_%d' % step] = r, sample(3, r.tolist(), 50 + step)
    Ref.class_index_cache = Ref.class_num_cache = None

    params = SimpleNamespace(data='cifar10', cuda=False, mem_size=50, update='random', retrieve='random',
                             eps_mem_batch=10, buffer_tracker=False)
    buf = SimpleNamespace(buffer_img=torch.zeros(50, 3, 32, 32), buffer_label=torch.zeros(50, dtype=torch.int64),
                          current_index=0, n_seen_so_far=0, params=params)
    upd = reservoir_update.Reservoir_update(params)
    rs = np.random.RandomState(0)
    labels, imgs, n_seen = [], [], []
    for step in range(30):
        x = torch.from_numpy(rs.rand(10, 3, 32, 32).astype(np.float32))
        y = torch.from_numpy(rs.randint(0, 10, 10).astype(np.int64))
        torch.manual_seed(step)
        out['reservoir_ret_%d' % step] = np.array(list(upd.update(buf, x, y)), dtype=np.int64)
        labels.append(buf.buffer_label.numpy().copy()); imgs.append(_digest(buf.buffer_img)); n_seen.append(buf.n_seen_so_far)
    out.update(reservoir_label=np.stack(labels), reservoir_img_sha256=np.stack(imgs), reservoir_n_seen=np.array(n_seen))

    rs = np.random.RandomState(1)
    x = rs.randint(0, 256, (57, 32, 32, 3)).astype(np.uint8)
    y = rs.randint(0, 10, 57).astype(np.int64)
    torch.manual_seed(11)
    loader = data.DataLoader(dataset_transform(x, y, transform=transforms_match['cifar10']), batch_size=10,
                             shuffle=True, num_workers=0, drop_last=True)
    batches = [(bx.clone(), by.clone()) for bx, by in loader]
    out.update(stream_label=np.stack([by.numpy() for _, by in batches]),
               stream_img_sha256=np.stack([_digest(bx) for bx, _ in batches]),
               stream_img_shape=np.array(batches[0][0].shape), stream_rand_after=torch.rand(1).numpy())
    np.savez_compressed(os.path.join(HERE, 'parity.npz'), **out)


def gen_registry():
    """The registry keys of utils/name_match.py and the module-level names the drop-in switch rebinds."""
    import agents.base as base
    import experiment.run as run
    import utils.name_match as nm
    out = {t: np.array(sorted(getattr(nm, t))) for t in ('agents', 'retrieve_methods', 'update_methods')}
    out['run_agents_is_name_match_agents'] = np.bool_(run.agents is nm.agents)
    out['patched'] = np.array(['agents.base:SupConLoss', 'utils.buffer.aser_retrieve:compute_knn_sv',
                               'utils.buffer.aser_update:compute_knn_sv'])
    assert all(hasattr(m, 'compute_knn_sv') for m in (aser_retrieve, aser_update)) and hasattr(base, 'SupConLoss')
    np.savez_compressed(os.path.join(HERE, 'registry.npz'), **out)


if __name__ == '__main__':
    only = sys.argv[2:]            # e.g. `make_golden.py /root/reference gss`: regenerate one file
    for name, fn in (('knn_sv', gen_knn_sv), ('supcon', gen_supcon), ('resnet', gen_resnet), ('aser', gen_aser),
                     ('reservoir', gen_reservoir), ('steps', gen_steps), ('gss', gen_gss), ('parity', gen_parity),
                     ('registry', gen_registry)):
        if not only or name in only:
            fn()
    for f in sorted(os.listdir(HERE)):
        if f.endswith('.npz'):
            print(f, os.path.getsize(os.path.join(HERE, f)))
