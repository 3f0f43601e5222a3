"""Drive the UNMODIFIED reference (compiled into oracle/_ref by oracle/fetch_ref.py) the way
experiment/run.py:38-49 does: setup_architecture -> maybe_cuda -> setup_opt -> agents[...](model, opt,
params) -> train_learner(uint8 NHWC array, labels).  Import recipe = SURVEY.md Appendix B: three stub
modules that are not on the arithmetic path (matplotlib, skimage, kornia -- none is installed here and
there is no network).  The kornia stub is the identity: the reference arm therefore does LESS work than
the real reference (no augmentation), which only makes the reported speed-up conservative.

    python baseline/ref_harness.py --device cuda|cpu --steps K --warmup W [--threads T]

prints one JSON line with ms per ER+ASER step, ms per SCR step and stream images/s for the pair.
The device is chosen the way the reference chooses it (torch.cuda.is_available(), utils/utils.py:14,
buffer.py:22, aser_retrieve.py:12): --device cpu hides the GPUs with CUDA_VISIBLE_DEVICES="" before
torch is imported.
"""
import argparse
import json
import os
import sys
import time
import types
from types import SimpleNamespace

HERE = os.path.dirname(os.path.abspath(__file__))
MEM_SIZE, BATCH, NUM_CLASSES = 5000, 10, 100
TRICK = {'labels_trick': False, 'kd_trick': False, 'separated_softmax': False, 'review_trick': False,
         'ncm_trick': False, 'kd_trick_star': False}


def locate():
    p = os.path.join(os.path.dirname(HERE), 'oracle', '_ref')
    return p if os.path.exists(os.path.join(p, 'utils', 'name_match.pyc')) else None


def import_reference(path=None):
    """Put the reference tree first on sys.path and register the three stub modules."""
    import torch.nn as nn
    path = path or locate()
    if path is None:
        raise RuntimeError('no reference build: run `python oracle/fetch_ref.py <reference checkout>`')
    if path not in sys.path:
        sys.path.insert(0, path)
    if 'kornia.augmentation' not in sys.modules:
        for name in ['matplotlib', 'matplotlib.pyplot', 'skimage', 'skimage.filters', 'kornia', 'kornia.augmentation']:
            sys.modules.setdefault(name, types.ModuleType(name))
        sys.modules['skimage.filters'].gaussian = lambda *a, **k: None

        class Identity(nn.Module):
            def __init__(self, *a, **k):
                super().__init__()

            def forward(self, x):
                return x
        for n in ['RandomResizedCrop', 'RandomHorizontalFlip', 'ColorJitter', 'RandomGrayscale']:
            setattr(sys.modules['kornia.augmentation'], n, Identity)
    import warnings
    warnings.filterwarnings('ignore')
    _torch2_compat()
    return path


def _torch2_compat():
    """The reference pins torch 1.7.1 (requirements.txt:2).  Under torch >= 2 two statements of its GPU path
    raise (the second is handled further down): aser_update.py:102 indexes the CPU index tensor that random_retrieve returns
    (buffer_utils.py:17, torch.from_numpy) with a CUDA tensor.  The shim wraps the `random_retrieve` name
    bound in utils.buffer.aser_update so that the returned indices live on the buffer's device -- same
    values, same numpy draw, no file of the reference is edited.  It is a no-op on the CPU."""
    import torch
    from utils.buffer import aser_update
    if getattr(aser_update.random_retrieve, '_b200ocl_compat', False):
        return
    orig = aser_update.random_retrieve

    def random_retrieve(buffer, num_retrieve, excl_indices=None, return_indices=False):
        out = orig(buffer, num_retrieve, excl_indices, return_indices)
        if return_indices:
            x, y, ind = out
            return x, y, ind.to(buffer.buffer_img.device)
        return out
    random_retrieve._b200ocl_compat = True
    aser_update.random_retrieve = random_retrieve
    # A second statement of the same kind: gss_greedy_update.py:43-46 index CPU tensors (`index`, `added_indx`) with
    # the CUDA mask that torch.multinomial returned for CUDA probabilities (:38).  The name `torch` bound in that
    # module becomes a proxy whose multinomial hands its result back on the CPU -- same call, same generator, same
    # values; everything else is torch itself.
    from utils.buffer import gss_greedy_update

    class _TorchProxy(object):
        def __getattr__(self, name):
            return getattr(torch, name)

        @staticmethod
        def multinomial(*a, **k):
            return torch.multinomial(*a, **k).cpu()
    if not isinstance(gss_greedy_update.torch, _TorchProxy) and type(gss_greedy_update.torch).__name__ != '_TorchProxy':
        gss_greedy_update.torch = _TorchProxy()


def make_params(kind, **over):
    """Exactly the fields the replay path reads (SURVEY.md section 5.6 / Appendix B)."""
    base = dict(data='cifar100', cuda=True, epoch=1, batch=BATCH, verbose=False, mem_size=MEM_SIZE, mem_iters=1,
                k=3, aser_type='asvm', n_smp_cls=1.5, num_tasks=10, buffer_tracker=False, optimizer='SGD',
                learning_rate=0.1, weight_decay=0, temp=0.07, head='mlp', subsample=50, error_analysis=False,
                trick=dict(TRICK), test_batch=128, num_workers=0)
    if kind == 'aser':
        base.update(agent='ER', retrieve='ASER', update='ASER', eps_mem_batch=10)
    elif kind == 'scr':
        base.update(agent='SCR', retrieve='random', update='random', eps_mem_batch=100)
    elif kind == 'er':
        base.update(agent='ER', retrieve='random', update='random', eps_mem_batch=10)
    elif kind == 'mir':
        base.update(agent='ER', retrieve='MIR', update='random', eps_mem_batch=10)
    elif kind == 'agem':
        base.update(agent='AGEM', retrieve='random', update='random', eps_mem_batch=10)
    elif kind == 'gss':
        base.update(agent='ER', retrieve='random', update='GSS', eps_mem_batch=10, gss_mem_strength=10, gss_batch_size=10)
    elif kind == 'scr_aser':
        base.update(agent='SCR', retrieve='ASER', update='ASER', eps_mem_batch=100)
    else:
        raise ValueError(kind)
    base.update(over)
    return SimpleNamespace(**base)


def build_agent(params):
    """experiment/run.py:38-41."""
    from utils.name_match import agents
    from utils.setup_elements import setup_architecture, setup_opt
    from utils.utils import maybe_cuda
    model = setup_architecture(params)
    model = maybe_cuda(model, params.cuda)
    opt = setup_opt(params.optimizer, model, params.learning_rate, params.weight_decay)
    return agents[params.agent](model, opt, params)


def synthetic_task(rs, n, hw=32, num_classes=NUM_CLASSES):
    import numpy as np
    return rs.randint(0, 256, (n, hw, hw, 3)).astype(np.uint8), rs.randint(0, num_classes, n).astype(np.int64)


def prefill(agent, rs, hw=32, num_classes=NUM_CLASSES):
    """Fill the memory through the agent's own buffer.update (fill phase of either update plugin)."""
    import numpy as np
    import torch
    mem = agent.buffer.buffer_img.shape[0]
    x = torch.from_numpy(rs.rand(mem, 3, hw, hw).astype(np.float32))
    y = torch.from_numpy(rs.randint(0, num_classes, mem).astype(np.int64))
    dev = agent.buffer.buffer_img.device
    agent.buffer.update(x.to(dev), y.to(dev))
    assert agent.buffer.current_index == mem


def timed_train(agent, x, y, cuda):
    import torch
    if cuda:
        torch.cuda.synchronize()
    t0 = time.perf_counter()
    agent.train_learner(x, y)
    if cuda:
        torch.cuda.synchronize()
    return time.perf_counter() - t0


def run(device, steps, warmup, threads=None, kinds=('aser', 'scr'), hw=32, data='cifar100', mem=MEM_SIZE):
    import numpy as np
    import torch
    import random
    if threads:
        torch.set_num_threads(threads)
    cuda = device == 'cuda'
    if cuda:
        assert torch.cuda.is_available()
        torch.backends.cudnn.deterministic = True      # general_main.py:15-18
        torch.backends.cudnn.benchmark = False
    else:
        assert not torch.cuda.is_available(), 'hide the GPUs (CUDA_VISIBLE_DEVICES="") for the CPU arm'
    import_reference()
    np.random.seed(0); random.seed(0); torch.manual_seed(0)
    if cuda:
        torch.cuda.manual_seed(0)
    out = {'device': device, 'steps': steps, 'warmup': warmup, 'threads': torch.get_num_threads(),
           'torch': torch.__version__, 'reference': locate()}
    total = 0.0
    import contextlib
    for kind in kinds:
        rs = np.random.RandomState(31 if kind == 'aser' else 32)
        with contextlib.redirect_stdout(sys.stderr):
            agent = build_agent(make_params(kind, data=data, mem_size=mem))
            prefill(agent, rs, hw)
            xw, yw = synthetic_task(rs, BATCH * max(warmup, 1), hw)
            timed_train(agent, xw, yw, cuda)               # also pushes n_seen_so_far past mem_size
            xt, yt = synthetic_task(rs, BATCH * steps, hw)
            dt = timed_train(agent, xt, yt, cuda)
        out[kind + '_ms_per_step'] = 1e3 * dt / steps
        total += dt
    out['ms_per_step_pair'] = 1e3 * total / steps
    out['stream_images_per_s'] = len(kinds) * BATCH * steps / total
    out['seconds'] = total
    return out


if __name__ == '__main__':
    ap = argparse.ArgumentParser()
    ap.add_argument('--device', default='cuda', choices=['cuda', 'cpu'])
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--threads', type=int, default=0)
    ap.add_argument('--kinds', default='aser,scr')
    ap.add_argument('--data', default='cifar100')
    ap.add_argument('--mem', type=int, default=MEM_SIZE)
    a = ap.parse_args()
    if a.device == 'cpu':
        os.environ['CUDA_VISIBLE_DEVICES'] = ''
    hw = 84 if a.data == 'mini_imagenet' else 32
    print(json.dumps(run(a.device, a.steps, a.warmup, a.threads or None, tuple(a.kinds.split(',')), hw, a.data, a.mem)))
