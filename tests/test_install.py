"""CPU: the drop-in switch patches the reference's registries in place and restores them.
The reference's modules are stood in for by stubs that carry the registry keys and the module-level names
recorded from it in tests/golden/registry.npz (tests/golden/make_golden.py)."""
import os
import sys
import types

import numpy as np


def _reference_stubs(g):
    """utils.name_match, experiment.run and the modules whose names install() rebinds, as sys.modules entries."""
    mods = {n: types.ModuleType(n) for n in ('utils', 'utils.buffer', 'agents', 'experiment', 'utils.name_match',
                                             'experiment.run', 'agents.base', 'utils.buffer.aser_retrieve',
                                             'utils.buffer.aser_update')}
    nm = mods['utils.name_match']
    for table in ('agents', 'retrieve_methods', 'update_methods'):
        setattr(nm, table, {k: type('Reference%s' % k, (), {}) for k in g[table].tolist()})
    mods['experiment.run'].agents = nm.agents if bool(g['run_agents_is_name_match_agents']) else dict(nm.agents)
    for entry in g['patched'].tolist():
        mod, attr = entry.split(':')
        setattr(mods[mod], attr, type('Reference' + attr, (), {}))
    return mods


def test_install_patches_reference_registries(golden_dir):
    g = np.load(os.path.join(golden_dir, 'registry.npz'), allow_pickle=False)
    stubs = _reference_stubs(g)
    saved = {k: sys.modules[k] for k in stubs if k in sys.modules}
    sys.modules.update(stubs)
    try:
        import utils.name_match as nm
        import agents.base as base
        import utils.buffer.aser_retrieve as ar
        import experiment.run as run
        from b200ocl import registry
        before = (nm.agents['ER'], nm.retrieve_methods['ASER'], nm.update_methods['random'], base.SupConLoss,
                  ar.compute_knn_sv, nm.agents['EWC'])
        registry.install(nm)
        assert nm.agents['ER'] is registry.agents['ER'] and nm.agents['SCR'] is registry.agents['SCR']
        assert run.agents is nm.agents and run.agents['ER'] is registry.agents['ER']     # same dict object (run.py:5)
        assert nm.retrieve_methods['MIR'] is registry.retrieve_methods['MIR']
        assert nm.update_methods['ASER'] is registry.update_methods['ASER']
        assert nm.agents['EWC'] is before[5]                                             # others untouched
        assert base.SupConLoss.__module__.startswith('b200ocl')
        assert ar.compute_knn_sv.__module__.startswith('b200ocl')
        registry.uninstall(nm)
        assert (nm.agents['ER'], nm.retrieve_methods['ASER'], nm.update_methods['random'], base.SupConLoss,
                ar.compute_knn_sv, nm.agents['EWC']) == before
    finally:
        for k in stubs:
            sys.modules.pop(k, None)
        sys.modules.update(saved)


def test_host_sampling_logic():
    import numpy as np
    from b200ocl import memory, update
    rs = np.random.RandomState(0)
    lab = rs.randint(0, 10, 500)
    ex = np.zeros(500, bool)
    ex[rs.choice(500, 100, replace=False)] = True
    idx = memory.class_balanced_indices(lab, 500, 3, ex, rng=rs)
    assert len(set(idx.tolist())) == len(idx) and not ex[idx].any()
    counts = np.bincount(lab[idx], minlength=10)
    assert (counts == 3).all()
    # classes with fewer members than requested contribute what they have
    lab2 = np.array([0, 0, 0, 1, 2, 2])
    idx2 = memory.class_balanced_indices(lab2, 6, 2, None, rng=rs)
    assert sorted(lab2[idx2].tolist()) == [0, 0, 1, 2, 2]
    # reference-identical uniform retrieval stream
    np.random.seed(3)
    a = memory.uniform_indices(100, 10, excl_indices={1, 2, 3})
    np.random.seed(3)
    valid = np.setdiff1d(np.arange(100), np.array([1, 2, 3]))
    b = np.random.choice(valid, 10, replace=False)
    assert np.array_equal(a, b)
    ind_cur, ind_buf = update.aser_update_partition(np.array([3, 0, 5, 1, 2, 4]), 4, np.array([10, 11, 12, 13]))
    assert ind_cur.tolist() == [1] and ind_buf.tolist() == [12]
    assert update.reservoir_plan([5, 50, 5, 7], 40) == ([5, 7], [2, 3])


def test_class_cache_bookkeeping():
    import numpy as np
    from b200ocl.memory import ClassBalancedRandomSampling as CB
    CB.reset()
    lab = np.array([0, 1, 1, 2, 0, 2, 2, 1])
    CB.update_cache(np.zeros(8), 3, new_y=lab, ind=np.arange(8))
    assert CB.class_num_cache.tolist() == [2, 3, 3]
    CB.update_cache(np.zeros(8), 3, new_y=np.array([0, 0]), ind=np.array([1, 6]))      # relabel two slots
    assert CB.class_num_cache.tolist() == [4, 2, 2]
    assert CB.class_index_cache[0] == {0, 1, 4, 6} and 1 not in CB.class_index_cache[1]
    idx = CB.sample_indices(1)
    assert sorted(CB.labels_host[idx].tolist()) == [0, 1, 2]
    idx2 = CB.sample_indices(5, excl_indices=idx)
    assert not set(idx.tolist()) & set(idx2.tolist()) and len(idx2) == 5
    CB.reset()
