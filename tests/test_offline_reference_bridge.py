"""Reference Trace objects -> TraceColumns.from_reference_traces -> trace file -> OfflineDataset.batch must describe the
same minibatch as the reference's own Batch: the oracle loss on the re-read arrays equals the UNMODIFIED reference's
_loss on the traces.  The traces, the reference Batch's grouping, the network and the loss are stored golden data
(tests/golden/make_bridge_golden.py); the traces are rebuilt here as objects with the attributes the bridge reads."""
import json
import os
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _golden():
    z = np.load(os.path.join(ROOT, 'tests', 'golden', 'bridge_golden.npz'))
    params = {k[len('param.'):]: torch.from_numpy(z[k]) for k in z.files if k.startswith('param.')}
    return json.loads(str(z['meta'])), params


def _distribution(name, num_categories, prior):
    fields = {'Normal': ('mean', 'stddev'), 'Uniform': ('low', 'high')}.get(name, ())
    attrs = dict(zip(fields, prior))
    if name == 'Categorical':
        attrs['num_categories'] = num_categories
    return type(name, (), attrs)()


def _trace(rec):
    ctrl = [SimpleNamespace(address=v['address'], value=torch.tensor(v['value']),
                            distribution=_distribution(v['distribution'], v['num_categories'], v['prior']))
            for v in rec['controlled']]
    named = {nm: SimpleNamespace(value=torch.tensor(val)) for nm, val in rec['observed'].items()}
    return SimpleNamespace(variables_controlled=ctrl, named_variables=named)


def test_reference_traces_survive_the_columnar_store(tmp_path):
    from oracle import network as onet
    from pyprob_b200 import offline

    meta, params = _golden()
    traces = [_trace(rec) for rec in meta['traces']]
    names = list(meta['observe_embeddings'])
    cols = offline.TraceColumns.from_reference_traces(traces, names)
    offline.save_columns(str(tmp_path), cols)
    data = offline.OfflineDataset(str(tmp_path))
    assert len(data) == 40 and data.num_trace_types == len(meta['sub_batch_sizes'])
    arr = data.batch(list(range(40)))
    # same grouping as the reference Batch: sub-batches in order of first appearance, same sizes
    assert [sb['values'].shape[1] for sb in arr.subs] == meta['sub_batch_sizes']
    assert [sb['addresses'] for sb in arr.subs] == meta['sub_batch_addresses']
    tsubs = [{k: (torch.from_numpy(np.ascontiguousarray(v)) if isinstance(v, np.ndarray) else v) for k, v in sb.items()}
             for sb in arr.subs]
    got, _ = onet.loss(params, tsubs, names, [1, 1], meta['mixture_components'])
    ref_loss = meta['loss']
    assert abs(float(got) - ref_loss) <= 2e-6 * abs(ref_loss)
