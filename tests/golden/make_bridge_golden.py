"""Golden data for tests/test_offline_reference_bridge.py, from the UNMODIFIED reference.

    python tests/golden/make_bridge_golden.py <pyprob checkout>   # writes tests/golden/bridge_golden.npz

Needs a checkout of the reference pyprob and the import stubs of oracle/ref_stubs.  A branching model is traced by
the reference's OnlineDataset; its network is grown on those traces (_polymorph) and scores them with its own _loss.
Stored: what TraceColumns.from_reference_traces reads of each trace (address, distribution name, categories, value,
the Normal / Uniform prior parameters, the observed values), the grouping of the reference's Batch, the network's
parameters and the loss.
"""
import contextlib
import io
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))

OBSERVE_EMBEDDINGS = {'y0': {'dim': 8, 'depth': 2}, 'y1': {'dim': 4, 'depth': 1}}
NUM_TRACES = 40
MIXTURE_COMPONENTS = 3


def _prior_params(d):
    name = type(d).__name__
    if name == 'Normal':
        return float(d.mean), float(d.stddev)
    if name == 'Uniform':
        return float(d.low), float(d.high)
    return 0.0, 0.0


def main(reference):
    sys.path.insert(0, os.path.join(ROOT, 'oracle', 'ref_stubs'))
    sys.path.insert(1, reference)
    import numpy as np
    import torch
    import pyprob
    from pyprob import InferenceNetwork, Model
    from pyprob.distributions import Categorical, Normal, Poisson, Uniform
    from pyprob.nn.dataset import Batch, OnlineDataset

    class Branching(Model):
        def forward(self):
            u = pyprob.sample(Uniform(-1, 2))
            k = pyprob.sample(Categorical([0.2, 0.3, 0.5]))
            if int(k) == 0:
                z = pyprob.sample(Normal(u, 0.5))
            else:
                z = pyprob.sample(Poisson(3.0)) * 0.25
            mu = pyprob.sample(Normal(z * 0.1, 1))
            pyprob.observe(Normal(mu, 0.3), name='y0')
            pyprob.observe(Normal(u, 0.7), name='y1')
            return mu

    pyprob.set_verbosity(0)
    pyprob.seed(5)
    model = Branching()
    with contextlib.redirect_stdout(io.StringIO()):
        model.learn_inference_network(num_traces=48, batch_size=24, inference_network=InferenceNetwork.LSTM,
                                      observe_embeddings=OBSERVE_EMBEDDINGS, lstm_dim=16,
                                      proposal_mixture_components=MIXTURE_COMPONENTS)
    net = model._inference_network
    ds = OnlineDataset(model)
    traces = [ds[i] for i in range(NUM_TRACES)]
    batch = Batch(traces)
    with contextlib.redirect_stdout(io.StringIO()):
        net._polymorph(batch)
    with torch.no_grad():
        ok, loss = net._loss(batch)
    assert ok
    names = list(OBSERVE_EMBEDDINGS)
    meta = {
        'observe_embeddings': OBSERVE_EMBEDDINGS,
        'mixture_components': MIXTURE_COMPONENTS,
        'loss': float(loss),
        'traces': [{
            'controlled': [{'address': v.address, 'distribution': type(v.distribution).__name__,
                            'num_categories': int(getattr(v.distribution, 'num_categories', 0)),
                            'value': float(v.value), 'prior': _prior_params(v.distribution)}
                           for v in tr.variables_controlled],
            'observed': {nm: np.asarray(tr.named_variables[nm].value, np.float64).reshape(-1).tolist() for nm in names},
        } for tr in traces],
        'sub_batch_sizes': [len(sb) for sb in batch.sub_batches],
        'sub_batch_addresses': [[v.address for v in sb[0].variables_controlled] for sb in batch.sub_batches],
    }
    arrays = {'param.' + k: v.detach().cpu().numpy() for k, v in net.state_dict().items()}
    out = os.path.join(HERE, 'bridge_golden.npz')
    np.savez_compressed(out, meta=np.array(json.dumps(meta)), **arrays)
    print('wrote {}: {} traces, {} sub-batches, {} parameter tensors, loss {!r}'.format(
        out, len(traces), len(batch.sub_batches), len(arrays), float(loss)))


if __name__ == '__main__':
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
