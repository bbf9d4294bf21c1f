"""CPU: what `bench.py --dump-outputs` writes for a training step -- the losses and the updated weights under the reference's
tensor names, with encoder.0.weight reduced to a sample at seeded flat positions.  No kernel is launched."""
from types import SimpleNamespace

import numpy as np
import torch


def test_step_outputs_are_the_weights_under_reference_names():
    import bench
    from hvae_b200.model import HybridVAE
    from hvae_b200.synth import make_item_embeddings
    torch.manual_seed(0)
    m = HybridVAE(300, make_item_embeddings(300, 32, 0), 16, [48], 0.5, 0.2, precision="fp32")
    x = SimpleNamespace(model=m, trainer=SimpleNamespace(last_losses=lambda: (3.0, 2.5, 0.5)))
    sd = m.state_dict()
    for n in (1000, 300 * 48):                 # sampled W1, then W1 whole (no larger than the sample)
        out = bench.step_outputs(x, w1_sample=n)
        assert all(a.dtype == np.float32 for a in out.values())
        assert np.array_equal(out.pop("losses"), np.float32([3.0, 2.5, 0.5]))
        w1 = "encoder.0.weight.sample" if n < 300 * 48 else "encoder.0.weight"
        assert set(out) == (set(sd) - {"item_embeddings", "encoder.0.weight"}) | {w1}
        for k, a in out.items():
            if k == "encoder.0.weight.sample":
                pos = np.sort(np.random.default_rng(0).integers(0, 300 * 48, n))
                assert np.array_equal(a, sd["encoder.0.weight"].numpy().reshape(-1)[pos])
            else:
                assert np.array_equal(a, sd[k].numpy()), k
