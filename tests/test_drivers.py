"""The drop-in constructors start from the reference's tables.

north_star: "nn.Modules with the same constructors and forward() signatures as the reference
classes so the three run_*.py entry points and -model_type dispatch call them unchanged".  With the
same torch seed the package's model classes draw bit-identical initial tables (same generator
consumption as the reference constructors, transE.py:31-46 ...) and leave the generator in the same
state, so a driver that seeds torch sees the same model and the same batches afterwards.  The
reference's tables and the draw after them are stored in ``tests/golden/dropin_init.npz``
(recorded by ``tests/golden/make_golden_live.py``).
"""
import numpy as np
import torch

_IMAP = {i: i for i in range(70)}
_NMAP = {i: ((i * 7) % 40 if i % 3 else -1, i) for i in range(70)}
DROPIN_INIT_CASES = [
    ("transE", (False, 16, 50, 7)), ("transH", (True, 16, 50, 7)), ("transR", (False, 8, 50, 7)),
    ("transUP", (False, 16, 50, 70, 5, True)), ("jTransUP", (False, 16, 50, 70, 40, 5, _IMAP, _NMAP, False, False)),
]


def test_dropin_constructors_start_from_the_reference_tables(golden):
    """Same torch seed -> bit-identical initial tables and generator state (transE.py:31-46 ...)."""
    import kgrec_b200 as K
    g = golden("dropin_init")
    classes = {"transE": K.TransEModel, "transH": K.TransHModel, "transR": K.TransRModel, "transUP": K.TransUPModel,
               "jTransUP": K.jTransUPModel}
    for name, args in DROPIN_INIT_CASES:
        torch.manual_seed(11)
        b = classes[name](*args)
        rb = torch.rand(3)
        want = {k[len(name) + 1:]: v for k, v in g.items() if k.startswith(name + "/") and k != name + "/rand"}
        sb = b.state_dict()
        assert set(want) == set(sb), name
        for k in want:
            assert np.array_equal(want[k], sb[k].cpu().numpy()), (name, k)
        assert np.array_equal(g[name + "/rand"], rb.numpy())
