"""B200-native GraphMI attack of the defence repo -- same surface as the reference's MC-GPB/topology_attack.py.

`PGDAttack(model, embedding, nnodes, loss_type, device).attack(ori_features, ori_adj, labels, idx_attack, num_edges,
epochs, sample)` (MC-GPB/topology_attack.py:36-87): plain gradient descent with lr 0.1 on nll + 0.001 ||x||, from
iteration 50 on plus 1e-4 * tr(X^T L~ X) (feature smoothing, :57-61, 163-177), budget projection with the true edge
count (`--density 1`, so the device bisection is active every iteration), final decode relu(Z Z^T) WITHOUT row
normalisation (:247-254).  Runs on engine.PGDEngine (plain_gd) + the smoothing tile pass (csrc/misc.cu).
"""
import numpy as np

from .baseline import PGDAttack as _Baseline


class PGDAttack(_Baseline):
    plain_gd = True
    decode_normalised = False

    def attack(self, ori_features, ori_adj, labels, idx_attack, num_edges, epochs=200, sample=False, **kwargs):
        if int(epochs) > 201:
            raise NotImplementedError("epochs > 201 switch to a dense SVD truncation every iteration "
                                      "(MC-GPB/topology_attack.py:72-73); not part of the native path")

        def setup(eng, X):
            eng.enable_smoothing(X, 1e-4)

        def pre_iter(eng, t):
            eng.smooth_on = t >= 50                                   # :51-61
            eng.lr = 200.0 / np.sqrt(t + 1) if sample else 0.1        # :66-69
        return self._run(0.1, 1.0, ori_features, ori_adj, labels, idx_attack, num_edges, epochs,
                         trace=bool(kwargs.get("_trace")), gather_x=kwargs.get("_gather_x", True),
                         setup=setup if int(epochs) > 50 or kwargs.get("_smooth_from") is not None else None,
                         pre_iter=pre_iter if kwargs.get("_smooth_from") is None else
                         (lambda eng, t: (setattr(eng, "smooth_on", t >= kwargs["_smooth_from"]),
                                          setattr(eng, "lr", 0.1))))
