"""Panel models: the linear model behind the fitness of one genome (a selected SNP panel).

The reference fits it and throws it away: ``gblup`` forms the predictions of every animal and keeps the validation
entries (tblup/evaluator.py:284), ``snp_blup`` drops its ``Ridge`` model after one ``predict`` (:311-314).  A
``PanelModel`` keeps it, one effect per listed marker:

    yhat_b = intercept + sum_q (x_{b, markers[q]} - centre[q]) * effects[q]

``GblupEngine.fit_models`` produces them on the GPU and ``GblupEngine.predict`` applies them there; this module only
holds and stores them (there is no CPU path in the package).
"""
import numpy as np

BRANCHES = ("gblup", "snp_blup")


class PanelModel:
    """Marker effects of one genome on one training set.

    ``markers``: listed marker indices (duplicates kept, as numpy fancy indexing counts them); ``centre``: 2p of each
    listed marker over the frequency animals of the branch; ``effects``: one effect per listed marker; ``intercept``:
    0 for gblup, the mean training phenotype for snp_blup; ``branch``: "gblup" or "snp_blup"; ``h2``: heritability
    of the fit; ``fitness``: |Pearson r| on the validation animals of the row set it was fitted on (the value the
    fitness path reports for that genome), or nan when unknown."""

    def __init__(self, markers, centre, effects, intercept, branch, h2, fitness=float("nan")):
        self.markers = np.ascontiguousarray(np.asarray(markers, dtype=np.int64).ravel())
        self.centre = np.ascontiguousarray(np.asarray(centre, dtype=np.float64).ravel())
        self.effects = np.ascontiguousarray(np.asarray(effects, dtype=np.float64).ravel())
        if not (self.markers.size == self.centre.size == self.effects.size) or self.markers.size == 0:
            raise ValueError("a panel model needs one centre and one effect per listed marker (and at least one marker)")
        if branch not in BRANCHES:
            raise ValueError("branch must be one of %r, got %r" % (BRANCHES, branch))
        self.intercept = float(intercept)
        self.branch = branch
        self.h2 = float(h2)
        self.fitness = float(fitness)

    def __len__(self):
        return int(self.markers.size)

    def __repr__(self):
        return "PanelModel(%d markers, branch=%s, h2=%g, intercept=%.6g, fitness=%.6g)" % (
            len(self), self.branch, self.h2, self.intercept, self.fitness)

    def save(self, path):
        """Write the model as an ``.npz`` archive (numpy adds the suffix when ``path`` has none)."""
        np.savez(path, markers=self.markers, centre=self.centre, effects=self.effects,
                 intercept=np.float64(self.intercept), branch=np.array(self.branch), h2=np.float64(self.h2),
                 fitness=np.float64(self.fitness))

    @classmethod
    def load(cls, path):
        with np.load(path, allow_pickle=False) as z:
            return cls(z["markers"], z["centre"], z["effects"], float(z["intercept"]), str(z["branch"]),
                       float(z["h2"]), float(z["fitness"]))
