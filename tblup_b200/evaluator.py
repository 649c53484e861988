"""Drop-in evaluators: the interface of tblup/evaluator.py on top of the B200 engine.

Same class names, constructor arguments, attributes, RNG consumption and error behaviour as the reference
(tblup/evaluator.py:14-55 factory, :63-99 ABC, :158-431 BlupParallelEvaluator, :434-561 CV variants,
:569-633 SNPRemovalHandler), so ``tblup.Population``, the evolvers, selector, seeder, monitor, scheduler and
``main.py`` drive it unchanged (``tblup_b200.install`` plugs it into an importable reference package).

What differs is the engine room: where the reference spawns ``n_procs`` worker processes in ``__enter__``
(evaluator.py:120-131) and pickles one job per individual through an ``mp.Queue`` (:227-241, :392-398), this
class uploads the genotypes to the GPU(s) once in ``__enter__`` and ships each generation's genomes in one
C-ABI call per device (``GblupEngine.evaluate_packed``).  There is no CPU path here.
"""
import abc
import os
import random
import threading
from math import sqrt

import numpy as np
from sklearn.model_selection import train_test_split

from .engine import GblupEngine, MODE_AUTO, MODE_GBLUP, MODE_SNPBLUP, pack_genomes

TESTING_SLOT = 1          # row set (training + validation -> testing) of evaluate_testing
FIRST_FOLD_SLOT = 2       # cross-validation folds live in slots 2, 3, ...
MONTE_CARLO_SLOT = 2


def _devices_from_env():
    spec = os.environ.get("TBLUP_B200_DEVICES", "").strip()
    if not spec:
        return [int(os.environ.get("LOCAL_RANK", "0"))] if "LOCAL_RANK" in os.environ else [0]
    if spec == "all":
        import torch
        return list(range(torch.cuda.device_count()))
    return [int(t) for t in spec.split(",") if t.strip() != ""]


def get_evaluator(args):
    """Evaluator for ``args.regressor`` (argparse namespace of tblup/config.py); mirrors evaluator.py:14-55."""
    splitter = None
    if args.splitter == "pca":
        # start-up helper (SURVEY.md 8f row F4): the full-marker GRM behind the split comes from the GPU kernels
        from .splitter import pca_splitter
        device = _devices_from_env()[0]
        splitter = lambda data: pca_splitter(data, outliers=args.pca_outliers, device=device)  # noqa: E731
    r = args.features if args.removal_r is None else args.removal_r
    positional = [args.geno, args.pheno, args.heritability]
    keyword = {"n_procs": args.processes, "splitter": splitter,
               "snp_remover": SNPRemovalHandler(r, args.h2_alpha, args.heritability, args.remove_snps)}
    kinds = {
        args.REGRESSOR_TYPE_BLUP: (BlupParallelEvaluator, False),
        args.REGRESSOR_TYPE_INTRACV_BLUP: (IntraGCVBlupParallelEvaluator, True),
        args.REGRESSOR_TYPE_INTERCV_BLUP: (InterGCVBlupParallelEvaluator, True),
        args.REGRESSOR_TYPE_MONTECV_BLUP: (MonteCarloCVBlupParallelEvaluator, False),
    }
    if args.regressor not in kinds:
        raise NotImplementedError("Regressor described by {} not implemented.".format(args.regressor))
    cls, wants_folds = kinds[args.regressor]
    if wants_folds:
        keyword["n_folds"] = args.cv_folds
    return cls(*positional, **keyword)


class Evaluator(abc.ABC):
    """The four-method contract of tblup/evaluator.py:63-99."""

    def __init__(self, data_path, labels_path):
        assert os.path.isfile(data_path), "Argument for data_path {} not found.".format(data_path)
        assert os.path.isfile(labels_path), "Argument for labels_path {} not found.".format(labels_path)
        self.data_path = data_path
        self.labels_path = labels_path

    @abc.abstractmethod
    def __enter__(self):
        pass

    @abc.abstractmethod
    def __exit__(self, exc_type, exc_val, exc_tb):
        pass

    @abc.abstractmethod
    def evaluate(self, previous_population, next_population, generation):
        raise NotImplementedError()

    @abc.abstractmethod
    def genomes_to_evaluate(self, population):
        raise NotImplementedError()


class ParallelEvaluator(Evaluator):
    """Lifetime of the device contexts.  ``consumers`` lists the live engines the way the reference lists its
    worker processes (evaluator.py:102-155); ``evaluate`` refuses to run outside the ``with`` block."""

    def __init__(self, data_path, labels_path, n_procs=-1):
        super().__init__(data_path, labels_path)
        self.n_procs = n_procs          # accepted for signature compatibility; the GPU needs no worker processes
        self.consumers = []

    def __exit__(self, exc_type, exc_val, exc_tb):
        for engine in self.consumers:
            engine.close()
        self.consumers = []

    def genomes_to_evaluate(self, population):
        raise NotImplementedError()

    def evaluate(self, previous_population, next_population, generation):
        if len(self.consumers) == 0:
            raise AttributeError("Workers are not set up.")


class BlupParallelEvaluator(ParallelEvaluator):
    """GBLUP / SNP-BLUP prediction accuracy of every individual of a generation, on the GPU.

    Constructor draws from the global ``random`` and ``numpy.random`` states exactly as
    tblup/evaluator.py:196-203 does (one ``random.sample`` and two ``train_test_split`` calls), so a seeded run
    sees the same splits and the same DE trajectory as the reference."""

    TRAIN_TEST_SPLIT = 0.8
    TRAIN_VALID_SPLIT = 0.8

    def __init__(self, data_path, labels_path, h2, n_procs=-1, splitter=None, snp_remover=None, devices=None):
        super().__init__(data_path, labels_path, n_procs=n_procs)
        self.archive = {}
        self.snp_remover = snp_remover
        self.h2 = h2
        self.devices = list(devices) if devices is not None else _devices_from_env()
        # how the genotypes stay resident in HBM: "int8" or "packed2" (2 bits per dosage; bit-identical results)
        self.storage = os.environ.get("TBLUP_B200_STORAGE", "packed2")
        if str(data_path).endswith(".bed"):
            # PLINK binary genotypes (not a reference format: its float64 .npy stops fitting in host memory long
            # before the GPU is full); animals = length of the phenotype vector
            self.n_samples = int(np.asarray(np.load(labels_path)).size)
            self.n_columns = (os.path.getsize(data_path) - 3) // ((self.n_samples + 3) // 4)
        else:
            shape = np.load(data_path, mmap_mode="r").shape
            self.n_samples, self.n_columns = shape[0], shape[1]
        if splitter:
            self.training_indices, self.testing_indices = splitter(self._load_dense())
        else:
            shuffled = random.sample(range(self.n_samples), self.n_samples)
            self.training_indices, self.testing_indices = train_test_split(
                shuffled, train_size=self.TRAIN_TEST_SPLIT, test_size=1 - self.TRAIN_TEST_SPLIT)
        self.training_indices, self.validation_indices = train_test_split(
            self.training_indices, train_size=self.TRAIN_VALID_SPLIT, test_size=1 - self.TRAIN_VALID_SPLIT)

    # ---- device lifetime ---------------------------------------------------------------------------------
    def _load_dense(self):
        """What the reference hands a custom splitter (evaluator.py:188): the dense matrix as float64."""
        if str(self.data_path).endswith(".bed"):
            from .genoio import read_bed
            return read_bed(self.data_path, self.n_samples).unpack().astype(np.float64)
        return np.load(self.data_path)

    def __enter__(self):
        from .genoio import load_genotypes
        geno = load_genotypes(self.data_path, self.n_samples)
        pheno = np.load(self.labels_path)
        order = np.concatenate((self.training_indices, self.validation_indices, self.testing_indices)).astype(np.int64)
        if len(np.unique(order)) != self.n_samples:      # a custom splitter may not cover every animal
            order = np.concatenate((order, np.setdiff1d(np.arange(self.n_samples), order)))
        # one ingest (validate, permute, transpose, pack) on the first device; the other GPUs of the box receive the
        # resident matrix by a device-to-device copy (the reference has every worker np.load() the file, :215-216)
        for device in self.devices:
            if self.consumers and hasattr(self.consumers[0], "clone"):
                self.consumers.append(self.consumers[0].clone(device))
            else:
                self.consumers.append(GblupEngine(geno, pheno, perm=order, device=device, storage=self.storage))
        self._define_rowsets()
        return self

    def _define_rowsets(self):
        both = np.concatenate((self.training_indices, self.validation_indices))
        for engine in self.consumers:
            engine.set_rowset(0, self.training_indices, self.validation_indices)
            engine.set_rowset(TESTING_SLOT, both, self.testing_indices)

    # ---- the reference's static entry points (used by tblup/local.py:65) -------------------------------------
    _adhoc = {}

    @classmethod
    def _adhoc_engine(cls, data, labels, train_indices, validation_indices):
        # one cached data set at a time, recognised by IDENTITY of the arrays the caller holds; the entry keeps a
        # reference to both, so their ids cannot be recycled for other arrays while the entry lives
        entry = cls._adhoc.get("entry")
        if entry is None or entry["data"] is not data or entry["labels"] is not labels:
            if entry is not None:
                entry["engine"].close()
            cls._adhoc.clear()
            entry = {"engine": GblupEngine(data, labels, device=_devices_from_env()[0]), "rows": None,
                     "data": data, "labels": labels}
            cls._adhoc["entry"] = entry
        rows = (hash(np.asarray(train_indices).tobytes()), hash(np.asarray(validation_indices).tobytes()))
        if entry["rows"] != rows:
            entry["engine"].set_rowset(0, train_indices, validation_indices)
            entry["rows"] = rows
        return entry["engine"]

    @staticmethod
    def blup(indices, train_indices, validation_indices, data, labels, h2):
        """evaluator.py:244-263: GBLUP when the subset is larger than the animal count, else SNP-BLUP."""
        eng = BlupParallelEvaluator._adhoc_engine(data, labels, train_indices, validation_indices)
        return float(eng.evaluate([indices], slots=[0], h2=h2, mode=MODE_AUTO)[0, 0])

    @staticmethod
    def gblup(indices, train_indices, validation_indices, data, labels, h2):
        """evaluator.py:265-286."""
        eng = BlupParallelEvaluator._adhoc_engine(data, labels, train_indices, validation_indices)
        return float(eng.evaluate([indices], slots=[0], h2=h2, mode=MODE_GBLUP)[0, 0])

    @staticmethod
    def snp_blup(indices, train_indices, validation_indices, data, labels, h2):
        """evaluator.py:288-314."""
        eng = BlupParallelEvaluator._adhoc_engine(data, labels, train_indices, validation_indices)
        return float(eng.evaluate([indices], slots=[0], h2=h2, mode=MODE_SNPBLUP)[0, 0])

    # ---- per-generation driver -----------------------------------------------------------------------------
    def train_validation_indices(self, generation):
        return self.training_indices, self.validation_indices

    def _slots_for(self, generation):
        """Row-set slots the fitness of this generation is computed on (mean over them)."""
        return [0]

    def __getstate__(self):
        return {k: v for k, v in self.__dict__.items() if k not in ("archive", "pool", "consumers")}

    def genomes_to_evaluate(self, population):
        """evaluator.py:339-357: every individual whose uid is not archived (or the remover's filtered view)."""
        if self.snp_remover is not None and self.snp_remover.should_remove():
            return self.snp_remover.genomes_to_evaluate(population, self.archive)
        to_evaluate, indices = [], []
        for i, indv in enumerate(population):
            if indv.uid not in self.archive:
                indices.append(i)
                to_evaluate.append(indv.genome)
        return to_evaluate, indices, False

    def evaluate(self, previous_population, next_population, generation):
        """evaluator.py:359-378."""
        super().evaluate(previous_population, next_population, generation)
        to_evaluate, indices, reevaluate = self.genomes_to_evaluate(next_population)
        next_population = self._evaluate(next_population, to_evaluate, indices, generation)
        if reevaluate:
            to_evaluate, indices, _ = self.genomes_to_evaluate(previous_population)
            self._evaluate(previous_population, to_evaluate, indices, generation)
            previous_population.monitor.log_snp_removal_event(generation)
        return next_population

    def _fitness_matrix(self, genomes, slots):
        """(len(genomes), len(slots)) fitness values; the batch is sharded over the engines (one host thread per
        device; the C calls release the GIL) in contiguous slices balanced by genome length."""
        if len(genomes) == 0:
            return np.empty((0, len(slots)))
        engines = self.consumers
        flat, off = pack_genomes(genomes, self.n_columns)
        if len(engines) == 1:
            from . import dist as tdist
            if tdist.rank_world()[1] > 1:
                # one process per GPU (torchrun): every rank runs the same seeded main loop, scores its contiguous
                # slice of the generation and the fitness vector is all-gathered (NCCL; gloo in the CPU tests)
                return tdist.evaluate_sharded(
                    lambda f, o: engines[0].evaluate_packed(np.ascontiguousarray(f), np.ascontiguousarray(o), slots,
                                                            self.h2, MODE_AUTO), flat, off, len(slots))
            return engines[0].evaluate_packed(flat, off, slots, self.h2, MODE_AUTO)
        cuts = shard_bounds(np.diff(off), len(engines))
        out = np.empty((len(genomes), len(slots)))
        errors = []

        def run(e, lo, hi):
            try:
                if hi > lo:
                    sub_off = off[lo:hi + 1] - off[lo]
                    out[lo:hi] = engines[e].evaluate_packed(flat[off[lo]:off[hi]], sub_off, slots, self.h2, MODE_AUTO)
            except Exception as exc:       # re-raised in the caller's thread
                errors.append(exc)

        threads = [threading.Thread(target=run, args=(e, cuts[e], cuts[e + 1])) for e in range(len(engines))]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if errors:
            raise errors[0]
        return out

    def _evaluate(self, population, to_evaluate, indices, generation):
        """evaluator.py:380-405 (and :509-537 for the intra-generation CV: fitness = mean over the folds)."""
        slots = self._slots_for(generation)
        fitness = self._fitness_matrix(to_evaluate, slots)
        values = fitness.sum(axis=1) / len(slots) if len(slots) > 1 else fitness[:, 0]
        for index, value in zip(indices, values):
            population[index].set_fitness(float(value))
            self.archive[population[index].uid] = population[index].fitness
        return population

    def evaluate_testing(self, population):
        """evaluator.py:407-431: train on training + validation, score on the testing animals, genomes united
        with every SNP removed so far."""
        if len(self.consumers) == 0:
            raise AttributeError("Workers are not set up.")
        genomes = [self.snp_remover.combine_with_removed(individual.genome) for individual in population]
        return [float(v) for v in self._fitness_matrix(genomes, [TESTING_SLOT])[:, 0]]


    # ---- panel models (the model behind evaluate_testing's number) ----------------------------------------------
    def _testing_genome(self, genome):
        if self.snp_remover is None:
            return np.asarray(genome).astype(int)
        return self.snp_remover.combine_with_removed(genome)

    def fit_model(self, genome):
        """The ``PanelModel`` whose testing accuracy ``evaluate_testing`` reports: trained on training + validation
        (the testing row set), on the genome united with every SNP removed so far, on the first engine."""
        if len(self.consumers) == 0:
            raise AttributeError("Workers are not set up.")
        return self.consumers[0].fit_models([self._testing_genome(genome)], slot=TESTING_SLOT, h2=self.h2,
                                            mode=MODE_AUTO)[0]

    def breeding_values(self, genome, animals=None):
        """Genomic estimated breeding values under ``fit_model(genome)`` of ``animals`` (original indices; default:
        the testing animals, whose |Pearson r| with the phenotypes is the testing accuracy)."""
        model = self.fit_model(genome)
        if animals is None:
            animals = self.testing_indices
        return self.consumers[0].predict([model], animals)[0]

    # ---- REML heritability ------------------------------------------------------------------------------------
    def estimate_h2(self, genome=None, **search):
        """REML estimate (``reml.H2Estimate``) of h2 on the training animals (row set 0) for ``genome``, by default
        every marker: the ``h2`` to run this evaluator with.  On the first engine, like ``fit_model``; ``search``
        passes ``tol`` / ``bounds`` on to ``GblupEngine.estimate_h2``."""
        if len(self.consumers) == 0:
            raise AttributeError("Workers are not set up.")
        g = np.arange(self.n_columns) if genome is None else np.asarray(genome).astype(int)
        return self.consumers[0].estimate_h2([g], slot=0, mode=MODE_AUTO, **search)[0]


class InterGCVBlupParallelEvaluator(BlupParallelEvaluator):
    """Validation fold rotates with the generation (evaluator.py:434-491)."""

    def __init__(self, data_path, labels_path, h2, n_procs=-1, n_folds=5, splitter=None, snp_remover=None,
                 devices=None):
        super().__init__(data_path, labels_path, h2, n_procs=n_procs, splitter=splitter, snp_remover=snp_remover,
                         devices=devices)
        self.n_folds = n_folds
        self.fold_indices = self.make_fold_indices(self.training_indices, self.n_folds)

    @staticmethod
    def make_fold_indices(indices, n_folds):
        """[[train, valid], ...] per fold: contiguous slices of ``indices``, the first ``len % n_folds`` folds one
        element longer (evaluator.py:455-483)."""
        indices = list(indices)
        base, extra = divmod(len(indices), n_folds)
        stops = np.cumsum([base + (1 if f < extra else 0) for f in range(n_folds)])
        starts = np.concatenate(([0], stops[:-1]))
        folds = [indices[a:b] for a, b in zip(starts, stops)]
        return [[[i for g, fold in enumerate(folds) if g != f for i in fold], folds[f]] for f in range(n_folds)]

    def _define_rowsets(self):
        super()._define_rowsets()
        for f, (train, valid) in enumerate(self.fold_indices):
            for engine in self.consumers:
                engine.set_rowset(FIRST_FOLD_SLOT + f, train, valid)

    def train_validation_indices(self, generation):
        return self.fold_indices[generation % self.n_folds]

    def _slots_for(self, generation):
        return [FIRST_FOLD_SLOT + generation % self.n_folds]


class IntraGCVBlupParallelEvaluator(InterGCVBlupParallelEvaluator):
    """k-fold cross-validation inside every fitness evaluation (evaluator.py:494-537).  The Gram of an individual
    does not depend on the fold, so the device forms it once and factors one matrix per fold."""

    def _slots_for(self, generation):
        return [FIRST_FOLD_SLOT + f for f in range(self.n_folds)]


class MonteCarloCVBlupParallelEvaluator(BlupParallelEvaluator):
    """A fresh random 80/20 split of training + validation for every batch (evaluator.py:540-561)."""

    def __init__(self, data_path, labels_path, h2, n_procs=-1, splitter=None, snp_remover=None, devices=None):
        super().__init__(data_path, labels_path, h2, n_procs=n_procs, splitter=splitter, snp_remover=snp_remover,
                         devices=devices)
        self.indices = np.concatenate((self.training_indices, self.validation_indices))

    def train_validation_indices(self, generation):
        return train_test_split(self.indices, test_size=0.2)

    def _slots_for(self, generation):
        train, valid = self.train_validation_indices(generation)     # consumes np.random like the reference
        for engine in self.consumers:
            engine.set_rowset(MONTE_CARLO_SLOT, train, valid)
        return [MONTE_CARLO_SLOT]


class SNPRemovalHandler:
    """Host-side index filtering of evaluator.py:569-633 (set arithmetic on marker lists; the kernels only ever
    see the filtered lists)."""

    def __init__(self, r, alpha, h2, remove_snps):
        self.r = r
        self.threshold = sqrt(h2) * (1 + alpha)
        self.removed = np.array([])
        self.remove_snps = remove_snps

    def should_remove(self):
        return self.remove_snps

    def genomes_to_evaluate(self, population, archive):
        best = max(population, key=lambda individual: individual.fitness)
        fire = best.fitness > self.threshold
        if fire:
            # reference quirk kept: when r < len(best) the WHOLE best genome is banned (evaluator.py:604)
            count = len(best) if self.r < len(best) else self.r
            self.removed = np.union1d(self.removed, best.genome[-count:])
            for key in list(archive.keys()):       # flush in place: callers hold a reference to this dict
                del archive[key]
        to_evaluate, indices = [], []
        for i, indv in enumerate(population):
            if indv.uid in archive:
                continue
            kept = np.setdiff1d(indv.genome, self.removed)
            if len(kept) == 0:
                archive[indv.uid] = 0.0
                indv.set_fitness(0.0)
            else:
                indices.append(i)
                to_evaluate.append(kept)
        return to_evaluate, indices, fire

    def combine_with_removed(self, genome):
        return np.union1d(genome, self.removed).astype(int)


def shard_bounds(lengths, n_shards):
    """Contiguous shard boundaries over a batch that balance the per-shard cost (k_i + c: the Cholesky cost is
    the same for every genome, the Gram cost grows with its length)."""
    lengths = np.asarray(lengths, dtype=np.float64)
    if len(lengths) == 0:
        return [0] * (n_shards + 1)
    cost = lengths + lengths.mean()
    csum = np.concatenate(([0.0], np.cumsum(cost)))
    targets = csum[-1] * np.arange(1, n_shards) / n_shards
    cuts = [0] + [int(np.searchsorted(csum, t, side="left")) for t in targets] + [len(lengths)]
    for i in range(1, len(cuts)):
        cuts[i] = max(cuts[i], cuts[i - 1])
    return cuts
