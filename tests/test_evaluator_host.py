"""Host-side logic of the drop-in evaluators on CPU: constructor RNG parity, the evaluator contract, SNP removal,
CV row-set handling, multi-device sharding and -- when the reference checkout is present -- the reference's own
main loop driving our classes through the ``tblup.get_evaluator`` seam.  The device is replaced by
tests/fake_engine.OracleEngine (oracle-backed; test infrastructure)."""
import os
import random
import sys

import numpy as np
import pytest

from conftest import load_golden, unpack
from fake_engine import OracleEngine
from oracle import stage_ref

REF = stage_ref.ref_path()
HAVE_REF = REF is not None


class Indv:
    """Minimal individual: what tblup/individual.py exposes to the evaluator (uid, genome, fitness, set_fitness)."""
    _uid = 0

    def __init__(self, genome):
        Indv._uid += 1
        self.uid = Indv._uid
        self.genome = np.asarray(genome)
        self.fitness = None

    def set_fitness(self, f):
        self.fitness = f

    def __len__(self):
        return len(self.genome)


@pytest.fixture()
def dataset(tmp_path, monkeypatch):
    g = load_golden("fit_small")
    geno, pheno = tmp_path / "geno.npy", tmp_path / "pheno.npy"
    np.save(geno, g["x"].astype(np.float64))
    np.save(pheno, g["y"])
    import tblup_b200.evaluator as ev
    monkeypatch.setattr(ev, "GblupEngine", OracleEngine)
    OracleEngine.instances.clear()
    return g, str(geno), str(pheno), ev


def seeded(seed):
    random.seed(seed)
    np.random.seed(seed)


def test_constructor_consumes_rng_like_reference(dataset):
    g, geno, pheno, ev = dataset
    seeded(int(g["seed"]))
    e = ev.InterGCVBlupParallelEvaluator(geno, pheno, float(g["h2"]), n_procs=1, n_folds=int(g["n_folds"]),
                                         snp_remover=ev.SNPRemovalHandler(10, 0.0, float(g["h2"]), False))
    assert list(e.training_indices) == list(g["train"])
    assert list(e.validation_indices) == list(g["valid"])
    assert list(e.testing_indices) == list(g["test"])
    f_tr = unpack(g["fold_train_flat"], g["fold_train_off"])
    f_va = unpack(g["fold_valid_flat"], g["fold_valid_off"])
    for f, (tr, va) in enumerate(e.fold_indices):
        assert tr == list(f_tr[f]) and va == list(f_va[f])
    after = (random.random(), np.random.rand())
    seeded(int(g["seed"]))
    from oracle import gblup_oracle as O
    O.ref_splits(g["x"].shape[0])
    assert after == (random.random(), np.random.rand())


def test_split_sets_are_disjoint(dataset):
    """The reference's only evaluator unit test (tblup/test/evaluator.py:26-39)."""
    g, geno, pheno, ev = dataset
    e = ev.BlupParallelEvaluator(geno, pheno, 0.5)
    sets = [e.training_indices, e.validation_indices, e.testing_indices]
    for s in sets:
        assert len(s) == len(set(s))
    assert not set(sets[0]) & set(sets[1]) and not set(sets[0]) & set(sets[2]) and not set(sets[1]) & set(sets[2])
    assert sum(len(s) for s in sets) == g["x"].shape[0]


def test_evaluate_outside_with_block_raises(dataset):
    g, geno, pheno, ev = dataset
    e = ev.BlupParallelEvaluator(geno, pheno, 0.4, snp_remover=ev.SNPRemovalHandler(5, 0.0, 0.4, False))
    with pytest.raises(AttributeError, match="Workers are not set up"):
        e.evaluate([], [Indv([1, 2])], 0)
    with pytest.raises(AssertionError):
        ev.BlupParallelEvaluator("/no/such/file.npy", pheno, 0.4)


def test_evaluate_sets_fitness_and_archive(dataset):
    g, geno, pheno, ev = dataset
    h2 = float(g["h2"])
    seeded(int(g["seed"]))
    e = ev.BlupParallelEvaluator(geno, pheno, h2, snp_remover=ev.SNPRemovalHandler(5, 0.0, h2, False))
    genomes = unpack(g["genomes_flat"], g["genomes_off"])
    pop = [Indv(x) for x in genomes]
    with e:
        assert len(e.consumers) == 1
        out = e.evaluate(pop, pop, 0)
        assert out is pop
        for ind, ref in zip(pop, g["ref_blup"]):
            assert isinstance(ind.fitness, float) and abs(ind.fitness - ref) < 1e-9
            assert e.archive[ind.uid] == ind.fitness
        n_calls = len(OracleEngine.instances[0].calls)
        e.evaluate(pop, pop, 1)                         # everything archived: nothing to do
        assert len(OracleEngine.instances[0].calls) == n_calls
        testing = e.evaluate_testing(pop)
        # evaluate_testing unites each genome with the removed SNPs (np.union1d: sorted AND de-duplicated,
        # tblup/evaluator.py:418,627-633), so genomes with repeated markers are scored on their unique set
        from oracle import gblup_oracle as O
        tv = np.concatenate((e.training_indices, e.validation_indices))
        for i, gen in enumerate(genomes):
            if len(np.unique(gen)) == len(gen):
                assert abs(testing[i] - g["ref_blup_testing"][i]) < 1e-9
            else:
                assert abs(testing[i] - O.exact_blup(np.unique(gen), tv, e.testing_indices, g["x"], g["y"], h2)) < 1e-12
    assert e.consumers == [] and OracleEngine.instances[0].closed


def test_bed_input_and_packed_storage_reach_the_engine(dataset, tmp_path, monkeypatch):
    """A PLINK .bed data path gives the same splits (same RNG consumption) and hands the engine the same dosages."""
    from tblup_b200.genoio import pack_dosages, write_bed
    g, geno, pheno, ev = dataset
    bed = tmp_path / "geno.bed"
    write_bed(str(bed), pack_dosages(g["x"]))
    monkeypatch.setenv("TBLUP_B200_STORAGE", "packed2")
    seeded(int(g["seed"]))
    e = ev.BlupParallelEvaluator(str(bed), pheno, float(g["h2"]), snp_remover=ev.SNPRemovalHandler(10, 0.0, 0.4, False))
    assert (e.n_samples, e.n_columns) == g["x"].shape
    assert list(e.training_indices) == list(g["train"]) and list(e.testing_indices) == list(g["test"])
    with e:
        inst = OracleEngine.instances[-1]
        assert inst.storage == "packed2" and np.array_equal(inst.x, g["x"])


def test_cv_variants_pick_the_right_row_sets(dataset):
    g, geno, pheno, ev = dataset
    h2, nf = float(g["h2"]), int(g["n_folds"])
    genomes = unpack(g["genomes_flat"], g["genomes_off"])[:5]
    rem = lambda: ev.SNPRemovalHandler(5, 0.0, h2, False)  # noqa: E731
    seeded(int(g["seed"]))
    inter = ev.InterGCVBlupParallelEvaluator(geno, pheno, h2, n_folds=nf, snp_remover=rem())
    with inter:
        for gen in range(nf + 1):
            pop = [Indv(x) for x in genomes]
            inter.evaluate(pop, pop, gen)
            want = g["ref_blup_folds"][:5, gen % nf]
            assert np.abs(np.array([p.fitness for p in pop]) - want).max() < 1e-9
    seeded(int(g["seed"]))
    intra = ev.IntraGCVBlupParallelEvaluator(geno, pheno, h2, n_folds=nf, snp_remover=rem())
    with intra:
        pop = [Indv(x) for x in genomes]
        intra.evaluate(pop, pop, 3)
        assert np.abs(np.array([p.fitness for p in pop]) - g["ref_blup_folds"][:5].mean(axis=1)).max() < 1e-9
        assert OracleEngine.instances[-1].calls[-1] == (5, tuple(range(2, 2 + nf)))   # one call, all folds
    seeded(int(g["seed"]))
    monte = ev.MonteCarloCVBlupParallelEvaluator(geno, pheno, h2, snp_remover=rem())
    state = np.random.get_state()
    from sklearn.model_selection import train_test_split
    tr, va = train_test_split(monte.indices, test_size=0.2)
    np.random.set_state(state)
    with monte:
        pop = [Indv(x) for x in genomes]
        monte.evaluate(pop, pop, 0)
        got_tr, got_va = OracleEngine.instances[-1].rowsets[2]
        assert list(got_tr) == list(tr) and list(got_va) == list(va)


def test_snp_removal_handler(dataset):
    g, geno, pheno, ev = dataset
    h = ev.SNPRemovalHandler(2, 0.0, 0.25, True)     # threshold 0.5
    a, b, c = Indv([5, 6, 7]), Indv([6, 7]), Indv([1, 2, 3])
    a.fitness, b.fitness, c.fitness = 0.9, 0.1, 0.2
    archive = {a.uid: 0.9, b.uid: 0.1, c.uid: 0.2, 999: 1.0}
    same = archive
    to_eval, idx, fired = h.genomes_to_evaluate([a, b, c], archive)
    assert fired and archive is same
    assert sorted(h.removed.tolist()) == [5, 6, 7]          # r < len(best): the whole best genome goes
    assert a.fitness == 0.0 and b.fitness == 0.0 and archive[a.uid] == 0.0 and 999 not in archive
    assert idx == [2] and to_eval[0].tolist() == [1, 2, 3]
    assert h.combine_with_removed(np.array([9, 1])).tolist() == [1, 5, 6, 7, 9]
    quiet = ev.SNPRemovalHandler(2, 0.0, 0.25, False)
    assert not quiet.should_remove()


def test_batch_is_sharded_over_devices(dataset):
    g, geno, pheno, ev = dataset
    h2 = float(g["h2"])
    genomes = unpack(g["genomes_flat"], g["genomes_off"])
    seeded(int(g["seed"]))
    e = ev.BlupParallelEvaluator(geno, pheno, h2, snp_remover=ev.SNPRemovalHandler(5, 0.0, h2, False),
                                 devices=[0, 1, 2])
    pop = [Indv(x) for x in genomes]
    with e:
        e.evaluate(pop, pop, 0)
        sizes = [inst.calls[0][0] for inst in OracleEngine.instances]
        assert len(sizes) == 3 and sum(sizes) == len(genomes) and min(sizes) >= 1
    assert np.abs(np.array([p.fitness for p in pop]) - g["ref_blup"]).max() < 1e-9
    cuts = ev.shard_bounds([10] * 8, 3)
    assert cuts[0] == 0 and cuts[-1] == 8 and all(b >= a for a, b in zip(cuts, cuts[1:]))
    assert ev.shard_bounds([], 4) == [0, 0, 0, 0, 0]


def _dist_worker(rank, world, port, flat, off, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from tblup_b200.dist import evaluate_sharded

    def eval_fn(f, o):   # fitness stand-in: (sum of the genome, its length)
        return np.array([[f[o[i]:o[i + 1]].sum(), o[i + 1] - o[i]] for i in range(o.size - 1)], dtype=np.float64)

    out = evaluate_sharded(eval_fn, flat, off, 2)
    q.put((rank, out))
    dist.destroy_process_group()


def test_population_sharding_over_ranks_gloo():
    import torch.multiprocessing as mp
    rng = np.random.default_rng(0)
    lens = rng.integers(1, 40, size=11)
    off = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    flat = rng.integers(0, 1000, size=int(off[-1])).astype(np.int32)
    want = np.array([[flat[off[i]:off[i + 1]].sum(), lens[i]] for i in range(11)], dtype=np.float64)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_dist_worker, args=(r, 2, port, flat, off, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert np.array_equal(got[0], want) and np.array_equal(got[1], want)


def _dist_eval_worker(rank, world, port, geno, pheno, genomes, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import tblup_b200.evaluator as ev
    ev.GblupEngine = OracleEngine
    seeded(3)
    e = ev.IntraGCVBlupParallelEvaluator(geno, pheno, 0.4, n_folds=3, snp_remover=ev.SNPRemovalHandler(10, 0.0, 0.4, False),
                                         devices=[0])
    pop = [Indv(g) for g in genomes]
    with e:
        e.evaluate(pop, pop, 0)
        sizes = [c[0] for c in OracleEngine.instances[-1].calls]
    q.put((rank, [p.fitness for p in pop], sizes))
    dist.destroy_process_group()


def test_evaluator_shards_over_torch_distributed_ranks_gloo(tmp_path):
    """One process per GPU (torchrun): the evaluator class scores its slice and all-gathers -- every rank ends with the
    whole generation's fitness, equal to a single-process run."""
    import torch.multiprocessing as mp
    g = load_golden("fit_small")
    geno, pheno = tmp_path / "geno.npy", tmp_path / "pheno.npy"
    np.save(geno, g["x"].astype(np.float64))
    np.save(pheno, g["y"])
    genomes = [np.asarray(x) for x in unpack(g["genomes_flat"], g["genomes_off"])]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + os.getpid() % 2000
    procs = [ctx.Process(target=_dist_eval_worker, args=(r, 2, port, str(geno), str(pheno), genomes, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = {r: (f, s) for r, f, s in (q.get(timeout=180) for _ in procs)}
    for p in procs:
        p.join(timeout=60)
    assert got[0][0] == got[1][0] and all(np.isfinite(got[0][0]))
    assert got[0][1][0] + got[1][1][0] == len(genomes) and min(got[0][1][0], got[1][1][0]) >= 1
    import tblup_b200.evaluator as ev
    seeded(3)
    e = ev.IntraGCVBlupParallelEvaluator(str(geno), str(pheno), 0.4, n_folds=3,
                                         snp_remover=ev.SNPRemovalHandler(10, 0.0, 0.4, False), devices=[0])
    saved = ev.GblupEngine
    ev.GblupEngine = OracleEngine
    try:
        pop = [Indv(x) for x in genomes]
        with e:
            e.evaluate(pop, pop, 0)
    finally:
        ev.GblupEngine = saved
    assert np.abs(np.array([p.fitness for p in pop]) - np.array(got[0][0])).max() < 1e-12


@pytest.mark.skipif(not HAVE_REF, reason="no reference checkout or oracle/_ref mirror (oracle/stage_ref.py)")
@pytest.mark.parametrize("name", ["traj_gblup", "traj_intracv"])
def test_reference_main_loop_drives_our_evaluator(name, tmp_path, monkeypatch):
    """The UNMODIFIED reference Population / evolver / selector / monitor, wired by its own build_kwargs, with our
    evaluator plugged in through tblup.get_evaluator: same best-fitness trajectory and selected panel as the
    recording of the reference's own evaluator (tests/golden/make_golden.py)."""
    g = load_golden(name)
    if REF not in sys.path:
        monkeypatch.syspath_prepend(REF)
    import tblup
    import tblup_b200.evaluator as ev
    from tblup_b200.install import install
    monkeypatch.setattr(ev, "GblupEngine", OracleEngine)
    monkeypatch.setattr(tblup, "get_evaluator", tblup.get_evaluator)     # restored after the test
    install(tblup)
    geno, pheno = tmp_path / "geno.npy", tmp_path / "pheno.npy"
    np.save(geno, g["x"].astype(np.float64))
    np.save(pheno, g["y"])
    monkeypatch.chdir(tmp_path)
    from tblup.config import parser
    gens = int(g["gens"])
    args = parser.parse_args(["--geno", str(geno), "--pheno", str(pheno), "--seed", str(int(g["seed"])),
                              "--features", str(int(g["features"])), "--population_size", str(int(g["pop"])),
                              "--generations", str(gens), "--heritability", str(float(g["h2"])),
                              "--regressor", str(g["regressor"]), "--cv_folds", "3", "-p", "1"])
    seeded(args.seed)
    kwargs = tblup.build_kwargs(args)
    evaluator = kwargs["evaluator"]
    assert isinstance(evaluator, tblup.BlupParallelEvaluator) and isinstance(evaluator, ev.BlupParallelEvaluator)
    best_fit, best_genome = [], []
    with evaluator:
        population = tblup.Population(**kwargs)
        for _ in range(gens + 1):
            b = max(population, key=lambda ind: ind.fitness)
            best_fit.append(float(b.fitness))
            best_genome.append(np.sort(np.asarray(b.genome)))
            if population.generation > gens:
                break
            population.do_generation()
        testing = evaluator.evaluate_testing(population)
    assert len(testing) == int(g["pop"]) and all(isinstance(t, float) for t in testing)
    assert np.abs(np.array(best_fit) - g["best_fitness"]).max() < 1e-9
    assert np.array_equal(np.stack(best_genome), g["best_genome"])
