"""On-device differential evolution (DE/rand/1, binary crossover) over random-key individuals.

Host handle for the ``tb_de_*`` entry points: the P x m key matrix, the decoded genomes, the fitness vector and the
greedy selection all stay on the GPU; per generation the host passes a handful of scalars (and, optionally, the
random draws -- which is how the parity tests replay the reference's own Mersenne-Twister stream).
Mirrors tblup/evolver.py:86-157 (DERandOneEvolver), tblup/individual.py:132-167 (RandomKeyIndividual) and
tblup/selector.py:18-34 for the default configuration of the reference (``--de_strategy de_rand_1``).
"""
import ctypes as C

import numpy as np

from .engine import MODE_AUTO


def mutation_intensity(generation, configured):
    """F used in ``generation``: 5 on every fifth generation, else the configured value (tblup/evolver.py:147-151)."""
    return 5.0 if generation % 5 == 0 else float(configured)


class DeviceDE:
    def __init__(self, engine, population_size, length, keys=None, seed=0):
        self.eng = engine
        self.P, self.k, self.m = int(population_size), int(length), engine.m
        kp = None
        if keys is not None:
            keys = np.ascontiguousarray(np.asarray(keys, dtype=np.float64))
            if keys.shape != (self.P, self.m):
                raise ValueError("keys must have shape (population, markers)")
            kp = keys.ctypes.data
        engine._check(engine._lib.tb_de_init(engine._ctx, self.P, self.k, kp, int(seed)), "tb_de_init")
        self.generation = 0

    def evaluate(self, slots=(0,), h2=0.4, mode=MODE_AUTO):
        """Fitness of the current population (generation 0, tblup/population.py:47)."""
        s = np.ascontiguousarray(np.asarray(slots, dtype=np.int32))
        self.eng._check(self.eng._lib.tb_de_evaluate(self.eng._ctx, s.ctypes.data, s.size, float(h2), int(mode)),
                        "tb_de_evaluate")
        return self.fitness()

    def step(self, F, CR, slots=(0,), h2=0.4, mode=MODE_AUTO, clip=False, abc=None, fixed=None, mask=None, seed=0):
        """One generation: evolve -> decode -> evaluate -> select.  Returns the boolean 'child replaced parent' vector."""
        s = np.ascontiguousarray(np.asarray(slots, dtype=np.int32))
        pa = pf = pm = None
        if abc is not None:
            abc = np.ascontiguousarray(np.asarray(abc, dtype=np.int32).reshape(self.P, 3))
            fixed = np.ascontiguousarray(np.asarray(fixed, dtype=np.int32).reshape(self.P))
            pa, pf = abc.ctypes.data, fixed.ctypes.data
        if mask is not None:
            mask = np.ascontiguousarray(np.asarray(mask).astype(np.uint8).reshape(self.P, self.m))
            pm = mask.ctypes.data
        take = np.zeros(self.P, dtype=np.int32)
        self.eng._check(self.eng._lib.tb_de_step(self.eng._ctx, s.ctypes.data, s.size, float(h2), int(mode), float(F),
                                                 float(CR), int(bool(clip)), pa, pf, pm, int(seed), take.ctypes.data),
                        "tb_de_step")
        self.generation += 1
        return take.astype(bool)

    # ---- population replicated on every GPU of the box, evaluation sharded over the ranks (SURVEY 8e) ---------------
    class _DeviceVector:
        """Zero-copy view of a device vector of the library for torch (CUDA array interface)."""

        def __init__(self, ptr, n):
            self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (int(ptr), False), "version": 2}

    def _shard(self, group=None):
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        return self.P * rank // world, self.P * (rank + 1) // world

    def _share(self, what, lo, hi, group=None):
        """Every rank filled [lo, hi) of the fitness vector `what`; afterwards every rank holds all of it.  A sum of
        vectors that are zero outside the own shard: P doubles over NCCL, exact (x + 0 = x, NaN stays NaN), and shards
        may differ in size."""
        import torch
        import torch.distributed as dist
        ptr = self.eng._lib.tb_de_device_ptr(self.eng._ctx, int(what))
        v = torch.as_tensor(self._DeviceVector(ptr, self.P), device=torch.device("cuda", self.eng.device))
        v[:lo] = 0.0
        v[hi:] = 0.0
        dist.all_reduce(v, group=group)
        torch.cuda.synchronize(self.eng.device)

    def evaluate_distributed(self, slots=(0,), h2=0.4, mode=MODE_AUTO, group=None):
        """Generation 0 with the evaluation sharded over the ranks of ``group`` (keys must be identical on all ranks:
        same host keys or same seed)."""
        lo, hi = self._shard(group)
        s = np.ascontiguousarray(np.asarray(slots, dtype=np.int32))
        self.eng._check(self.eng._lib.tb_de_evaluate_shard(self.eng._ctx, s.ctypes.data, s.size, float(h2), int(mode),
                                                           lo, hi - lo), "tb_de_evaluate_shard")
        self._share(0, lo, hi, group)
        return self.fitness()

    def step_distributed(self, F, CR, slots=(0,), h2=0.4, mode=MODE_AUTO, clip=False, seed=0, group=None):
        """One generation: every rank evolves all offspring (device draws from ``seed``: identical everywhere), scores
        its shard, the offspring fitness is shared, every rank applies the same selection.  No key crosses NVLink."""
        lo, hi = self._shard(group)
        s = np.ascontiguousarray(np.asarray(slots, dtype=np.int32))
        self.eng._check(self.eng._lib.tb_de_step_begin(self.eng._ctx, s.ctypes.data, s.size, float(h2), int(mode),
                                                       float(F), float(CR), int(bool(clip)), None, None, None, int(seed),
                                                       lo, hi - lo), "tb_de_step_begin")
        self._share(1, lo, hi, group)
        take = np.zeros(self.P, dtype=np.int32)
        self.eng._check(self.eng._lib.tb_de_step_end(self.eng._ctx, take.ctypes.data), "tb_de_step_end")
        self.generation += 1
        return take.astype(bool)

    def run(self, generations, mutation=0.5, CR=0.8, slots=(0,), h2=0.4, mode=MODE_AUTO, clip=False, seed=0):
        """``generations`` device-driven generations with the reference's F schedule; returns best fitness per generation."""
        best = []
        for _ in range(generations):
            gen = self.generation + 1
            self.step(mutation_intensity(gen, mutation), CR, slots, h2, mode, clip, seed=seed * 1000003 + gen)
            best.append(float(np.nanmax(self.fitness())))
        return best

    # ---- SNP removal on the device (tblup/evaluator.py:569-633) ----------------------------------------------------
    def set_removed(self, markers):
        """Replace the removed-marker set with a host list (e.g. the state of a host-side SNPRemovalHandler)."""
        a = np.ascontiguousarray(np.asarray(markers, dtype=np.int32).ravel())
        self.eng._check(self.eng._lib.tb_de_set_removed(self.eng._ctx, a.ctypes.data if a.size else None, a.size),
                        "tb_de_set_removed")

    def ban_genome(self, i):
        """Add the decoded genome of individual ``i`` to the removed set (device side); returns the set's new size."""
        n = C.c_int32(0)
        self.eng._check(self.eng._lib.tb_de_ban_genome(self.eng._ctx, int(i), C.byref(n)), "tb_de_ban_genome")
        return int(n.value)

    def removed(self):
        """Removed markers, ascending (the handler's ``removed`` array)."""
        lens = self._removed_count()
        return self._get(6, (lens,), np.int32) if lens else np.empty(0, dtype=np.int32)

    def _removed_count(self):
        return int(self.eng.info("de_removed"))

    def maybe_remove(self, threshold, slots=(0,), h2=0.4, mode=MODE_AUTO):
        """The handler's rule (evaluator.py:601-611): when the best fitness exceeds ``threshold`` the best individual's
        markers are removed and the population is scored again without them.  Returns True when it fired."""
        fit = self.fitness()
        if not np.any(fit > threshold):
            return False
        self.ban_genome(int(np.nanargmax(fit)))
        self.evaluate(slots, h2, mode)
        return True

    def evaluate_testing(self, slot, h2=0.4, mode=MODE_AUTO):
        """Testing accuracy of the population: union(genome, removed) on row set ``slot`` (evaluator.py:407-431)."""
        out = np.empty(self.P, dtype=np.float64)
        self.eng._check(self.eng._lib.tb_de_evaluate_testing(self.eng._ctx, int(slot), float(h2), int(mode),
                                                             out.ctypes.data), "tb_de_evaluate_testing")
        return out

    def _staged(self):
        """Genomes of the last scored batch: P, or this rank's shard after a sharded evaluation."""
        return int(self.eng.info("staged"))

    def last_lengths(self):
        """Marker counts of the last batch scored with a non-empty removed set (shard-local after a sharded step)."""
        return self._get(7, (min(self.P, self._staged()),), np.int32)

    def last_lists(self):
        """The ragged marker lists of the last scored batch (after removal / union), one array per individual."""
        off = np.asarray(self.eng.staged_offsets())
        flat = self._get(8, (int(off[-1]),), np.int32)
        return [flat[off[i]:off[i + 1]] for i in range(off.size - 1)]

    def _get(self, what, shape, dtype, which=0):
        out = np.empty(shape, dtype=dtype)
        self.eng._check(self.eng._lib.tb_de_get(self.eng._ctx, what, int(which), out.ctypes.data, out.nbytes), "tb_de_get")
        return out

    def fitness(self):
        return self._get(0, (self.P,), np.float64)

    def child_fitness(self):
        return self._get(1, (self.P,), np.float64)

    def keys(self):
        return self._get(2, (self.P, self.m), np.float64)

    def child_keys(self):
        return self._get(3, (self.P, self.m), np.float64)

    def genome(self, i):
        """Decoded genome of individual ``i`` (the set of its ``length`` largest keys, ascending marker index)."""
        return self._get(4, (self.k,), np.int32, which=i)

    def last_draws(self):
        """(abc [P, 3], fixed [P]) of the last generation: the host's draws, or the ones made on the device."""
        return self._get(9, (self.P, 3), np.int32), self._get(10, (self.P,), np.int32)

    def last_genomes(self):
        """Genomes of the last scored batch, (staged, k); only meaningful while no marker is removed (fixed length)."""
        return self._get(5, (self._staged(), self.k), np.int32)
