"""Host-side handle on one GPU context of libtblup_b200.so.

``GblupEngine`` owns a data set resident on one B200 (genotypes as int8 dosages, SNP-major; phenotypes;
row sets) and evaluates batches of genomes (marker-index lists) on it.  It is the object the evaluator
classes in ``tblup_b200.evaluator`` hold in place of the reference's worker pool
(tblup/evaluator.py:116-131): where the reference pickles one job per individual into an ``mp.Queue``
(evaluator.py:227-241) this class ships the whole generation in one call.
"""
import ctypes as C

import numpy as np

from . import _lib

MODE_AUTO, MODE_GBLUP, MODE_SNPBLUP = 0, 1, 2
STAGES = ["h2d", "gather", "centre", "gram", "scale", "chol_update", "chol_panel", "solve", "d2h"]
DBG_C, DBG_S, DBG_SQ, DBG_M, DBG_ALPHA, DBG_PRED, DBG_DIMS, DBG_L32, DBG_SWEEPS = range(9)
PRECISION_MIXED, PRECISION_FP64 = 0, 1
LAYOUT_INT8_ANIMAL_MAJOR, LAYOUT_PACKED2_SNP_MAJOR = 0, 1
STORAGE = {"int8": 0, "packed2": 1}


def as_dosage_int8(geno):
    """Validate a genotype matrix (any real dtype) holds dosages {0,1,2} and return it as C-contiguous int8.

    The reference keeps ``data`` as the float64 ``.npy`` it loaded (tblup/evaluator.py:215); the dosages are
    small integers, so int8 is lossless and an eighth of the bytes."""
    g = np.asarray(geno)
    if g.ndim != 2:
        raise ValueError("genotype matrix must be 2-D (animals x markers), got shape %r" % (g.shape,))
    if g.dtype != np.int8:
        gi = g.astype(np.int8)
        if not np.array_equal(gi, g):
            raise ValueError("genotype matrix must hold integer dosages 0/1/2")
        g = gi
    if g.size and (g.min() < 0 or g.max() > 2):
        raise ValueError("genotype matrix must hold dosages in {0, 1, 2}")
    return np.ascontiguousarray(g)


def pack_genomes(genomes, n_markers):
    """Ragged list of index arrays -> (flat int32, offsets int64) with numpy fancy-indexing semantics
    (tblup/evaluator.py:275, :298): negative indices wrap, out-of-range raises IndexError, duplicates stay.
    The copy / narrowing / range check of a generation's worth of indices (5 M for 1 000 genomes of 5 001 markers) runs in
    the library on several host threads (`tb_pack_index_lists`) instead of four numpy passes over the batch (concatenate,
    min / max, wrap, narrow): a third of their time on the 8-core build container."""
    arrs = []
    for g in genomes:
        a = np.asarray(g)
        if a.dtype.kind not in "iu":                 # the reference hands float arrays after union1d / setdiff1d
            ai = a.astype(np.int64)
            if not np.array_equal(ai, a):
                raise IndexError("arrays used as indices must be of integer type")
            a = ai
        a = a.ravel()
        if a.dtype not in (np.int32, np.int64) or not a.flags.c_contiguous or not a.dtype.isnative:
            a = np.ascontiguousarray(a, dtype=np.int64)
        arrs.append(a)
    P = len(arrs)
    off = np.zeros(P + 1, dtype=np.int64)
    if P == 0:
        return np.empty(0, dtype=np.int32), off
    lens = np.fromiter((a.size for a in arrs), dtype=np.int64, count=P)
    ptrs = np.fromiter((a.ctypes.data for a in arrs), dtype=np.uintp, count=P)
    width = np.fromiter((a.dtype.itemsize for a in arrs), dtype=np.int32, count=P)
    flat = np.empty(int(lens.sum()), dtype=np.int32)
    bad = C.c_int64(0)
    rc = _lib.load().tb_pack_index_lists(ptrs.ctypes.data, lens.ctypes.data, width.ctypes.data, P, int(n_markers),
                                    flat.ctypes.data, off.ctypes.data, C.byref(bad))
    if rc == -3:
        raise IndexError("index %d is out of bounds for axis 1 with size %d" % (bad.value, n_markers))
    if rc != 0:
        raise ValueError("tb_pack_index_lists rejected its arguments (rc = %d)" % rc)
    return flat, off


class GblupEngine:
    """One data set on one GPU.  Not thread-safe (one host thread per context, like the C-ABI)."""

    def __init__(self, geno, pheno=None, perm=None, device=0, storage="packed2"):
        """``geno``: dense dosages (animals x markers, any real dtype holding 0/1/2) or a
        ``genoio.PackedGenotypes``; ``storage``: how the matrix stays resident in HBM, ``"int8"`` (one byte per
        dosage) or ``"packed2"`` (2 bits per dosage, a quarter of the bytes; same results bit for bit).
        ``pheno=None``: a context without phenotypes, which only scores animals with models fitted elsewhere
        (``predict``); row sets, evaluations and fits are refused on it."""
        from .genoio import PackedGenotypes
        self._lib = _lib.load()
        self._ctx = C.c_void_p()
        if storage not in STORAGE:
            raise ValueError("storage must be 'int8' or 'packed2', got %r" % (storage,))
        if isinstance(geno, PackedGenotypes):
            g, layout, shape = geno.data, LAYOUT_PACKED2_SNP_MAJOR, geno.shape
        else:
            g, layout = as_dosage_int8(geno), LAYOUT_INT8_ANIMAL_MAJOR
            shape = g.shape
        self.has_phenotypes = pheno is not None
        y = None
        if pheno is not None:
            y = np.ascontiguousarray(np.asarray(pheno, dtype=np.float64).ravel())
            if y.shape[0] != shape[0]:
                raise ValueError("phenotype vector has %d entries for %d animals" % (y.shape[0], shape[0]))
        self.n, self.m = shape
        self.storage = storage
        p = None
        if perm is not None:
            p = np.ascontiguousarray(np.asarray(perm, dtype=np.int32))
            if p.shape != (self.n,):
                raise ValueError("perm must list every animal exactly once")
        rc = self._lib.tb_create_ex(g.ctypes.data, layout, STORAGE[storage], self.n, self.m,
                                    y.ctypes.data if y is not None else None,
                                    p.ctypes.data if p is not None else None, int(device), C.byref(self._ctx))
        if rc != 0:
            self._ctx = C.c_void_p()
            raise RuntimeError("tb_create failed (%d): %s" % (rc, self._lib.tb_last_error(None).decode()))
        self.device = int(device)
        self._n_staged = 0

    # -- lifetime ------------------------------------------------------------------------------
    def clone(self, device):
        """The same data set on another GPU of the box: device-to-device copy of the resident matrix (tb_clone), no
        second host ingest.  Row sets have to be defined on the clone."""
        other = object.__new__(GblupEngine)
        other._lib = self._lib
        other._ctx = C.c_void_p()
        rc = self._lib.tb_clone(self._ctx, int(device), C.byref(other._ctx))
        if rc != 0:
            other._ctx = C.c_void_p()
            raise RuntimeError("tb_clone failed (%d): %s" % (rc, self._lib.tb_last_error(None).decode()))
        other.n, other.m, other.storage, other.device, other._n_staged = self.n, self.m, self.storage, int(device), 0
        other.has_phenotypes = self.has_phenotypes
        return other

    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx:
            self._lib.tb_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise RuntimeError("%s failed (%d): %s" % (what, rc, self._lib.tb_last_error(self._ctx).decode()))

    # -- configuration -------------------------------------------------------------------------
    def set_rowset(self, slot, train, valid):
        if not self.has_phenotypes:
            raise RuntimeError("this context holds no phenotypes: it can only score animals (predict)")
        t = np.ascontiguousarray(np.asarray(train, dtype=np.int32))
        v = np.ascontiguousarray(np.asarray(valid, dtype=np.int32))
        self._check(self._lib.tb_set_rowset(self._ctx, int(slot), t.ctypes.data, t.size, v.ctypes.data, v.size),
                    "tb_set_rowset")

    def set_option(self, name, value):
        self._check(self._lib.tb_set_option(self._ctx, name.encode(), int(value)), "tb_set_option")

    # -- evaluation ----------------------------------------------------------------------------
    def stage(self, genomes=None, flat=None, off=None):
        """Copy a batch to the device.  Pass ``genomes`` (list of index arrays) or pre-packed flat/off."""
        if genomes is not None:
            flat, off = pack_genomes(genomes, self.m)
        flat = np.ascontiguousarray(flat, dtype=np.int32)
        off = np.ascontiguousarray(off, dtype=np.int64)
        self._check(self._lib.tb_stage_genomes(self._ctx, flat.ctypes.data, off.ctypes.data, off.size - 1),
                    "tb_stage_genomes")
        self._n_staged = off.size - 1

    def evaluate_staged(self, slots=(0,), h2=0.4, mode=MODE_AUTO, out=None, out_device_ptr=None):
        """Fitness of the staged batch on each row set -> array (P, n_slots), or written to a device pointer."""
        s = np.ascontiguousarray(np.asarray(slots, dtype=np.int32))
        if out_device_ptr is not None:
            self._check(self._lib.tb_eval_staged(self._ctx, s.ctypes.data, s.size, float(h2), int(mode),
                                                 C.c_void_p(int(out_device_ptr)), 1), "tb_eval_staged")
            return None
        if out is None:
            out = np.empty((self._n_staged, s.size), dtype=np.float64)
        self._check(self._lib.tb_eval_staged(self._ctx, s.ctypes.data, s.size, float(h2), int(mode),
                                             out.ctypes.data, 0), "tb_eval_staged")
        return out

    def evaluate(self, genomes, slots=(0,), h2=0.4, mode=MODE_AUTO):
        """One generation: host index lists in, host fitness out (P, n_slots)."""
        flat, off = pack_genomes(genomes, self.m)
        return self.evaluate_packed(flat, off, slots, h2, mode)

    def evaluate_packed(self, flat, off, slots=(0,), h2=0.4, mode=MODE_AUTO, out=None):
        s = np.ascontiguousarray(np.asarray(slots, dtype=np.int32))
        P = off.size - 1
        if out is None:
            out = np.empty((P, s.size), dtype=np.float64)
        self._check(self._lib.tb_eval(self._ctx, s.ctypes.data, s.size, flat.ctypes.data, off.ctypes.data, P,
                                      float(h2), int(mode), out.ctypes.data), "tb_eval")
        self._n_staged = P
        return out

    # -- panel models: marker effects and breeding values -----------------------------------------
    def fit_models(self, genomes, slot=0, h2=0.4, mode=MODE_AUTO):
        """One ``PanelModel`` per genome, trained on row set ``slot`` exactly as the fitness is computed there (same
        branch rule, precision and fp64 fallback; each model's ``fitness`` is the value ``evaluate`` returns).  The
        genomes become the staged batch (``stage``)."""
        from .model import PanelModel
        flat, off = pack_genomes(genomes, self.m)
        self.stage(flat=flat, off=off)
        P = off.size - 1
        effects = np.empty(flat.size, dtype=np.float64)
        centre = np.empty(flat.size, dtype=np.float64)
        intercept = np.empty(P, dtype=np.float64)
        fitness = np.empty(P, dtype=np.float64)
        self._check(self._lib.tb_fit_effects(self._ctx, int(slot), float(h2), int(mode), effects.ctypes.data,
                                             centre.ctypes.data, intercept.ctypes.data, fitness.ctypes.data),
                    "tb_fit_effects")
        models = []
        for i in range(P):
            a, b = int(off[i]), int(off[i + 1])
            k = b - a
            gblup = mode == MODE_GBLUP or (mode == MODE_AUTO and k > self.n)
            models.append(PanelModel(flat[a:b], centre[a:b], effects[a:b], intercept[i],
                                     "gblup" if gblup else "snp_blup", h2, fitness[i]))
        return models

    def predict(self, models, animals):
        """Breeding values of ``animals`` (original indices of this context's data set) under each model:
        array (len(models), len(animals)).  The models may come from another context holding the same markers."""
        flat, off = pack_genomes([mdl.markers for mdl in models], self.m)
        centre = np.ascontiguousarray(np.concatenate([mdl.centre for mdl in models]), dtype=np.float64)
        effects = np.ascontiguousarray(np.concatenate([mdl.effects for mdl in models]), dtype=np.float64)
        intercept = np.ascontiguousarray([mdl.intercept for mdl in models], dtype=np.float64)
        a = np.ascontiguousarray(np.asarray(animals, dtype=np.int32).ravel())
        out = np.empty((len(models), a.size), dtype=np.float64)
        self._check(self._lib.tb_predict_effects(self._ctx, flat.ctypes.data, off.ctypes.data, len(models),
                                                 centre.ctypes.data, effects.ctypes.data, intercept.ctypes.data,
                                                 a.ctypes.data, a.size, out.ctypes.data), "tb_predict_effects")
        return out

    # -- REML heritability --------------------------------------------------------------------------
    def reml_profile(self, genomes, h2, slot=0, mode=MODE_AUTO):
        """Restricted log-likelihood of each genome's model on row set ``slot`` at heritabilities ``h2``: one list
        (G,) shared by every genome, or (P, G), one list per genome.  Returns arrays (P, G) of l, sigma_g^2 and mu
        (include/tblup_b200.h, tb_reml_profile, states the model).  Always fp64, whatever ``set_precision`` says; a
        point whose factorisation fails is NaN.  The genomes become the staged batch (``stage``)."""
        flat, off = pack_genomes(genomes, self.m)
        P = off.size - 1
        h = np.ascontiguousarray(np.asarray(h2, dtype=np.float64))
        if h.ndim == 1:
            per_genome = 0
        elif h.ndim == 2 and h.shape[0] == P:
            per_genome = 1
        else:
            raise ValueError("h2 must be one list of values or one list per genome, got shape %r for %d genomes"
                             % (h.shape, P))
        G = h.shape[-1]
        self.stage(flat=flat, off=off)
        out = np.empty((3, P, G), dtype=np.float64)
        self._check(self._lib.tb_reml_profile(self._ctx, int(slot), int(mode), h.ctypes.data, G, per_genome,
                                              out[0].ctypes.data, out[1].ctypes.data, out[2].ctypes.data),
                    "tb_reml_profile")
        return out[0], out[1], out[2]

    def estimate_h2(self, genomes, slot=0, mode=MODE_AUTO, tol=1e-4, bounds=(0.01, 0.99)):
        """REML estimate of h2 for each genome on row set ``slot``: a list of ``reml.H2Estimate`` (the search is
        described in ``tblup_b200.reml``)."""
        from .reml import estimate_h2
        return estimate_h2(self, genomes, slot=slot, mode=mode, tol=tol, bounds=bounds)

    # -- per-marker statistics (top-SNPs seeder, tblup/seeder.py:144-160) ------------------------
    def marker_stats(self, animals, weights):
        """(sum_x, sum_xx, sum_xw) per marker over the listed animals (original indices), weights one per animal."""
        a = np.ascontiguousarray(np.asarray(animals, dtype=np.int32))
        w = np.ascontiguousarray(np.asarray(weights, dtype=np.float64))
        if a.shape != w.shape:
            raise ValueError("one weight per listed animal")
        out = np.empty((3, self.m), dtype=np.float64)
        self._check(self._lib.tb_marker_stats(self._ctx, a.ctypes.data, a.size, w.ctypes.data, out[0].ctypes.data,
                                              out[1].ctypes.data, out[2].ctypes.data), "tb_marker_stats")
        return out[0], out[1], out[2]

    # -- knockout local search (tblup/local.py:50-76) -------------------------------------------
    def knockout(self, genome, start_fitness, slot=0, h2=0.4, mode=MODE_AUTO):
        """Greedy knockout of the reference's ``KnockoutLocalSearch.search``: returns (keep mask, best fitness,
        evaluations consumed, batched passes)."""
        flat, _ = pack_genomes([genome], self.m)
        keep = np.ones(flat.size, dtype=np.uint8)
        best, n_ev, n_b = C.c_double(0.0), C.c_int32(0), C.c_int32(0)
        self._check(self._lib.tb_knockout(self._ctx, flat.ctypes.data, flat.size, int(slot), float(h2), int(mode),
                                          float(start_fitness), keep.ctypes.data, C.byref(best), C.byref(n_ev),
                                          C.byref(n_b)), "tb_knockout")
        return keep.astype(bool), float(best.value), int(n_ev.value), int(n_b.value)

    def knockout_scan(self, genome, slot=0, h2=0.4, mode=MODE_AUTO):
        """Fitness of every leave-one-out list of ``genome`` (one batched pass per 1 024 markers)."""
        flat, _ = pack_genomes([genome], self.m)
        out = np.empty(flat.size, dtype=np.float64)
        self._check(self._lib.tb_knockout_scan(self._ctx, flat.ctypes.data, flat.size, int(slot), float(h2), int(mode),
                                               out.ctypes.data), "tb_knockout_scan")
        return out

    # -- diagnostics ---------------------------------------------------------------------------
    def gram_debug(self, indices, rows, impl="tc"):
        flat, _ = pack_genomes([indices], self.m)
        out = np.empty((rows, rows), dtype=np.int32)
        self._check(self._lib.tb_gram_debug(self._ctx, flat.ctypes.data, flat.size, int(rows),
                                            {"tc": 0, "simt": 1, "fp4": 2, "tc_pair": 3, "fp4_pair": 4, "tc_cg2": 5, "fp4_cg2": 6}[impl], out.ctypes.data), "tb_gram_debug")
        return out

    def debug_dims(self, job=0):
        d = np.zeros(4, dtype=np.int32)
        self._check(self._lib.tb_debug_fetch(self._ctx, DBG_DIMS, job, d.ctypes.data, d.nbytes), "tb_debug_fetch")
        return dict(rpad=int(d[0]), ntp=int(d[1]), n_v=int(d[2]), kstride=int(d[3]))

    def debug_fetch(self, what, job=0):
        d = self.debug_dims(job)
        shape, dt = {
            DBG_C: ((d["rpad"], d["rpad"]), np.int32),
            DBG_S: ((d["rpad"],), np.int64),
            DBG_SQ: ((2,), np.int64),
            DBG_M: ((d["ntp"] + d["n_v"], d["ntp"]), np.float64),
            DBG_ALPHA: ((d["ntp"],), np.float64),
            DBG_PRED: ((d["n_v"],), np.float64),
            DBG_L32: ((d["ntp"], d["ntp"]), np.float32),
            DBG_SWEEPS: ((1,), np.int32),
        }[what]
        out = np.empty(shape, dtype=dt)
        self._check(self._lib.tb_debug_fetch(self._ctx, what, job, out.ctypes.data, out.nbytes), "tb_debug_fetch")
        return out

    def stage_times(self):
        ms = np.zeros(len(STAGES), dtype=np.float64)
        ln = np.zeros(len(STAGES), dtype=np.uint64)
        self._check(self._lib.tb_stage_times(self._ctx, ms.ctypes.data, ln.ctypes.data), "tb_stage_times")
        return {s: (float(ms[i]), int(ln[i])) for i, s in enumerate(STAGES)}

    def launch_count(self):
        return int(self._lib.tb_launch_count(self._ctx))

    def reset_counters(self):
        self._check(self._lib.tb_reset_counters(self._ctx), "tb_reset_counters")

    def set_stream(self, cuda_stream_handle):
        """Run on a caller-owned stream (pass ``torch.cuda.current_stream().cuda_stream``); None restores."""
        self._check(self._lib.tb_set_stream(self._ctx, C.c_void_p(int(cuda_stream_handle or 0))), "tb_set_stream")

    def microbench(self, which=0):
        out = C.c_double(0.0)
        self._check(self._lib.tb_microbench(self._ctx, int(which), C.byref(out)), "tb_microbench")
        return float(out.value)

    def set_precision(self, mode):
        """'mixed' (default): TF32 tensor-core Cholesky as preconditioner + fp64 refinement against the exact integer
        operator; 'fp64': fp64 Cholesky throughout."""
        self.set_option("precision", {"mixed": PRECISION_MIXED, "fp64": PRECISION_FP64}[mode])

    def last_precision(self):
        return {0: "mixed", 1: "fp64"}[int(self._lib.tb_last_precision(self._ctx))]

    def info(self, name):
        """Facts about the last evaluation: 'last_c16', 'last_fused_scale', 'last_mixed', 'last_wave', 'storage'."""
        v = C.c_longlong(0)
        if self._lib.tb_get_info(self._ctx, name.encode(), C.byref(v)) != 0:
            raise KeyError(name)
        return int(v.value)

    def staged_offsets(self):
        """Offsets (P + 1) of the ragged batch currently staged on the device."""
        P = self.info("staged")
        off = np.zeros(P + 1, dtype=np.int64)
        self._check(self._lib.tb_staged_offsets(self._ctx, off.ctypes.data, off.size), "tb_staged_offsets")
        return off

    def resident_genotype_bytes(self):
        b = C.c_uint64(0)
        self._check(self._lib.tb_storage_info(self._ctx, None, C.byref(b)), "tb_storage_info")
        return int(b.value)

    def last_wave(self):
        return int(self._lib.tb_last_wave(self._ctx))
