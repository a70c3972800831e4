"""ctypes binding of include/goldpolish_b200.h (no compute here)."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

BF_BYTES = 524288       # src/goldpolish_targeted_bfs.cpp:271
CBF_BYTES = 10485760    # src/goldpolish_targeted_bfs.cpp:270
DEFAULT_KS = (32, 28, 24, 20)  # scripts/goldpolish:189-190
GP_MAX_K = 8

_HERE = os.path.dirname(os.path.abspath(__file__))


def lib_path() -> str:
    """The CUDA library built in-tree (GP_LIB_PATH: another build of it, for A/B experiments)."""
    return os.environ.get("GP_LIB_PATH") or os.path.join(_HERE, "libgoldpolish_b200.so")


class GpError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"goldpolish_b200 error {code}: {msg}")
        self.code = code


class _Config(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("device", C.c_int32), ("nk", C.c_uint32),
                ("k", C.c_uint32 * GP_MAX_K), ("max_insertions", C.c_uint32), ("max_deletions", C.c_uint32),
                ("mode", C.c_int32), ("mask", C.c_int32), ("missing_ratio", C.c_float),
                ("edit_ratio", C.c_float), ("jump", C.c_uint32), ("min_contig_len", C.c_uint32),
                ("max_resident_batches", C.c_uint32), ("use_ratio", C.c_int32),
                ("missing_threshold", C.c_float), ("edit_threshold", C.c_float), ("keep_counters", C.c_int32),
                ("prep_mode", C.c_int32), ("prep_k", C.c_uint32), ("to_upper", C.c_int32),
                ("max_resident_filters", C.c_uint32), ("track_edits", C.c_int32),
                ("kmer_support", C.c_int32)]


class _Stats(C.Structure):
    _fields_ = [("kmer_ops", C.c_uint64), ("serial_kmers", C.c_uint64), ("triggers", C.c_uint64),
                ("edits", C.c_uint64), ("masked", C.c_uint64), ("rollbacks", C.c_uint64),
                ("build_ms", C.c_float), ("polish_ms", C.c_float), ("pack_ms", C.c_float),
                ("build_kernel_ms", C.c_float), ("edit_kernel_ms", C.c_float),
                ("build_launches", C.c_uint32), ("polish_launches", C.c_uint32), ("pack_launches", C.c_uint32),
                ("build_kernel", C.c_uint32), ("build_slots", C.c_uint32), ("polish_reruns", C.c_uint32),
                ("edit_sms", C.c_uint32), ("level_time_bits", C.c_uint32)]


READ_ENTRY_DTYPE = np.dtype([("read_id", np.uint32), ("kmer_threshold", np.uint32)])
EDIT_DTYPE = np.dtype([("pos", np.uint32), ("ref_len", np.uint32), ("alt_len", np.uint32), ("type", np.uint32),
                       ("allele_off", np.uint64)])  # gp_edit
UNSUPPORTED_DTYPE = np.dtype([("start", np.uint32), ("end", np.uint32), ("kmers", np.uint32)])  # gp_unsupported_run
EDIT_TYPES = ("SNV", "MNV", "INS", "DEL", "COMPLEX")  # GP_EDIT_SNV .. GP_EDIT_COMPLEX
EDIT_INSERTED = 0xFFFFFFFF  # GP_EDIT_INSERTED

_lib = None

EXPORTS = ["gp_default_config", "gp_ctx_create", "gp_ctx_destroy", "gp_last_error", "gp_ctx_set_stream",
           "gp_ctx_synchronize", "gp_get_stats", "gp_reads_upload", "gp_build_filters", "gp_build_stage",
           "gp_build_run", "gp_build_fetch", "gp_build_fetch_cbf", "gp_filters_load", "gp_polish",
           "gp_polish_stage", "gp_polish_run", "gp_polish_fetch", "gp_kmer_threshold", "gp_mappings_cap",
           "gp_guard_rejects", "gp_roof_microbench", "gp_build_round_times", "gp_pipeline_run", "gp_prep", "gp_build_output_host", "gp_host_alloc", "gp_host_free",
           "gp_build_cta_times", "gp_flagged_bed", "gp_debug_nthash", "gp_reads_begin", "gp_reads_append", "gp_reads_end",
           "gp_polish_fetch_edits", "gp_polish_fetch_support", "gp_polish_fetch_unsupported"]


def load_library():
    """Load libgoldpolish_b200.so; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    p = lib_path()
    if not os.path.exists(p):
        raise ImportError(f"{p} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "or `make -C goldpolish_b200/csrc`; goldpolish_b200 has no CPU fallback")
    l = C.CDLL(p)
    vp, u32, u64 = C.c_void_p, C.c_uint32, C.c_uint64
    l.gp_default_config.argtypes = [C.POINTER(_Config)]
    l.gp_default_config.restype = None
    l.gp_ctx_create.argtypes = [C.POINTER(_Config), C.POINTER(vp)]
    l.gp_ctx_destroy.argtypes = [vp]
    l.gp_ctx_destroy.restype = None
    l.gp_last_error.argtypes = [vp]
    l.gp_last_error.restype = C.c_char_p
    l.gp_ctx_set_stream.argtypes = [vp, vp]
    l.gp_ctx_synchronize.argtypes = [vp]
    l.gp_get_stats.argtypes = [vp, C.POINTER(_Stats)]
    l.gp_reads_upload.argtypes = [vp, vp, vp, u64]
    l.gp_build_filters.argtypes = [vp, u32, vp, vp, vp]
    l.gp_build_stage.argtypes = [vp, u32, vp, vp]
    l.gp_build_run.argtypes = [vp]
    l.gp_build_fetch.argtypes = [vp, vp]
    l.gp_build_fetch_cbf.argtypes = [vp, u32, u32, vp]
    l.gp_filters_load.argtypes = [vp, u32, vp]
    l.gp_polish.argtypes = [vp, u32, vp, vp, vp, vp, u64, vp, vp]
    l.gp_polish_stage.argtypes = [vp, u32, vp, vp, vp]
    l.gp_polish_run.argtypes = [vp]
    l.gp_polish_fetch.argtypes = [vp, vp, u64, vp, vp]
    l.gp_kmer_threshold.argtypes = [u64]
    l.gp_kmer_threshold.restype = C.c_int
    l.gp_mappings_cap.argtypes = [u64, C.c_double]
    l.gp_mappings_cap.restype = u64
    l.gp_guard_rejects.argtypes = [u64, u64]
    l.gp_guard_rejects.restype = C.c_int
    l.gp_roof_microbench.argtypes = [vp, u32, u32, u64, C.POINTER(C.c_double), C.POINTER(C.c_float)]
    l.gp_build_round_times.argtypes = [vp, C.POINTER(u64)]
    l.gp_pipeline_run.argtypes = [vp]
    l.gp_reads_begin.argtypes = [vp, u64, vp]
    l.gp_reads_append.argtypes = [vp, vp, u64]
    l.gp_reads_end.argtypes = [vp]
    l.gp_debug_nthash.argtypes = [vp, u64, u32, vp, vp, u64, C.POINTER(u64)]
    l.gp_flagged_bed.argtypes = [vp, vp, u32, vp, vp, vp, u64]
    l.gp_flagged_bed.restype = u64
    l.gp_build_cta_times.argtypes = [vp, vp, u32, C.POINTER(u32)]
    l.gp_build_output_host.argtypes = [vp, vp]
    l.gp_host_alloc.argtypes = [u64]
    l.gp_host_alloc.restype = vp
    l.gp_host_free.argtypes = [vp]
    l.gp_host_free.restype = None
    l.gp_prep.argtypes = [vp, u32, vp, vp, C.c_int32, u32, C.c_int32, vp, u64, vp]
    l.gp_polish_fetch_edits.argtypes = [vp, vp, vp, u64, vp, u64, vp]
    l.gp_polish_fetch_support.argtypes = [vp, vp, vp]
    l.gp_polish_fetch_unsupported.argtypes = [vp, vp, vp, u64, vp]
    _lib = l
    return l


def kmer_threshold(mappings_bases: int) -> int:
    return load_library().gp_kmer_threshold(int(mappings_bases))


def mappings_cap(target_len: int, subsample_max_per_10kbp: float) -> int:
    return int(load_library().gp_mappings_cap(int(target_len), float(subsample_max_per_10kbp)))


def guard_rejects(input_bytes: int, output_bytes: int) -> bool:
    return bool(load_library().gp_guard_rejects(int(input_bytes), int(output_bytes)))


def flagged_bed(seqs, offsets, names=None):
    """Flagged (soft-masked, ntedit.cpp:1131-1146) regions of polished records as BED rows (name, start, end):
    one per maximal run of lower-case letters, 0-based half-open.  `names` defaults to the record indices."""
    l = load_library()
    off = np.ascontiguousarray(offsets, dtype=np.uint64)
    n = len(off) - 1
    cap = 1024
    while True:
        rec = np.zeros(cap, dtype=np.uint32)
        st = np.zeros(cap, dtype=np.uint64)
        en = np.zeros(cap, dtype=np.uint64)
        got = int(l.gp_flagged_bed(_ptr(seqs), _ptr(off), n, _ptr(rec), _ptr(st), _ptr(en), cap))
        if got <= cap:
            break
        cap = got
    return [((names[int(rec[i])] if names is not None else int(rec[i])), int(st[i]), int(en[i])) for i in range(got)]


def _ptr(a):
    """Device-independent pointer of a numpy array or a torch CPU tensor (pinned or not)."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        if not a.flags["C_CONTIGUOUS"]:
            raise ValueError("array must be C-contiguous")
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        if a.is_cuda or not a.is_contiguous():
            raise ValueError("tensor must be a contiguous host tensor")
        return a.data_ptr()
    raise TypeError(type(a))


class Context:
    """One gp_ctx (one GPU).  Mirrors the two reference tools of the hot path:
    ``build_filters`` == goldpolish-targeted-bfs' serve_batch, ``polish`` == goldpolish-ntedit."""

    def __init__(self, device: int = 0, ks=DEFAULT_KS, max_insertions=5, max_deletions=5, mode=1, mask=1,
                 missing_ratio=0.5, edit_ratio=0.5, jump=3, min_contig_len=100, max_resident_batches=0,
                 keep_counters=0, prep_mode=0, prep_k=0, to_upper=0, max_resident_filters=0, track_edits=False,
                 kmer_support=False):
        self._l = load_library()
        cfg = _Config()
        self._l.gp_default_config(C.byref(cfg))
        cfg.device = device
        cfg.nk = len(ks)
        for i, k in enumerate(ks):
            cfg.k[i] = k
        cfg.max_insertions, cfg.max_deletions, cfg.mode, cfg.mask = max_insertions, max_deletions, mode, mask
        cfg.missing_ratio, cfg.edit_ratio, cfg.jump, cfg.min_contig_len = missing_ratio, edit_ratio, jump, min_contig_len
        cfg.max_resident_batches = max_resident_batches
        cfg.keep_counters = keep_counters
        cfg.prep_mode, cfg.prep_k, cfg.to_upper = prep_mode, prep_k, to_upper
        cfg.max_resident_filters = max_resident_filters
        cfg.track_edits = 1 if track_edits else 0
        cfg.kmer_support = 1 if kmer_support else 0
        h = C.c_void_p()
        rc = self._l.gp_ctx_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise GpError(rc, self._l.gp_last_error(None).decode())
        self._h = h
        self.ks = tuple(ks)
        self.nk = len(ks)
        self.n_batches = 0

    def close(self):
        if getattr(self, "_h", None):
            self._l.gp_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc):
        if rc != 0:
            raise GpError(rc, self._l.gp_last_error(self._h).decode())

    def set_stream(self, cuda_stream: int | None):
        self._ck(self._l.gp_ctx_set_stream(self._h, C.c_void_p(cuda_stream or 0)))

    def synchronize(self):
        self._ck(self._l.gp_ctx_synchronize(self._h))

    def stats(self) -> dict:
        s = _Stats()
        self._ck(self._l.gp_get_stats(self._h, C.byref(s)))
        return {n: getattr(s, n) for n, _ in _Stats._fields_}

    # ---- reads ----
    def upload_reads(self, seqs, offsets):
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        self._keep = (seqs, offsets)
        self._ck(self._l.gp_reads_upload(self._h, _ptr(seqs), _ptr(offsets), len(offsets) - 1))

    def upload_reads_piecewise(self, lens, pieces):
        """gp_reads_begin / gp_reads_append / gp_reads_end: `lens` = all read lengths, `pieces` = iterable of
        (uint8 array of the bases of consecutive reads back to back, number of reads in it)."""
        lens = np.ascontiguousarray(lens, dtype=np.uint32)
        self._ck(self._l.gp_reads_begin(self._h, len(lens), _ptr(lens)))
        for seqs, n in pieces:
            seqs = np.ascontiguousarray(seqs, dtype=np.uint8)
            self._ck(self._l.gp_reads_append(self._h, _ptr(seqs) if seqs.size else None, int(n)))
        self._ck(self._l.gp_reads_end(self._h))

    # ---- filter build ----
    def build_stage(self, batch_entry_off, entries):
        off = np.ascontiguousarray(batch_entry_off, dtype=np.uint64)
        ent = np.ascontiguousarray(entries, dtype=READ_ENTRY_DTYPE)
        self.n_batches = len(off) - 1
        self._ck(self._l.gp_build_stage(self._h, self.n_batches, _ptr(off), _ptr(ent)))

    def build_run(self):
        self._ck(self._l.gp_build_run(self._h))

    def build_output(self, pinned):
        """Name a page-locked host buffer (e.g. a torch pinned tensor) that the build kernel fills with the filter
        payloads as they become final; build_fetch(out=<same buffer>) then only synchronises.  None: off."""
        self._bf_pinned = pinned
        self._ck(self._l.gp_build_output_host(self._h, _ptr(pinned) if pinned is not None else None))

    def build_fetch(self, out=None, want=True):
        if want and out is None:
            out = np.empty((self.n_batches, self.nk, BF_BYTES), dtype=np.uint8)
        self._ck(self._l.gp_build_fetch(self._h, _ptr(out) if want else None))
        return out if want else None

    def build_filters(self, batch_entry_off, entries, fetch=True, out=None):
        self.build_stage(batch_entry_off, entries)
        self.build_run()
        return self.build_fetch(out=out, want=fetch)

    def fetch_cbf(self, batch: int, k_index: int) -> np.ndarray:
        out = np.empty(CBF_BYTES, dtype=np.uint8)
        self._ck(self._l.gp_build_fetch_cbf(self._h, batch, k_index, _ptr(out)))
        return out

    def load_filters(self, payloads):
        payloads = np.ascontiguousarray(payloads, dtype=np.uint8)
        n = payloads.size // (self.nk * BF_BYTES)
        if n * self.nk * BF_BYTES != payloads.size:
            raise ValueError("payloads must be n_batches * nk * 524288 bytes")
        self.n_batches = n
        self._ck(self._l.gp_filters_load(self._h, n, _ptr(payloads)))

    # ---- polish ----
    def polish_stage(self, seqs, offsets, contig_batch):
        off = np.ascontiguousarray(offsets, dtype=np.uint64)
        cb = np.ascontiguousarray(contig_batch, dtype=np.uint32)
        self._n_contigs = len(off) - 1
        self._in_bases = int(off[-1])
        self._ck(self._l.gp_polish_stage(self._h, self._n_contigs, _ptr(seqs), _ptr(off), _ptr(cb)))

    def polish_run(self):
        self._ck(self._l.gp_polish_run(self._h))

    def pipeline_run(self):
        """build_run + polish_run of the staged work as one overlapped pass (gp_pipeline_run)."""
        self._ck(self._l.gp_pipeline_run(self._h))

    def polish_fetch(self, out=None):
        n = self._n_contigs
        out_off = np.zeros(n + 1, dtype=np.uint64)
        dropped = np.zeros(max(n, 1), dtype=np.uint8)
        if out is None:
            out = np.empty(self._in_bases + self._in_bases // 4 + 65536, dtype=np.uint8)
        rc = self._l.gp_polish_fetch(self._h, _ptr(out), out.nbytes if isinstance(out, np.ndarray) else out.numel(),
                                     _ptr(out_off), _ptr(dropped))
        if rc == -1 and int(out_off[n]) > (out.nbytes if isinstance(out, np.ndarray) else out.numel()):
            out = np.empty(int(out_off[n]), dtype=np.uint8)
            rc = self._l.gp_polish_fetch(self._h, _ptr(out), out.nbytes, _ptr(out_off), _ptr(dropped))
        self._ck(rc)
        return out, out_off, dropped[:n]

    def polish(self, seqs, offsets, contig_batch, out=None):
        self.polish_stage(seqs, offsets, contig_batch)
        self.polish_run()
        return self.polish_fetch(out=out)

    def polish_fetch_edits(self) -> dict:
        """Edit records of the last polish (needs Context(track_edits=True)), see gp_polish_fetch_edits: a dict of
        numpy arrays -- "offsets" (n_contigs + 1, records of contig c at [offsets[c], offsets[c + 1])), "pos" (0-based
        draft position), "ref_len", "alt_len", "type" (index into EDIT_TYPES), "allele_off" and "alleles" (uint8:
        REF then ALT of record r at alleles[allele_off[r]:])."""
        off = np.zeros(getattr(self, "_n_contigs", 0) + 1, dtype=np.uint64)
        need = np.zeros(2, dtype=np.uint64)
        rc = self._l.gp_polish_fetch_edits(self._h, _ptr(off), None, 0, None, 0, _ptr(need))
        if rc == -1 and need.any():
            recs = np.zeros(max(int(need[0]), 1), dtype=EDIT_DTYPE)
            alleles = np.zeros(max(int(need[1]), 1), dtype=np.uint8)
            rc = self._l.gp_polish_fetch_edits(self._h, _ptr(off), _ptr(recs), len(recs), _ptr(alleles), alleles.size,
                                               _ptr(need))
        else:
            recs, alleles = np.zeros(0, dtype=EDIT_DTYPE), np.zeros(0, dtype=np.uint8)
        self._ck(rc)
        recs, alleles = recs[:int(need[0])], alleles[:int(need[1])]
        return {"offsets": off, "pos": recs["pos"].copy(), "ref_len": recs["ref_len"].copy(),
                "alt_len": recs["alt_len"].copy(), "type": recs["type"].copy(), "allele_off": recs["allele_off"].copy(),
                "alleles": alleles}

    def polish_fetch_support(self):
        """k-mer support of the last polish (needs Context(kmer_support=True)), see gp_polish_fetch_support:
        (counts[n_contigs, nk, 4] uint64 -- draft k-mers, draft present, polished k-mers, polished present --,
        filter_bits_set[n_batches, nk] uint64)."""
        n = getattr(self, "_n_contigs", 0)
        counts = np.zeros((max(n, 1), self.nk, 4), dtype=np.uint64)
        bits = np.zeros((max(self.n_batches, 1), self.nk), dtype=np.uint64)
        self._ck(self._l.gp_polish_fetch_support(self._h, _ptr(counts), _ptr(bits)))
        return counts[:n], bits[:self.n_batches]

    def polish_fetch_unsupported(self) -> dict:
        """Runs of unsupported k-mers of the last polish (needs Context(kmer_support=True)), see
        gp_polish_fetch_unsupported: a dict of numpy arrays -- "offsets" (uint64 [n_contigs, 2, nk]: the first run of
        contig c, record r (0 draft, 1 polished) and k index j), "run_off" (the same n_contigs * 2 * nk + 1 offsets flat:
        runs of segment i at [run_off[i], run_off[i + 1])), "start", "end" (0-based, half-open) and "kmers" (uint32)."""
        n = getattr(self, "_n_contigs", 0)
        off = np.zeros(n * 2 * self.nk + 1, dtype=np.uint64)
        need = np.zeros(1, dtype=np.uint64)
        rc = self._l.gp_polish_fetch_unsupported(self._h, _ptr(off), None, 0, _ptr(need))
        runs = np.zeros(0, dtype=UNSUPPORTED_DTYPE)
        if rc == -1 and need[0]:
            runs = np.zeros(int(need[0]), dtype=UNSUPPORTED_DTYPE)
            rc = self._l.gp_polish_fetch_unsupported(self._h, _ptr(off), _ptr(runs), len(runs), _ptr(need))
        self._ck(rc)
        return {"offsets": off[:-1].reshape(n, 2, self.nk), "run_off": off, "start": runs["start"].copy(),
                "end": runs["end"].copy(), "kmers": runs["kmers"].copy()}

    # ---- goldpolish-mask / goldpolish-to-upper alone ----
    def prep(self, seqs, offsets, mode: int, k: int = 0, to_upper: int = 0):
        """mode 1 = `goldpolish-mask -s -k K`, 2 = `-n`, 0 = to-upper only.  Returns (bytes array, offsets)."""
        off = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = len(off) - 1
        out = np.empty(int(off[-1]) + n + 16, dtype=np.uint8)
        out_off = np.zeros(n + 1, dtype=np.uint64)
        self._ck(self._l.gp_prep(self._h, n, _ptr(seqs), _ptr(off), mode, k, to_upper, _ptr(out), out.nbytes, _ptr(out_off)))
        return out, out_off

    # ---- measurement ----
    def build_round_times(self):
        """Level-synchronous build kernel, CTA 0: {interval kind: (barrier wait ms, work ms, intervals)}."""
        out = (C.c_uint64 * 32)()
        self._ck(self._l.gp_build_round_times(self._h, out))
        r = {n: (out[3 * i] / 1e6, out[3 * i + 1] / 1e6, int(out[3 * i + 2])) for i, n in enumerate(self.INTERVAL_KINDS)}
        r["list_entries"] = int(out[31])
        return r

    INTERVAL_KINDS = ("clear", "round0", "level1", "late", "round0+late", "level1+late")

    def debug_nthash(self, read_id: int, k: int):
        """(positions, hashes[n, 4]) of the valid k-mers of an uploaded read, as the device computes them."""
        n = C.c_uint64()
        cap = 1 << 16
        while True:
            hs = np.zeros((cap, 4), dtype=np.uint64)
            valid = np.zeros(cap, dtype=np.uint8)
            rc = self._l.gp_debug_nthash(self._h, read_id, k, _ptr(hs), _ptr(valid), cap, C.byref(n))
            if rc == -1 and n.value > cap:
                cap = n.value
                continue
            self._ck(rc)
            break
        pos = np.nonzero(valid[:n.value])[0]
        return pos, hs[pos]

    def build_cta_times(self) -> np.ndarray:
        """[n_ctas, 6 kinds, 3] ns / counts of every CTA (needs GP_LEVEL_CTA_TIMES=1 during the build)."""
        out = np.zeros((1024, 32), dtype=np.uint64)
        n = C.c_uint32()
        self._ck(self._l.gp_build_cta_times(self._h, _ptr(out), 1024, C.byref(n)))
        return out[:n.value, :18].reshape(n.value, 6, 3)

    def roof_microbench(self, warps: int, iters: int, region_bytes: int = CBF_BYTES):
        sps, ms = C.c_double(), C.c_float()
        self._ck(self._l.gp_roof_microbench(self._h, warps, iters, region_bytes, C.byref(sps), C.byref(ms)))
        return sps.value, ms.value
