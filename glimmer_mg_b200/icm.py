"""ctypes host mirror of the reference's ICM operator surface over libgmgicm.so.

Names follow the reference (``/root/reference/src/ICM/icm.hh``): ``ICM.Read`` / ``Output`` /
``Score_String`` / ``Cumulative_Score`` / ``Frame_Score`` / ``Full_Window_Prob`` /
``Partial_Window_Prob`` / ``Build_Indep_WO_Stops``; ``ICMTraining.Train_Model``.  The batched calls
(``SeqSet.score_all_frames`` = ``Score_All_Frames`` glimmer-mg.cc:1468, ``find_orfs`` = ``Find_Orfs``
glimmer_base.cc:638, ``score_orfs_mg`` = ``Score_Orfs_Errors`` glimmer-mg.cc:1605, ``score_orfs_g3`` =
``Score_Orfs`` glimmer3.cc:1275) are the device-side equivalents of the drivers' scoring half.

Errors: the reference prints to stderr and exits (icm.cc:635-657); here every failing C-ABI call raises
:class:`GmgError` with the same message text.
"""
import ctypes as C
import os
import re

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))


class GmgError(RuntimeError):
    pass


def lib_path():
    return os.path.join(_HERE, "libgmgicm.so")


class _Params(C.Structure):
    _fields_ = [("min_gene_len", C.c_int32), ("allow_truncated", C.c_int32), ("allow_indels", C.c_int32),
                ("allow_subs", C.c_int32), ("min_indel_orf_len", C.c_int32),
                ("indel_quality_threshold", C.c_int32), ("indel_max", C.c_int32), ("ignore_score_len", C.c_int32),
                ("indel_suffix_score_threshold", C.c_double), ("have_quality_file", C.c_int32),
                ("n_start", C.c_int32), ("n_stop", C.c_int32), ("start_codon", (C.c_char * 4) * 8),
                ("stop_codon", (C.c_char * 4) * 8)]


class _EventModel(C.Structure):
    _fields_ = [("prior", C.c_double), ("start_threshold", C.c_double), ("event_threshold", C.c_double),
                ("pwm_bonus_max", C.c_double), ("n_start", C.c_int32), ("start_lo", C.c_double * 8),
                ("n_class", C.c_int32), ("n_len", C.c_int32), ("len_lo", C.c_void_p), ("seq_class", C.c_void_p)]


ORF_DTYPE = np.dtype([("frame", "<i4"), ("stop_position", "<i4"), ("orf_len", "<i4"), ("gene_len", "<i4")])
START_DTYPE = np.dtype([("j", "<i4"), ("pos", "<i4"), ("score", "<f8"), ("which", "<i4"), ("truncated", "<i4"),
                        ("first", "<i4"), ("n_err", "<i4"), ("err_pos", "<i4", (2,)), ("err_type", "<i4", (2,))])
assert START_DTYPE.itemsize == 48 and ORF_DTYPE.itemsize == 16

ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p)

_lib = None


def lib():
    """Load libgmgicm.so.  Fails loudly when the CUDA extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise GmgError(f"{path} not found: build it with `make -C glimmer_mg_b200/csrc` "
                       "(or __graft_entry__.build()); there is no CPU fallback")
    L = C.CDLL(path)
    vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int
    P = C.POINTER
    sig = {
        "gmg_abi_version": (i32, []),
        "gmg_last_error": (C.c_char_p, []),
        "gmg_ctx_create": (i32, [i32, vp, P(vp)]),
        "gmg_ctx_destroy": (None, [vp]),
        "gmg_ctx_sync": (i32, [vp]),
        "gmg_ctx_launch_count": (i64, [vp]),
        "gmg_ctx_profile": (i32, [vp, i32]),
        "gmg_ctx_profile_read": (i32, [vp, i32, P(C.c_double), P(i64)]),
        "gmg_host_alloc": (i32, [C.c_size_t, P(vp)]),
        "gmg_host_free": (None, [vp]),
        "gmg_ctx_memcpy_d2h": (i32, [vp, vp, vp, C.c_size_t]),
        "gmg_ctx_memcpy_h2d": (i32, [vp, vp, vp, C.c_size_t]),
        "gmg_params_default": (None, [P(_Params), i32]),
        "gmg_ignore_score_len": (i32, [C.c_double, P(_Params)]),
        "gmg_icm_load": (i32, [vp, C.c_char_p, P(vp)]),
        "gmg_icm_load_mem": (i32, [vp, vp, C.c_size_t, P(vp)]),
        "gmg_icm_write_mem": (i32, [vp, vp, C.c_size_t, P(C.c_size_t)]),
        "gmg_icm_from_tables": (i32, [vp, i32, i32, i32, vp, vp, P(vp)]),
        "gmg_icm_build_indep": (i32, [vp, C.c_double, P(C.c_char_p), i32, P(vp)]),
        "gmg_icm_write": (i32, [vp, C.c_char_p]),
        "gmg_icm_dims": (i32, [vp, vp]),
        "gmg_icm_tables": (i32, [vp, vp, vp]),
        "gmg_icm_mut_info": (i32, [vp, vp]),
        "gmg_icm_free": (None, [vp]),
        "gmg_seqset_create": (i32, [vp, vp, vp, i64, vp, P(vp)]),
        "gmg_seqset_create_device": (i32, [vp, vp, vp, i64, vp, P(vp)]),
        "gmg_seqset_free": (None, [vp]),
        "gmg_seqset_from_fasta": (i32, [vp, vp, i64, P(vp), P(i64)]),
        "gmg_seqset_count": (i64, [vp]),
        "gmg_seqset_offsets": (i32, [vp, vp]),
        "gmg_seqset_fasta_headers": (i32, [vp, vp, vp]),
        "gmg_quality_parse_fasta": (i32, [vp, vp, i64, P(i64), P(i64), vp, vp, i64, i64]),
        "gmg_seqset_quality_from_fasta": (i32, [vp, vp, vp, i64]),
        "gmg_seqset_from_fastq": (i32, [vp, vp, i64, i32, P(vp), P(i64)]),
        "gmg_seqset_qualities": (i32, [vp, vp]),
        "gmg_seqset_total_bases": (i64, [vp]),
        "gmg_seqset_gc_fraction": (i32, [vp, P(C.c_double)]),
        "gmg_seqset_unpack": (i32, [vp, vp]),
        "gmg_seqset_extract": (i32, [vp, vp, i64, vp, vp, vp, vp, P(vp)]),
        "gmg_icm_score_strings": (i32, [vp, vp, vp, i32, vp]),
        "gmg_icm_score_strings_many": (i32, [vp, P(vp), i32, vp, i32, vp]),
        "gmg_icm_cumulative_score": (i32, [vp, vp, vp, i32, vp]),
        "gmg_icm_frame_score": (i32, [vp, vp, vp, i32, vp]),
        "gmg_icm_full_window_prob": (i32, [vp, vp, C.c_char_p, i32, P(C.c_double)]),
        "gmg_icm_partial_window_prob": (i32, [vp, vp, i32, C.c_char_p, i32, P(C.c_double)]),
        "gmg_score_all_frames": (i32, [vp, vp, vp, vp, vp, i32]),
        "gmg_k1_score_planes": (i32, [vp, vp, vp]),
        "gmg_find_orfs": (i32, [vp, vp, P(_Params), P(i64)]),
        "gmg_get_orfs": (i32, [vp, vp, vp, vp]),
        "gmg_set_orfs": (i32, [vp, vp, vp, vp]),
        "gmg_score_orfs_g3": (i32, [vp, vp, vp, vp, P(_Params), P(i64)]),
        "gmg_score_orfs_mg": (i32, [vp, vp, vp, vp, P(_Params), P(i64)]),
        "gmg_score_orfs_mg_gc": (i32, [vp, vp, vp, vp, vp, P(_Params), P(i64)]),
        "gmg_ctx_indep_flagged": (i64, [vp]),
        "gmg_get_starts": (i32, [vp, vp, vp, vp]),
        "gmg_all_frame_scores": (i32, [vp, vp, vp, i64, vp, vp, vp, vp]),
        "gmg_reduce_starts_mg": (i32, [vp, vp, P(_Params), P(_EventModel), P(i64), P(i64)]),
        "gmg_get_reduced_starts": (i32, [vp, vp, vp, vp, vp, vp]),
        "gmg_get_orf_starts": (i32, [vp, vp, i64, vp, i64, P(i64)]),
        "gmg_uncertified_count": (i64, [vp]),
        "gmg_ordered_fallback_count": (i32, [vp, P(i64)]),
        "gmg_trainer_create": (i32, [vp, vp, i32, i32, i32, i32, P(vp)]),
        "gmg_trainer_free": (None, [vp]),
        "gmg_trainer_count_level": (i32, [vp, i32, P(vp), P(i64)]),
        "gmg_trainer_finish_level": (i32, [vp, i32]),
        "gmg_trainer_finish": (i32, [vp, P(vp)]),
        "gmg_icm_train": (i32, [vp, vp, i32, i32, i32, i32, ALLREDUCE_FN, vp, P(vp)]),
        "gmg_icm_train_sharded": (i32, [vp, vp, i32, i32, i32, i32, ALLREDUCE_FN, vp, i32, i32, i64, P(vp)]),
        "gmg_trainer_set_shard": (i32, [vp, i32, i32, i64, ALLREDUCE_FN, vp]),
        "gmg_icm_train_many": (i32, [vp, P(vp), i32, i32, i32, i32, i32, P(vp)]),
        "gmg_ctx_train_flagged": (i64, [vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)  # AttributeError = the library does not export what include/gmg_icm.h declares
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def _check(rc):
    if rc != 0:
        raise GmgError(lib().gmg_last_error().decode(errors="replace"))


class Params:
    """Options of the scoring half (glimmer-mg / glimmer3 command-line state)."""

    def __init__(self, metagenomic=True, **kw):
        self.c = _Params()
        lib().gmg_params_default(C.byref(self.c), 1 if metagenomic else 0)
        for k, v in kw.items():
            self.set(k, v)

    def set(self, k, v):
        if k in ("start_codons", "stop_codons"):
            arr = self.c.start_codon if k == "start_codons" else self.c.stop_codon
            for i, s in enumerate(v):
                arr[i].value = s.lower().encode()
            setattr(self.c, "n_start" if k == "start_codons" else "n_stop", len(v))
        else:
            setattr(self.c, k, v)

    def __getattr__(self, k):
        return getattr(self.__dict__["c"], k)

    @property
    def stop_codons(self):
        return [self.c.stop_codon[i].value.decode() for i in range(self.c.n_stop)]

    def set_ignore_score_len(self, gc):
        """Set_Ignore_Score_Len (glimmer_base.cc:2597)."""
        self.c.ignore_score_len = lib().gmg_ignore_score_len(gc, C.byref(self.c))
        return self.c.ignore_score_len


class EventModel:
    """What Add_Events_Fwd / Add_Events_Rev (glimmer_base.cc:43-235) add to a start's score, for the device-side
    start-list reduction: prior, start-codon log-odds, the gene-length log-odds table
    ``len_lo[class, truncated_5p, truncated_3p, length]`` and the two thresholds.  Defaults = glimmer-mg without a
    feature file (-u 0): length log-odds 0, default start-codon probabilities."""

    def __init__(self, prior=-1.0, start_threshold=-6.0, event_threshold=-3.0, pwm_bonus_max=0.0,
                 start_lo=None, len_lo=None, seq_class=None):
        import math
        if start_lo is None:  # Start_Dist_t(DEFAULT_START_PROB): log(p) - log(1/n) (Common/gene.cc, glimmer_base.hh:27)
            probs = (0.60, 0.30, 0.10)
            start_lo = [math.log(x) - math.log(1.0 / len(probs)) for x in probs]
        self.start_lo = [float(x) for x in start_lo]
        # default Length_Dist_t: log-odds 0 for every length (Common/gene.cc:369-382); the device wants a table that
        # covers every gene length of the batch
        self.len_lo = np.ascontiguousarray(np.zeros((1, 2, 2, 4096)) if len_lo is None else len_lo, np.float64)
        assert self.len_lo.ndim == 4 and self.len_lo.shape[1:3] == (2, 2)
        self.seq_class = None if seq_class is None else np.ascontiguousarray(seq_class, np.int32)
        self.prior, self.start_threshold, self.event_threshold = float(prior), float(start_threshold), float(event_threshold)
        self.pwm_bonus_max = float(pwm_bonus_max)

    def c(self):
        m = _EventModel()
        m.prior, m.start_threshold, m.event_threshold, m.pwm_bonus_max = (self.prior, self.start_threshold,
                                                                          self.event_threshold, self.pwm_bonus_max)
        m.n_start = len(self.start_lo)
        for i, x in enumerate(self.start_lo):
            m.start_lo[i] = x
        m.n_class, m.n_len = self.len_lo.shape[0], self.len_lo.shape[3]
        m.len_lo = self.len_lo.ctypes.data
        m.seq_class = None if self.seq_class is None else self.seq_class.ctypes.data
        return m


class Context:
    """One per GPU: device, stream, scratch.  ``stream`` may be a raw cudaStream_t (int) -- e.g.
    ``torch.cuda.current_stream().cuda_stream`` -- so that torch events bracket our kernels."""

    def __init__(self, device=0, stream=None):
        self.h = C.c_void_p()
        self._pinned = {}
        _check(lib().gmg_ctx_create(device, C.c_void_p(stream) if stream else None, C.byref(self.h)))
        self.device = device

    def sync(self):
        _check(lib().gmg_ctx_sync(self.h))

    @property
    def launches(self):
        return int(lib().gmg_ctx_launch_count(self.h))

    @property
    def indep_flagged(self):
        """model entries of the last score_orfs_mg_gc call whose logarithm the host recomputed (diagnostic)"""
        return int(lib().gmg_ctx_indep_flagged(self.h))

    PROF = {"k1": 0, "k2": 1, "k3": 2, "k4": 3, "orf": 4, "pack": 5, "fs": 6}

    def profile(self, enable=True):
        """Bracket every hot-kernel launch with CUDA events on the context's stream."""
        _check(lib().gmg_ctx_profile(self.h, 1 if enable else 0))

    def profile_read(self, kernel):
        """-> (summed device ms, launches) of one kernel class since the last read."""
        ms, n = C.c_double(), C.c_int64()
        _check(lib().gmg_ctx_profile_read(self.h, self.PROF[kernel], C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def d2h(self, dptr, count, dtype):
        out = np.zeros(count, dtype)
        _check(lib().gmg_ctx_memcpy_d2h(self.h, out.ctypes.data, C.c_void_p(dptr), out.nbytes))
        return out

    def pinned(self, name, count, dtype):
        """A page-locked host array (gmg_host_alloc) owned by the context and reused by name: D2H copies into
        it run at PCIe rate.  The returned view is overwritten by the next request for the same name."""
        dtype = np.dtype(dtype)
        need = max(1, count) * dtype.itemsize
        buf = self._pinned.get(name)
        if buf is None or buf[1] < need:
            if buf is not None:
                lib().gmg_host_free(buf[0])
            cap = need + need // 4 + 4096
            ptr = C.c_void_p()
            _check(lib().gmg_host_alloc(cap, C.byref(ptr)))
            buf = (ptr, cap, (C.c_uint8 * cap).from_address(ptr.value))
            self._pinned[name] = buf
        return np.frombuffer(buf[2], dtype=dtype, count=count)

    def close(self):
        if self.h:
            for ptr, _, _ in self._pinned.values():
                lib().gmg_host_free(ptr)
            self._pinned = {}
            lib().gmg_ctx_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _ascii_concat(seqs):
    """list of bytes/str -> (uint8 array, int64 offsets)."""
    bs = [s if isinstance(s, (bytes, bytearray)) else s.encode() for s in seqs]
    off = np.zeros(len(bs) + 1, np.int64)
    if bs:
        off[1:] = np.cumsum([len(b) for b in bs])
    data = np.frombuffer(b"".join(bs), np.uint8) if bs else np.zeros(0, np.uint8)
    return data, off


class SeqSet:
    """A batch of sequences packed 2 bits/base in HBM (Filter + lower-case applied on the device)."""

    def __init__(self, ctx, seqs=None, ascii=None, offsets=None, qual=None, device_ptr=None, device_qual=None):
        self.ctx = ctx
        self.h = C.c_void_p()
        if seqs is not None:
            ascii, offsets = _ascii_concat(seqs)
        self.off = np.ascontiguousarray(offsets, np.int64)
        self.n = len(self.off) - 1
        if device_ptr is not None:
            _check(lib().gmg_seqset_create_device(ctx.h, C.c_void_p(device_ptr), self.off.ctypes.data, self.n,
                                                  C.c_void_p(device_qual) if device_qual else None, C.byref(self.h)))
        else:
            a = np.ascontiguousarray(ascii, np.uint8)
            q = None if qual is None else np.ascontiguousarray(qual, np.uint8)
            _check(lib().gmg_seqset_create(ctx.h, a.ctypes.data, self.off.ctypes.data, self.n,
                                           None if q is None else q.ctypes.data, C.byref(self.h)))
        self.total = int(self.off[-1])
        self.n_orfs = 0
        self.n_starts = 0

    @classmethod
    def from_fasta(cls, ctx, image):
        """Parse a multi-FASTA image (bytes / uint8 array) on the device (Fasta_Read, Common/fasta.cc:236).
        The returned set has ``headers``: the header text of every record."""
        buf = np.frombuffer(image, np.uint8) if isinstance(image, (bytes, bytearray, memoryview)) else \
            np.ascontiguousarray(image, np.uint8)
        h, n = C.c_void_p(), C.c_int64()
        _check(lib().gmg_seqset_from_fasta(ctx.h, buf.ctypes.data if len(buf) else None, len(buf), C.byref(h), C.byref(n)))
        return cls._adopt(ctx, h)._read_headers(buf)

    @classmethod
    def from_fastq(cls, ctx, image, phred_offset=33):
        """Parse a FASTQ image (bytes / uint8 array; four-line records) on the device: sequences, ``headers`` (as
        ``from_fasta`` reports the same lines with '>' for '@') and per-base qualities (byte - ``phred_offset``, 33 or
        64), attached as ``set_quality_fasta`` attaches them.  Malformed input raises GmgError naming the record and
        line."""
        buf = np.frombuffer(image, np.uint8) if isinstance(image, (bytes, bytearray, memoryview)) else \
            np.ascontiguousarray(image, np.uint8)
        h, n = C.c_void_p(), C.c_int64()
        _check(lib().gmg_seqset_from_fastq(ctx.h, buf.ctypes.data if len(buf) else None, len(buf), int(phred_offset),
                                           C.byref(h), C.byref(n)))
        return cls._adopt(ctx, h)._read_headers(buf)

    def _read_headers(self, buf):
        """``headers``: the header text of every record, from the offsets into the image ``buf``."""
        ho, he = np.zeros(self.n, np.int64), np.zeros(self.n, np.int64)
        if self.n:
            _check(lib().gmg_seqset_fasta_headers(self.h, ho.ctypes.data, he.ctypes.data))
        raw = buf.tobytes()
        self.headers = [raw[a:b].decode(errors="replace") for a, b in zip(ho.tolist(), he.tolist())]
        return self

    @classmethod
    def _adopt(cls, ctx, h):
        """Wrap a set the library has just created."""
        self = cls.__new__(cls)
        self.ctx = ctx
        self.h = h
        self.n = int(lib().gmg_seqset_count(h))
        self.off = np.zeros(self.n + 1, np.int64)
        _check(lib().gmg_seqset_offsets(self.h, self.off.ctypes.data))
        self.total = int(self.off[-1])
        self.n_orfs = 0
        self.n_starts = 0
        return self

    def extract(self, seq, lo, length, strand):
        """extract (Glimmer's Util/extract.cc) on the device: region i, bases [lo[i], lo[i] + length[i]) of sequence
        seq[i] (0-based), becomes sequence i of the returned set; strand[i] = -1 takes its reverse complement, with raw
        IUPAC codes complemented before Filter as extract + build-icm do.  Regions must lie inside their sequence.  The
        result has no qualities and no headers.  ``regions_from_coords`` turns coordinate files into these arrays."""
        seq, lo, length = (np.ascontiguousarray(x, np.int32).reshape(-1) for x in (seq, lo, length))
        strand = np.ascontiguousarray(strand, np.int8).reshape(-1)
        if not len(seq) == len(lo) == len(length) == len(strand):
            raise GmgError(f"extract: {len(seq)} sequences, {len(lo)} starts, {len(length)} lengths and {len(strand)} "
                           "strands given")
        h = C.c_void_p()
        _check(lib().gmg_seqset_extract(self.ctx.h, self.h, len(seq), seq.ctypes.data, lo.ctypes.data, length.ctypes.data,
                                        strand.ctypes.data, C.byref(h)))
        return SeqSet._adopt(self.ctx, h)

    def set_quality_fasta(self, image):
        """Per-base qualities from the image of a quality file (Fasta_Qual_Vec_Read, Common/fasta.cc:115), parsed on the
        device; records must match the set's sequences in number and length."""
        buf = np.frombuffer(image, np.uint8) if isinstance(image, (bytes, bytearray, memoryview)) else \
            np.ascontiguousarray(image, np.uint8)
        _check(lib().gmg_seqset_quality_from_fasta(self.ctx.h, self.h, buf.ctypes.data if len(buf) else None, len(buf)))

    def qualities(self):
        """Per-base qualities as attached (uint8 [total]), or None when the set has none."""
        if lib().gmg_seqset_qualities(self.h, None) != 0:
            return None
        out = np.zeros(self.total, np.uint8)
        _check(lib().gmg_seqset_qualities(self.h, out.ctypes.data))
        return out

    def close(self):
        if self.h:
            if self.ctx.h:  # a set outliving its context has nothing left to free (the context owned the device)
                lib().gmg_seqset_free(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def gc_fraction(self):
        gc = C.c_double()
        _check(lib().gmg_seqset_gc_fraction(self.h, C.byref(gc)))
        return gc.value

    def unpack(self):
        out = np.zeros(self.total, np.uint8)
        _check(lib().gmg_seqset_unpack(self.h, out.ctypes.data))
        return out.tobytes()

    # ---- Score_All_Frames ----
    def score_all_frames(self, gene, indep):
        """-> list of [6, len_i] float64 arrays (Frame_Scores, glimmer-mg.cc:140,1468)."""
        out = np.zeros(6 * self.total, np.float64)
        _check(lib().gmg_score_all_frames(self.ctx.h, gene.h, indep.h, self.h, out.ctypes.data, 0))
        res = []
        for i in range(self.n):
            a, b = int(self.off[i]), int(self.off[i + 1])
            res.append(out[6 * a:6 * b].reshape(6, b - a))
        return res

    def k1_score_planes(self, gene):
        _check(lib().gmg_k1_score_planes(self.ctx.h, gene.h, self.h))

    # ---- ORFs ----
    def find_orfs(self, params):
        n = C.c_int64()
        _check(lib().gmg_find_orfs(self.ctx.h, self.h, C.byref(params.c), C.byref(n)))
        self.n_orfs = n.value
        return self.n_orfs

    def get_orfs(self, pinned=False):
        """ORF table + per-sequence offsets.  pinned=True returns views of the context's page-locked staging
        buffers (valid until the next pinned get_orfs on this context)."""
        if pinned:
            orfs = self.ctx.pinned("orfs", self.n_orfs, ORF_DTYPE)
            off = self.ctx.pinned("orf_off", self.n + 1, np.int64)
        else:
            orfs = np.zeros(self.n_orfs, ORF_DTYPE)
            off = np.zeros(self.n + 1, np.int64)
        _check(lib().gmg_get_orfs(self.ctx.h, self.h, orfs.ctypes.data, off.ctypes.data))
        return orfs, off

    def set_orfs(self, orfs, orf_off):
        orfs = np.ascontiguousarray(orfs, ORF_DTYPE)
        orf_off = np.ascontiguousarray(orf_off, np.int64)
        _check(lib().gmg_set_orfs(self.ctx.h, self.h, orfs.ctypes.data, orf_off.ctypes.data))
        self.n_orfs = int(orf_off[-1])

    # ---- scoring halves ----
    def score_orfs_g3(self, gene, indep, params):
        n = C.c_int64()
        _check(lib().gmg_score_orfs_g3(self.ctx.h, gene.h, indep.h, self.h, C.byref(params.c), C.byref(n)))
        self.n_starts = n.value
        return self.n_starts

    def score_orfs_mg(self, gene, indep, params):
        n = C.c_int64()
        _check(lib().gmg_score_orfs_mg(self.ctx.h, gene.h, indep.h, self.h, C.byref(params.c), C.byref(n)))
        self.n_starts = n.value
        return self.n_starts

    def score_orfs_mg_gc(self, gene, gc, params, ignore_score_len=None):
        """score_orfs_mg with the independent model of every sequence's own GC fraction (glimmer-mg -c): sequence i is
        scored with Build_Indep_WO_Stops(gc[i], params' stop codons) and, when given, ignore_score_len[i] in place of
        params.ignore_score_len.  Bit-identical to scoring each sequence alone that way."""
        gc = np.ascontiguousarray(gc, np.float64)
        if gc.shape != (self.n,):
            raise GmgError(f"score_orfs_mg_gc: {gc.size} GC values for {self.n} sequences")
        isl = None
        if ignore_score_len is not None:
            isl = np.ascontiguousarray(ignore_score_len, np.int32)
            if isl.shape != (self.n,):
                raise GmgError(f"score_orfs_mg_gc: {isl.size} ignore lengths for {self.n} sequences")
        n = C.c_int64()
        _check(lib().gmg_score_orfs_mg_gc(self.ctx.h, gene.h, self.h, gc.ctypes.data,
                                          isl.ctypes.data if isl is not None else None, C.byref(params.c), C.byref(n)))
        self.n_starts = n.value
        return self.n_starts

    def get_starts(self, pinned=False):
        if pinned:
            starts = self.ctx.pinned("starts", self.n_starts, START_DTYPE)
            off = self.ctx.pinned("start_off", self.n_orfs + 1, np.int64)
        else:
            starts = np.zeros(self.n_starts, START_DTYPE)
            off = np.zeros(self.n_orfs + 1, np.int64)
        _check(lib().gmg_get_starts(self.ctx.h, self.h, starts.ctypes.data, off.ctypes.data))
        return starts, off

    def all_frame_scores(self, gene, seq, lo, length):
        """All_Frame_Score (glimmer3.cc:328) of regions [lo, lo + length) of sequences `seq` -> float64 [n, 6]: columns
        0..2 the region read downwards with first-base period 0, 1, 2; 3..5 its complement read upwards."""
        seq, lo, length = (np.ascontiguousarray(x, np.int32) for x in (seq, lo, length))
        out = np.zeros((len(seq), 6), np.float64)
        _check(lib().gmg_all_frame_scores(self.ctx.h, gene.h, self.h, len(seq), seq.ctypes.data, lo.ctypes.data,
                                          length.ctypes.data, out.ctypes.data))
        return out

    # ---- start-list reduction (row a11b) ----
    def reduce_starts_mg(self, params, model):
        """Reduce the raw start lists of the last score_orfs_mg call on the device -> number of surviving records."""
        n, nf = C.c_int64(), C.c_int64()
        cm = model.c()
        _check(lib().gmg_reduce_starts_mg(self.ctx.h, self.h, C.byref(params.c), C.byref(cm), C.byref(n), C.byref(nf)))
        self.n_red = n.value
        return self.n_red

    def get_reduced_starts(self, pinned=False):
        """-> (records, first[n_orfs], count[n_orfs], status[n_orfs]); status 0 dropped, 1 reduced, 2 take the raw list."""
        if pinned:
            st = self.ctx.pinned("red_starts", self.n_red, START_DTYPE)
            first = self.ctx.pinned("red_first", self.n_orfs, np.int64)
            cnt = self.ctx.pinned("red_cnt", self.n_orfs, np.int32)
            status = self.ctx.pinned("red_status", self.n_orfs, np.uint8)
        else:
            st = np.zeros(self.n_red, START_DTYPE)
            first, cnt, status = np.zeros(self.n_orfs, np.int64), np.zeros(self.n_orfs, np.int32), np.zeros(self.n_orfs, np.uint8)
        _check(lib().gmg_get_reduced_starts(self.ctx.h, self.h, st.ctypes.data, first.ctypes.data, cnt.ctypes.data,
                                            status.ctypes.data))
        return st, first, cnt, status

    def get_orf_starts(self, orf):
        n = C.c_int64()
        _check(lib().gmg_get_orf_starts(self.ctx.h, self.h, orf, None, 0, C.byref(n)))
        out = np.zeros(n.value, START_DTYPE)
        if n.value:
            _check(lib().gmg_get_orf_starts(self.ctx.h, self.h, orf, out.ctypes.data, n.value, C.byref(n)))
        return out

    @property
    def ordered_fallbacks(self):
        n = C.c_int64()
        _check(lib().gmg_ordered_fallback_count(self.h, C.byref(n)))
        return n.value

    @property
    def uncertified(self):
        return int(lib().gmg_uncertified_count(self.h))


class ICM:
    """ICM_t (icm.hh:116-213)."""

    def __init__(self, ctx, handle=None):
        self.ctx = ctx
        self.h = handle if handle is not None else C.c_void_p()

    # -- construction --
    @classmethod
    def Read(cls, ctx, path):
        """ICM_t::Read (icm.cc:846)."""
        h = C.c_void_p()
        _check(lib().gmg_icm_load(ctx.h, os.fsencode(path), C.byref(h)))
        return cls(ctx, h)

    @classmethod
    def Input(cls, ctx, image):
        """ICM_t::Input (icm.cc:614) from the bytes of a model file."""
        buf = bytes(image)
        h = C.c_void_p()
        _check(lib().gmg_icm_load_mem(ctx.h, buf, len(buf), C.byref(h)))
        return cls(ctx, h)

    def image(self):
        """The build-icm binary form as bytes (ICM_t::Output(fp, true), icm.cc:729)."""
        n = C.c_size_t()
        _check(lib().gmg_icm_write_mem(self.h, None, 0, C.byref(n)))
        buf = C.create_string_buffer(n.value)
        _check(lib().gmg_icm_write_mem(self.h, buf, n.value, C.byref(n)))
        return buf.raw[:n.value]

    @classmethod
    def from_tables(cls, ctx, w, d, p, mip, prob):
        mip = np.ascontiguousarray(mip, np.int16)
        prob = np.ascontiguousarray(prob, np.float32)
        h = C.c_void_p()
        _check(lib().gmg_icm_from_tables(ctx.h, w, d, p, mip.ctypes.data, prob.ctypes.data, C.byref(h)))
        return cls(ctx, h)

    @classmethod
    def Build_Indep_WO_Stops(cls, ctx, gc_frac, stop_codons=("taa", "tag", "tga")):
        """ICM_t(3,2,3).Build_Indep_WO_Stops (icm.cc:65)."""
        arr = (C.c_char_p * len(stop_codons))(*[s.encode() for s in stop_codons])
        h = C.c_void_p()
        _check(lib().gmg_icm_build_indep(ctx.h, gc_frac, arr, len(stop_codons), C.byref(h)))
        return cls(ctx, h)

    def Output(self, path, binary_form=True):
        """ICM_t::Output (icm.cc:729); only the binary form exists here."""
        if not binary_form:
            raise GmgError("text-form ICM output is not implemented (debug-only in the reference)")
        _check(lib().gmg_icm_write(self.h, os.fsencode(path)))

    def close(self):
        if self.h:
            if self.ctx.h:
                lib().gmg_icm_free(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- accessors --
    def dims(self):
        d = np.zeros(4, np.int32)
        _check(lib().gmg_icm_dims(self.h, d.ctypes.data))
        return tuple(int(x) for x in d)

    def Get_Model_Len(self):
        return self.dims()[0]

    def Get_Periodicity(self):
        return self.dims()[2]

    def tables(self):
        w, d, p, n = self.dims()
        mip = np.zeros((p, n), np.int16)
        prob = np.zeros((p, n, 4), np.float32)
        _check(lib().gmg_icm_tables(self.h, mip.ctypes.data, prob.ctypes.data))
        return mip, prob

    # -- scoring surface --
    def _one(self, s):
        return SeqSet(self.ctx, seqs=[s])

    def Full_Window_Prob(self, window, frame):
        out = C.c_double()
        w = window if isinstance(window, bytes) else window.encode()
        _check(lib().gmg_icm_full_window_prob(self.ctx.h, self.h, w, frame, C.byref(out)))
        return out.value

    def Partial_Window_Prob(self, predict_pos, string, frame):
        out = C.c_double()
        s = string if isinstance(string, bytes) else string.encode()
        _check(lib().gmg_icm_partial_window_prob(self.ctx.h, self.h, predict_pos, s, frame, C.byref(out)))
        return out.value

    def Score_String(self, string, frame=0, length=None):
        s = string if isinstance(string, bytes) else string.encode()
        if length is not None:
            s = s[:length]
        return float(self.score_strings([s], frame)[0])

    def score_strings(self, strings, frame=0):
        """Score_String of many strings in one launch."""
        ss = strings if isinstance(strings, SeqSet) else SeqSet(self.ctx, seqs=strings)
        out = np.zeros(ss.n, np.float64)
        _check(lib().gmg_icm_score_strings(self.ctx.h, self.h, ss.h, frame, out.ctypes.data))
        return out

    def Cumulative_Score(self, string, frame):
        ss = self._one(string)
        out = np.zeros(ss.total, np.float64)
        _check(lib().gmg_icm_cumulative_score(self.ctx.h, self.h, ss.h, frame, out.ctypes.data))
        return out

    def Frame_Score(self, string, frame):
        ss = self._one(string)
        out = np.zeros(ss.total, np.float64)
        _check(lib().gmg_icm_frame_score(self.ctx.h, self.h, ss.h, frame, out.ctypes.data))
        return out


def parse_quality_fasta(ctx, image):
    """Quality file image -> (offsets[n_records + 1], values int32) as Fasta_Qual_Vec_Read (Common/fasta.cc:115) reads it;
    parsed on the device."""
    buf = np.frombuffer(image, np.uint8) if isinstance(image, (bytes, bytearray, memoryview)) else \
        np.ascontiguousarray(image, np.uint8)
    ptr = buf.ctypes.data if len(buf) else None
    nr, nv = C.c_int64(), C.c_int64()
    _check(lib().gmg_quality_parse_fasta(ctx.h, ptr, len(buf), C.byref(nr), C.byref(nv), None, None, 0, 0))
    off, vals = np.zeros(nr.value + 1, np.int64), np.zeros(nv.value, np.int32)
    _check(lib().gmg_quality_parse_fasta(ctx.h, ptr, len(buf), C.byref(nr), C.byref(nv), off.ctypes.data, vals.ctypes.data,
                                         nr.value, nv.value))
    return off, vals


_FRAME = re.compile(r"[+-][0-9]+")


def regions_from_coords(lines, headers=None, trim_stop=True):
    """Coordinate text -> (seq, lo, length, strand) arrays for ``SeqSet.extract``, as extract (Util/extract.cc) reads a
    coordinate file.  A line is ``id start end ...``: 1-based inclusive positions, start > end for the minus strand.  That
    covers long-orfs output, the headers of a ``.train`` file and the body of a ``.predict`` file.

    ``headers`` (e.g. ``SeqSet.from_fasta(...).headers``): the ``>`` lines of a ``.predict`` file select the sequence of
    the lines that follow, by whole header or by its first word.  Without it every region is on sequence 0 and a ``>``
    line is an error.  ``trim_stop`` drops the last codon (the stop), as ``extract -t`` does.

    A fourth field that is a signed frame (``+2``, ``-1``) must agree with the orientation; where it does not, the gene
    wraps around the end of a circular sequence, which the device path does not support."""
    if isinstance(lines, (str, bytes)):
        lines = lines.splitlines()
    index = None
    if headers is not None:
        index = {}
        for i, h in enumerate(headers):
            index.setdefault(h.strip(), i)
        for i, h in enumerate(headers):
            if h.split():
                index.setdefault(h.split()[0], i)
    cur = 0 if headers is None else None
    seq, lo, length, strand = [], [], [], []
    for k, line in enumerate(lines, 1):
        if isinstance(line, bytes):
            line = line.decode()
        t = line.split()
        if not t:
            continue
        if line.startswith(">"):
            if index is None:
                raise GmgError(f"coordinates line {k}: a '>' line selects a sequence; pass headers= to say which")
            name = line[1:].strip()
            cur = index.get(name, index.get(name.split()[0] if name.split() else name))
            if cur is None:
                raise GmgError(f"coordinates line {k}: no sequence with header {name!r}")
            continue
        if cur is None:
            raise GmgError(f"coordinates line {k}: coordinates before the first '>' line")
        if len(t) < 3:
            raise GmgError(f"coordinates line {k}: expected `id start end`, got {line.strip()!r}")
        start, end = int(t[1]), int(t[2])
        fwd = start <= end
        if len(t) > 3 and _FRAME.fullmatch(t[3]) and (t[3][0] == "+") != fwd:
            raise GmgError(f"coordinates line {k}: {t[0]} runs from {start} to {end} in frame {t[3]}: it wraps around "
                           "the end of its sequence, which extraction does not support")
        a, b = (start - 1, end) if fwd else (end - 1, start)  # 0-based [a, b)
        if trim_stop:
            if fwd:
                b -= 3
            else:
                a += 3
        if b < a:
            raise GmgError(f"coordinates line {k}: {t[0]} is shorter than its stop codon")
        seq.append(cur)
        lo.append(a)
        length.append(b - a)
        strand.append(1 if fwd else -1)
    return (np.array(seq, np.int32), np.array(lo, np.int32), np.array(length, np.int32), np.array(strand, np.int8))


def score_strings_many(ctx, models, strings, frame=0, pinned=False):
    """Score_String of every string against every model (list of ICM) in one launch -> float64 [n_models, n_strings]."""
    ss = strings if isinstance(strings, SeqSet) else SeqSet(ctx, seqs=strings)
    arr = (C.c_void_p * len(models))(*[m.h for m in models])
    if pinned:  # page-locked staging owned by the context (valid until the next pinned call): D2H at PCIe rate
        out = ctx.pinned("score_many", len(models) * ss.n, np.float64).reshape(len(models), ss.n)
    else:
        out = np.zeros((len(models), ss.n), np.float64)
    _check(lib().gmg_icm_score_strings_many(ctx.h, arr, len(models), ss.h, frame, out.ctypes.data))
    return out


def build_indep_wo_stops(ctx, gc, stops=("taa", "tag", "tga")):
    return ICM.Build_Indep_WO_Stops(ctx, gc, stops)


class ICMTraining:
    """ICM_Training_t (icm.hh:190-213)."""

    def __init__(self, ctx, model_len=12, model_depth=7, periodicity=3):
        self.ctx = ctx
        self.w, self.d, self.p = model_len, model_depth, periodicity

    def Train_Model(self, data, reverse=False, allreduce=None, rank=0, world=1, global_bases=-1):
        """Train_Model (icm.cc:1356).  ``data``: training strings (or a SeqSet); ``reverse`` = build-icm -r.
        ``allreduce(dptr, count, stream)``: sums ``count`` int32 at device address ``dptr`` across ranks
        (ordered on ``stream``) -- the exchange step of multi-GPU training.  With ``world`` > 1 this rank holds
        1 / world of the strings (``global_bases`` = training bases of all ranks): the window histogram is summed
        once and every rank walks 1 / world of its cells per level (gmg_trainer_set_shard)."""
        ss = data if isinstance(data, SeqSet) else SeqSet(self.ctx, seqs=data)
        h = C.c_void_p()
        if allreduce is None:
            cb = C.cast(None, ALLREDUCE_FN)
        else:
            def _cb(user, dptr, count, stream):
                try:
                    allreduce(dptr, count, stream)
                    return 0
                except Exception:  # pragma: no cover
                    import traceback
                    traceback.print_exc()
                    return 1
            cb = ALLREDUCE_FN(_cb)
        _check(lib().gmg_icm_train_sharded(self.ctx.h, ss.h, self.w, self.d, self.p, 1 if reverse else 0, cb, None,
                                           rank, world, global_bases, C.byref(h)))
        self.flagged_nodes = int(lib().gmg_ctx_train_flagged(self.ctx.h))
        return ICM(self.ctx, h)

    def Train_Models(self, sets, reverse=False):
        """Train_Model for many training sets in one call (gmg_icm_train_many): element k of the result is the model of
        ``sets[k]`` (a SeqSet or a list of strings, as Train_Model takes), byte-identical to Train_Model on it alone.
        ``flagged_nodes`` is summed over the batch."""
        ss = [s if isinstance(s, SeqSet) else SeqSet(self.ctx, seqs=s) for s in sets]
        arr = (C.c_void_p * len(ss))(*[s.h for s in ss])
        hs = (C.c_void_p * len(ss))()
        _check(lib().gmg_icm_train_many(self.ctx.h, arr, len(ss), self.w, self.d, self.p, 1 if reverse else 0, hs))
        self.flagged_nodes = int(lib().gmg_ctx_train_flagged(self.ctx.h))
        return [ICM(self.ctx, C.c_void_p(h)) for h in hs]

    # split form, for callers that want to drive the levels themselves
    def levels(self, data, reverse=False):
        ss = data if isinstance(data, SeqSet) else SeqSet(self.ctx, seqs=data)
        t = C.c_void_p()
        _check(lib().gmg_trainer_create(self.ctx.h, ss.h, self.w, self.d, self.p, 1 if reverse else 0, C.byref(t)))
        return _Trainer(self.ctx, t, ss, self.d)


class _Trainer:
    def __init__(self, ctx, h, ss, depth):
        self.ctx, self.h, self.ss, self.depth = ctx, h, ss, depth

    def count_level(self, level):
        ptr, n = C.c_void_p(), C.c_int64()
        _check(lib().gmg_trainer_count_level(self.h, level, C.byref(ptr), C.byref(n)))
        return ptr.value, n.value

    def finish_level(self, level):
        _check(lib().gmg_trainer_finish_level(self.h, level))

    def finish(self):
        h = C.c_void_p()
        _check(lib().gmg_trainer_finish(self.h, C.byref(h)))
        return ICM(self.ctx, h)

    def close(self):
        if self.h:
            if self.ctx.h:
                lib().gmg_trainer_free(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
