"""Host-side mirror of the reference's interface for the hot path (names and argument meaning follow
the Go seams of pbenner/kmerLr listed in SURVEY.md section 8b), on top of the C ABI.

Go is not available in this image, so this module plays the part of the cgo shim's callers: the
same control flow the Go code keeps (leapfrog epoch loop, estimator state) with every hot call going
to libkmerlr_b200.so.  Nothing here computes on the CPU; no GPU -> KmerLrError.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import Config, KmerLrError, check, lib, TIE_GO118, TIE_INDEX, FLAG_SHARDED  # noqa: F401


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


# ---------------------------------------------------------------------------------------------------
# lifecycle / communicator
# ---------------------------------------------------------------------------------------------------
def init(device=0):
    check(lib().kmerlr_init(device))


def shutdown():
    check(lib().kmerlr_shutdown())


def last_device_ms():
    return lib().kmerlr_last_device_ms()


def launch_count():
    return lib().kmerlr_launch_count()


def option(name, value):
    """run-time switches of the library (kmerlr_option): "implicit", "super_len", "hot_cols", "p2p", "persistent"
    (see include/kmerlr_b200.h)"""
    check(lib().kmerlr_option(name.encode(), int(value)))


def profile(enable):
    check(lib().kmerlr_profile(int(enable)))


def profile_read(kernel_substr):
    """(total device ms, launches) of the kernels whose name contains kernel_substr"""
    ms, n = C.c_double(), C.c_int64()
    check(lib().kmerlr_profile_read(kernel_substr.encode(), ms, n))
    return ms.value, n.value


def profile_dump():
    buf = C.create_string_buffer(1 << 16)
    check(lib().kmerlr_profile_dump(buf, len(buf)))
    rows = [r.split("\t") for r in buf.value.decode().splitlines()]
    return {r[0]: (float(r[1]), int(r[2])) for r in rows}


def comm_unique_id():
    buf = C.create_string_buffer(128)
    check(lib().kmerlr_comm_unique_id(buf))
    return buf.raw


def comm_init(rank, world, unique_id):
    check(lib().kmerlr_comm_init(rank, world, C.create_string_buffer(unique_id, 128)))


def comm_destroy():
    check(lib().kmerlr_comm_destroy())


def comm_init_torch():
    """One process per GPU under torchrun: rank 0 creates the NCCL id, torch.distributed ships it."""
    import torch.distributed as dist
    rank, world = dist.get_rank(), dist.get_world_size()
    box = [comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    comm_init(rank, world, box[0])
    return rank, world


# ---------------------------------------------------------------------------------------------------
# NewKmerCounter configuration (kmerLr_learn.go:94, kmerLr_classifier.go:96-103)
# ---------------------------------------------------------------------------------------------------
def NewKmerCounter(M, N, complement=False, reverse=False, revcomp=False, max_ambiguous=None,
                   alphabet="nucleotide", binarize=False):
    return Config(M, N, int(complement), int(reverse), int(revcomp), int(binarize),
                  {"nucleotide": 0, "gapped-nucleotide": 1}[alphabet],
                  -1 if max_ambiguous is None else int(max_ambiguous))


def flatten(seqs):
    """[]string -> (concatenated uint8 buffer, int64 offsets[n+1]); what the cgo shim passes down."""
    if isinstance(seqs, tuple):
        return np.ascontiguousarray(seqs[0], dtype=np.uint8), np.ascontiguousarray(seqs[1], dtype=np.int64)
    bs = [s.encode() if isinstance(s, str) else bytes(s) for s in seqs]
    off = np.zeros(len(bs) + 1, dtype=np.int64)
    if bs:
        off[1:] = np.cumsum([len(b) for b in bs])
    buf = np.frombuffer(b"".join(bs), dtype=np.uint8).copy() if off[-1] else np.zeros(1, dtype=np.uint8)
    return buf, off


# ---------------------------------------------------------------------------------------------------
# CoeffIndex (kmerLr_coefficients_index.go:26-54)
# ---------------------------------------------------------------------------------------------------
class CoeffIndex(int):
    def Dim(self):
        return lib().kmerlr_coeff_dim(int(self))

    def Ind2Sub(self, k1, k2):
        return lib().kmerlr_coeff_ind2sub(int(self), k1, k2)

    def Sub2Ind(self, i):
        a, b = C.c_int64(), C.c_int64()
        lib().kmerlr_coeff_sub2ind(int(self), i, a, b)
        return a.value, b.value


# ---------------------------------------------------------------------------------------------------
# data (kmerLr_data.go)
# ---------------------------------------------------------------------------------------------------
class Sequences:
    """2-bit packed sequences resident in HBM.  A set parsed from FASTA text (import_fasta) also carries the
    record names (.names) and the number of records of every text (.records); for other sets both are None."""

    names = None
    records = None

    def __init__(self, seqs):
        buf, off = flatten(seqs)
        self.n = len(off) - 1
        self.total_bases = int(off[-1])
        h = C.c_uint64()
        check(lib().kmerlr_sequences_create(_p(buf), _p(off), self.n, h))
        self.h = h.value

    @classmethod
    def _resident(cls, handle):
        s = cls.__new__(cls)
        s.h = handle
        n, total = C.c_int64(), C.c_int64()
        check(lib().kmerlr_sequences_info(handle, n, total, None))
        s.n, s.total_bases = n.value, total.value
        return s

    def lengths(self):
        out = np.zeros(max(self.n, 1), dtype=np.int64)
        check(lib().kmerlr_sequences_info(self.h, None, None, _p(out)))
        return out[:self.n]

    def bases(self):
        """the bases of every sequence one after the other as b"acgt", b"n" at invalid positions (read-back)"""
        out = np.zeros(max(self.total_bases, 1), dtype=np.uint8)
        check(lib().kmerlr_sequences_bases(self.h, _p(out)))
        return out[:self.total_bases].tobytes()

    def regions(self, seq_index, from_, to):
        """the slicing of extractFasta (kmerLr_predict_genomic.go:93-112): sequence i of the new set is bases
        [from_[i], to[i]) of sequence seq_index[i], cut out on the device"""
        idx = np.ascontiguousarray(seq_index, dtype=np.int64)
        frm = np.ascontiguousarray(from_, dtype=np.int64)
        to = np.ascontiguousarray(to, dtype=np.int64)
        if not len(idx) == len(frm) == len(to):
            raise KmerLrError(_lib.ERR_ARG, "regions: seq_index, from and to differ in length")
        h = C.c_uint64()
        check(lib().kmerlr_sequences_regions(self.h, _p(idx), _p(frm), _p(to), len(idx), h))
        return Sequences._resident(h.value)

    def free(self):
        if getattr(self, "h", 0):
            lib().kmerlr_free(self.h)
            self.h = 0

    __del__ = free


def _host_bytes(t):
    """a text as a contiguous uint8 array without a copy where the buffer allows it"""
    if isinstance(t, np.ndarray):
        return np.ascontiguousarray(t).view(np.uint8).reshape(-1)
    return np.frombuffer(t, dtype=np.uint8) if len(t) else np.zeros(0, dtype=np.uint8)


def import_fasta(*texts):
    """import_fasta (kmerLr_data.go:101-121) for the bytes of one or more FASTA files (bytes, bytearray, memoryview
    or uint8 arrays): one resident Sequences with the records of text 0 first, then text 1, ...; .names are the
    record names (the whole header line after '>', stripped), .records the number of records of every text.  The
    caller decompresses gzip files."""
    arrs = [_host_bytes(t) for t in texts]
    ptrs = (C.c_void_p * max(len(arrs), 1))(*[a.ctypes.data if len(a) else None for a in arrs])
    nbytes = np.array([len(a) for a in arrs] or [0], dtype=np.int64)
    records = np.zeros(max(len(arrs), 1), dtype=np.int64)
    h = C.c_uint64()
    check(lib().kmerlr_sequences_from_fasta(ptrs, _p(nbytes), len(arrs), _p(records), h))
    s = Sequences._resident(h.value)
    s.records = records[:len(arrs)].tolist()
    off = np.zeros(s.n + 1, dtype=np.int64)
    check(lib().kmerlr_sequences_names(s.h, None, 0, _p(off)))
    buf = C.create_string_buffer(max(int(off[-1]), 1))
    check(lib().kmerlr_sequences_names(s.h, buf, len(buf), _p(off)))
    raw = buf.raw
    s.names = [raw[off[i]:off[i + 1]].decode("utf-8", "surrogateescape") for i in range(s.n)]
    return s


def _text_sets(seqs):
    """the sets of a FASTA-parsed Sequences, one per text it was read from, as resident copies (whole records)"""
    lens, sets, r = seqs.lengths(), [], 0
    for k in seqs.records:
        idx = np.arange(r, r + k, dtype=np.int64)
        sets.append(seqs.regions(idx, np.zeros(k, dtype=np.int64), lens[r:r + k]))
        r += k
    return sets


class KmerDataSet:
    """KmerDataSet{Data, Labels, Kmers} (kmerLr_data.go:34-38); Data stays in HBM behind a handle."""

    def __init__(self, handle):
        self.h = handle
        n, m, nnz, nc = (C.c_int64() for _ in range(4))
        check(lib().kmerlr_matrix_info(handle, n, m, nnz, nc))
        self.n, self.m, self.nnz, self.n_classes = n.value, m.value, nnz.value, nc.value
        check(lib().kmerlr_matrix_rows_global(handle, n))
        self.n_global = n.value          # rows of all ranks (= n unless the matrix is a shard)
        self.Labels = None

    def free(self):
        if getattr(self, "h", 0):
            try:
                lib().kmerlr_free(self.h)
            except Exception:
                pass
            self.h = 0

    __del__ = free

    def Dim(self):
        return self.m + 1

    def Kmers(self):
        """class list as (k, code) arrays; the Go side rebuilds KmerClass names from them"""
        if getattr(self, "_kmers", None) is not None:
            return self._kmers
        k = np.zeros(max(self.n_classes, 1), dtype=np.int32)
        code = np.zeros(max(self.n_classes, 1), dtype=np.uint64)
        check(lib().kmerlr_matrix_classes(self.h, _p(k), _p(code)))
        return k[:self.n_classes], code[:self.n_classes]

    def rows(self):
        """(rowptr, col, val): CSR without the bias column (Go sparse index = col + 1)"""
        rowptr = np.zeros(self.n + 1, dtype=np.int64)
        col = np.zeros(max(self.nnz, 1), dtype=np.int32)
        val = np.zeros(max(self.nnz, 1), dtype=np.float64)
        check(lib().kmerlr_matrix_rows(self.h, _p(rowptr), _p(col), _p(val)))
        return rowptr, col[:self.nnz], val[:self.nnz]

    def SetLabels(self, labels):
        lab = np.ascontiguousarray(labels, dtype=np.uint8)
        check(lib().kmerlr_matrix_set_labels(self.h, _p(lab), len(lab)))
        self.Labels = lab.astype(bool)

    def class_weights(self):
        cw = np.zeros(2)
        check(lib().kmerlr_class_weights(self.h, _p(cw)))
        return cw

    def subset(self, rows):
        """filterCvGroup (kmerLr_crossvalidation.go:95): rows[0..len) of this data set (any order, repeats allowed) as a
        new data set in HBM with the same columns and class numbering; Labels are carried, n_global = len(rows).  It
        stays valid after this data set is freed."""
        idx = np.ascontiguousarray(rows, dtype=np.int64).reshape(-1)
        h = C.c_uint64()
        check(lib().kmerlr_matrix_subset(self.h, _p(idx), len(idx), h))
        r = KmerDataSet(h.value)
        if self.Labels is not None:
            r.Labels = self.Labels[idx]
        if getattr(self, "_kmers", None) is not None:
            r._kmers = self._kmers
        return r


def from_csr(n, m, rowptr, col, val, sharded=False):
    rowptr = np.ascontiguousarray(rowptr, dtype=np.int64)
    col = np.ascontiguousarray(col, dtype=np.int32)
    val = np.ascontiguousarray(val, dtype=np.float64)
    h = C.c_uint64()
    check(lib().kmerlr_matrix_from_csr(n, m, _p(rowptr), _p(col), _p(val), FLAG_SHARDED if sharded else 0, h))
    return KmerDataSet(h.value)


def from_dense(d, sharded=False):
    d = np.asarray(d, dtype=np.float64)
    rowptr, col, val = [0], [], []
    for r in d:
        nz = np.nonzero(r)[0]
        col.extend(nz.tolist())
        val.extend(r[nz].tolist())
        rowptr.append(len(col))
    return from_csr(d.shape[0], d.shape[1], rowptr, col or [0], val or [0.0], sharded)


def _extract(config, seqs, kmers, features, sharded):
    fk = fc = ft = None
    nf = nft = 0
    if kmers is not None and len(kmers[0]):
        fk = np.ascontiguousarray(kmers[0], dtype=np.int32)
        fc = np.ascontiguousarray(kmers[1], dtype=np.uint64)
        nf = len(fk)
    if features is not None and len(features):
        ft = np.ascontiguousarray(features, dtype=np.int32).reshape(-1, 2)
        nft = ft.shape[0]
    h = C.c_uint64()
    flags = FLAG_SHARDED if sharded else 0
    if isinstance(seqs, Sequences):
        check(lib().kmerlr_extract_resident(C.byref(config), seqs.h, _p(fk), _p(fc), nf, _p(ft), nft, flags, h))
    else:
        buf, off = flatten(seqs)
        check(lib().kmerlr_extract(C.byref(config), _p(buf), _p(off), len(off) - 1, _p(fk), _p(fc), nf, _p(ft), nft,
                                   flags, h))
    return KmerDataSet(h.value)


def _convert(cfg, seqs, kmers, features, generate_features, sharded):
    """scan_sequences + convert_counts_list.  convert_counts (kmerLr_data.go:197-235) builds one column per class
    only when the feature list is empty AND generate_features is set; with an empty list and generate_features
    off (`n = len(features) + 1`, :212) the rows hold the bias alone, while Kmers stays the class list."""
    if generate_features or (features is not None and len(features)):
        return _extract(cfg, seqs, kmers, features, sharded)
    full = _extract(cfg, seqs, kmers, None, sharded)
    ks, n = full.Kmers(), full.n
    full.free()
    data = from_csr(n, 0, np.zeros(n + 1, dtype=np.int64), np.zeros(0, dtype=np.int32), np.zeros(0), sharded)
    data._kmers = ks
    return data


def compile_training_data(config, kmersCounter, kmers, features, generate_features, binarize, fg, bg=None,
                          sharded=False):
    """compile_training_data (kmerLr_data.go:306-325).  fg / bg are the sequences import_fasta returned
    (lists of str/bytes, or (buffer, offsets)); labels = true for fg.  Or fg = the resident set of
    import_fasta(fg_text, bg_text) and bg = None: its records per text give the labels."""
    del config
    cfg = Config.from_buffer_copy(kmersCounter)
    cfg.binarize = int(binarize)
    if isinstance(fg, Sequences):
        if bg is not None or fg.records is None or len(fg.records) != 2:
            raise KmerLrError(_lib.ERR_ARG, "compile_training_data: a resident set must come from import_fasta(fg, bg)")
        data = _convert(cfg, fg, kmers, features, generate_features, sharded)
        data.SetLabels(np.concatenate([np.ones(fg.records[0], dtype=np.uint8), np.zeros(fg.records[1], dtype=np.uint8)]))
        return data
    fb, fo = flatten(fg)
    bb, bo = flatten(bg)
    nfg, nbg = len(fo) - 1, len(bo) - 1
    buf = np.concatenate([fb[:fo[-1]], bb[:bo[-1]]]) if (fo[-1] + bo[-1]) else np.zeros(1, dtype=np.uint8)
    off = np.concatenate([fo, bo[1:] + fo[-1]])
    data = _convert(cfg, (buf, off), kmers, features, generate_features, sharded)
    data.SetLabels(np.concatenate([np.ones(nfg, dtype=np.uint8), np.zeros(nbg, dtype=np.uint8)]))
    return data


def compile_test_data(config, kmersCounter, kmers, features, generate_features, binarize, sequences):
    """compile_test_data (kmerLr_data.go:327-335): counter frozen to the classifier's k-mers.  sequences may be a
    resident set (Sequences, import_fasta)."""
    del config
    cfg = Config.from_buffer_copy(kmersCounter)
    cfg.binarize = int(binarize)
    return _convert(cfg, sequences, kmers, features, generate_features, False)


def compile_data(config, kmersCounter, kmers, features, generate_features, binarize, sequence_sets):
    """compile_data (kmerLr_data.go:339-358): several sequence sets, ONE class numbering (the union of the
    classes observed in all of them, or the supplied list), one KmerDataSet per set.  The union comes from one
    extraction over the concatenation; every set is then extracted against that frozen list, which gives the
    rows `counts_list.Slice(k[i], k[i+1])` would.  sequence_sets may also be the resident set of
    import_fasta(text_0, text_1, ...): one data set per text."""
    del config
    cfg = Config.from_buffer_copy(kmersCounter)
    cfg.binarize = int(binarize)
    if isinstance(sequence_sets, Sequences):
        if sequence_sets.records is None:
            raise KmerLrError(_lib.ERR_ARG, "compile_data: a resident set must come from import_fasta")
        if kmers is None or len(kmers[0]) == 0:
            joint = _extract(cfg, sequence_sets, None, None, False)
            kmers = joint.Kmers()
            joint.free()
        sets = _text_sets(sequence_sets)
        out = [_convert(cfg, s, kmers, features, generate_features, False) for s in sets]
        for s in sets:
            s.free()
        return out
    sets = [flatten(s) for s in sequence_sets]
    if kmers is None or len(kmers[0]) == 0:
        buf = np.concatenate([b[:o[-1]] for b, o in sets] + [np.zeros(1, dtype=np.uint8)])
        offs, base = [np.zeros(1, dtype=np.int64)], 0
        for b, o in sets:
            offs.append(o[1:] - o[0] + base)
            base += int(o[-1] - o[0])
        joint = _extract(cfg, (buf, np.concatenate(offs)), None, None, False)
        kmers = joint.Kmers()
        joint.free()
    return [_convert(cfg, s, kmers, features, generate_features, False) for s in sets]


def compute_class_weights(c):
    """compute_class_weights (kmerLr_data.go:178-193); pure arithmetic on the label counts"""
    c = np.asarray(c, dtype=bool)
    n1, n0 = int(c.sum()), int((~c).sum())
    return np.array([(n0 + n1) / (2.0 * n0), (n0 + n1) / (2.0 * n1)])


# ---------------------------------------------------------------------------------------------------
# data transforms (kmerLr_transform.go:33-317,584-629)
# ---------------------------------------------------------------------------------------------------
class Transform:
    """Offset / Scale per coefficient, index 0 = bias (offset 0, scale 1); None = absent, as in the reference.

    The reference applies (v - offset) * scale to every entry of every row, zeros included, which
    densifies the data (kmerLr_transform.go:600-609).  Here the rows stay sparse counts in HBM: for a
    linear model the transform is a reparameterisation,
        theta'_j = scale_j theta_j,   theta'_0 = theta_0 - sum_j offset_j scale_j theta_j,
        g_j = scale_j (g'_j - offset_j g'_0),
    so every kernel runs unchanged on theta' (logisticRegression below)."""

    def __init__(self, Offset=None, Scale=None):
        self.Offset = None if Offset is None else np.ascontiguousarray(Offset, dtype=np.float64)
        self.Scale = None if Scale is None else np.ascontiguousarray(Scale, dtype=np.float64)

    def Nil(self):
        return self.Offset is None and self.Scale is None

    def Select(self, b):
        """TransformFull.Select (kmerLr_transform.go:290-307): b = mask or ascending coefficient indices"""
        b = np.asarray(b)
        idx = np.nonzero(b)[0] if b.dtype == bool else b.astype(np.int64)
        return Transform(None if self.Offset is None else self.Offset[idx], None if self.Scale is None else self.Scale[idx])

    def Apply(self, data):
        """Transform.Apply (kmerLr_transform.go:584-629) on the rows of a reduced data set, as estimate() does before
        the solver runs (kmerLr_estimator.go:148): returns the transformed data set (a new matrix in HBM; with an
        offset its rows are dense).  A nil transform returns `data` itself."""
        if self.Nil():
            return data
        h = C.c_uint64()
        n = len(self.Offset if self.Offset is not None else self.Scale)
        check(lib().kmerlr_matrix_transform(data.h, _p(self.Offset), _p(self.Scale), n, h))
        r = KmerDataSet(h.value)
        r.Labels = data.Labels
        return r


class TransformFull(Transform):
    def Fit(self, data, kind, cooccurrence=False):
        """TransformFull.Fit (kmerLr_transform.go:40-252) from the column moments computed on the device"""
        kind = (kind or "none").lower()
        if kind in ("", "none"):
            self.Offset = self.Scale = None
            return self
        m = data.m
        s1, s2, mx = np.zeros(max(m, 1)), np.zeros(max(m, 1)), np.zeros(max(m, 1))
        cnt = np.zeros(max(m, 1), dtype=np.int64)
        check(lib().kmerlr_column_moments(data.h, _p(s1), _p(s2), _p(mx), _p(cnt)))
        s1, s2, mx = s1[:m], s2[:m], mx[:m]
        if cooccurrence:
            # pair features v_a v_b in CoeffIndex order after the single features (kmerLr_transform.go:90-99,118-127)
            npairs = m * (m - 1) // 2
            p1, p2, pm = np.zeros(max(npairs, 1)), np.zeros(max(npairs, 1)), np.zeros(max(npairs, 1))
            pc = np.zeros(max(npairs, 1), dtype=np.int64)
            check(lib().kmerlr_pair_moments(data.h, _p(p1), _p(p2), _p(pm), _p(pc)))
            s1, s2, mx = (np.concatenate([a, b[:npairs]]) for a, b in ((s1, p1), (s2, p2), (mx, pm)))
            m = m + npairs
        n = float(data.n_global)
        offset, scale = np.zeros(m + 1), np.ones(m + 1)
        if kind in ("standardizer", "variance-scaler"):
            mean = s1 / n
            # sum_i (v_i - mean)^2 over ALL n samples = sum v^2 - n mean^2 (the reference adds the zero entries as
            # (n - k) mean^2, :129-131)
            sj = s2 - n * mean * mean
            sj = np.where(sj < 0.0, 0.0, sj)
            with np.errstate(divide="ignore", invalid="ignore"):
                sc = 1.0 / np.sqrt(sj / (n - 1.0))
            scale[1:] = np.where(sj == 0.0, 1.0, sc)
            offset[1:] = mean
            self.Offset, self.Scale = (offset, scale) if kind == "standardizer" else (None, scale)
        elif kind == "max-abs-scaler":
            with np.errstate(divide="ignore"):
                scale[1:] = 1.0 / mx
            self.Offset, self.Scale = None, scale
        elif kind == "mean-scaler":
            with np.errstate(divide="ignore"):
                scale[1:] = n / s1
            self.Offset, self.Scale = None, scale
        else:
            raise KmerLrError(_lib.ERR_ARG, "invalid data transform")
        return self


# ---------------------------------------------------------------------------------------------------
# logisticRegression (kmerLr_logistic_regression.go:30-272)
# ---------------------------------------------------------------------------------------------------
class logisticRegression:
    def __init__(self, Theta, ClassWeights=(1.0, 1.0), Lambda=0.0, Cooccurrence=False, Transform=None):
        self.Theta = np.ascontiguousarray(Theta, dtype=np.float64)
        self.ClassWeights = np.ascontiguousarray(ClassWeights, dtype=np.float64)
        self.Lambda = float(Lambda)
        self.Cooccurrence = bool(Cooccurrence)
        self.Transform = Transform

    def Dim(self):
        return len(self.Theta) - 1

    def _transformed(self):
        return self.Transform is not None and not self.Transform.Nil()

    def _theta_eff(self):
        """theta' of the reparameterised model (see Transform)"""
        if not self._transformed():
            return self.Theta
        t = self.Theta.copy()
        sc = self.Transform.Scale if self.Transform.Scale is not None else np.ones(len(t))
        if len(sc) != len(t):
            raise KmerLrError(_lib.ERR_INTERNAL, "internal error")
        t[1:] = t[1:] * sc[1:]
        if self.Transform.Offset is not None:
            t[0] = t[0] - float(np.dot(self.Transform.Offset[1:], t[1:]))
        return np.ascontiguousarray(t)

    def _penalty(self):
        return self.Lambda == self.Lambda and self.Lambda != 0.0

    def LinearPdf(self, data):
        t = self._theta_eff()
        out = np.zeros(max(data.n, 1))
        check(lib().kmerlr_linear_pdf(data.h, _p(t), len(t), int(self.Cooccurrence), _p(out)))
        return out[:data.n]

    def LogPdf(self, data):
        t = self._theta_eff()
        out = np.zeros(max(data.n, 1))
        check(lib().kmerlr_logpdf(data.h, _p(t), len(t), int(self.Cooccurrence), _p(out)))
        return out[:data.n]

    def Gradient(self, g, data, labels=None):
        if labels is not None:
            data.SetLabels(labels)
        if g is None or len(g) == 0:
            g = np.zeros(len(self.Theta))
        elif len(g) != len(self.Theta):
            raise KmerLrError(_lib.ERR_INTERNAL, "internal error")
        if not self._transformed():
            check(lib().kmerlr_gradient(data.h, _p(self.Theta), len(self.Theta), _p(self.ClassWeights), self.Lambda,
                                        int(self.Cooccurrence), _p(g)))
            return g
        t = self._theta_eff()
        check(lib().kmerlr_gradient(data.h, _p(t), len(t), _p(self.ClassWeights), 0.0, int(self.Cooccurrence), _p(g)))
        g0 = g[0]
        if self.Transform.Offset is not None:
            g[1:] -= self.Transform.Offset[1:] * g0
        if self.Transform.Scale is not None:
            g[1:] *= self.Transform.Scale[1:]
        if self._penalty():                                  # (:237-246) on the ORIGINAL theta
            g[1:] += self.Lambda * np.sign(self.Theta[1:])
        return g

    def Loss(self, data, c=None):
        if c is not None:
            data.SetLabels(c)
        out = C.c_double()
        if not self._transformed():
            check(lib().kmerlr_loss(data.h, _p(self.Theta), len(self.Theta), _p(self.ClassWeights), self.Lambda,
                                    int(self.Cooccurrence), out))
            return out.value
        t = self._theta_eff()
        check(lib().kmerlr_loss(data.h, _p(t), len(t), _p(self.ClassWeights), 0.0, int(self.Cooccurrence), out))
        r = out.value
        if self._penalty():
            r += self.Lambda * float(np.sum(np.abs(self.Theta[1:data.m + 1])))
        return r


# ---------------------------------------------------------------------------------------------------
# featureSelector (kmerLr_feature_selection.go)
# ---------------------------------------------------------------------------------------------------
class featureSelection:
    def __init__(self, selector, b, c, theta_full):
        self.selector, self.b, self.c = selector, b, c
        self.sel = np.nonzero(b)[0].astype(np.int64)     # k of featureSelection.Data (:313-318)
        self._theta = theta_full[self.sel]

    def Theta(self):
        return self._theta.copy()

    def Data(self, data):
        return select_data(data, self.sel)


def select_data(data, sel):
    """featureSelection.Data (kmerLr_feature_selection.go:309-343) for an explicit, ascending list of
    coefficient indices (sel[0] = 0 is the bias)"""
    sel = np.ascontiguousarray(sel, dtype=np.int64)
    h = C.c_uint64()
    check(lib().kmerlr_reduce(data.h, _p(sel), len(sel), h))
    r = KmerDataSet(h.value)
    r.Labels = data.Labels
    return r


class featureSelector:
    def __init__(self, ClassWeights, Cooccurrence, N, M, Epsilon=0.0, tie=TIE_GO118, Transform=None):
        self.ClassWeights = np.ascontiguousarray(ClassWeights, dtype=np.float64)
        self.Cooccurrence, self.N, self.M, self.Epsilon, self.tie = bool(Cooccurrence), int(N), int(M), Epsilon, tie
        self.Transform = Transform          # TransformFull of the full space (featureSelector.Transform)

    def Select(self, data, theta0, active_idx, active_theta, lambda_prev, want_gradient=False):
        if self.M != data.Dim() - 1:
            raise KmerLrError(_lib.ERR_INTERNAL, "internal error")
        nt = CoeffIndex(self.M).Dim() if self.Cooccurrence else self.M + 1
        ai = np.ascontiguousarray(active_idx, dtype=np.int64)
        at = np.ascontiguousarray(active_theta, dtype=np.float64)
        mask = np.zeros(nt, dtype=np.uint8)
        lam, c, ok = C.c_double(), C.c_int64(), C.c_int()
        t = np.zeros(nt)
        t[0] = theta0
        nz = at != 0.0
        t[ai[nz]] = at[nz]
        if self.Transform is not None and not self.Transform.Nil():
            # gradient under the transform (kmerLr_feature_selection.go:221-229 with lr.Transform set):
            # reparameterised on the host side, then the selection proper
            g = logisticRegression(t, self.ClassWeights, 0.0, self.Cooccurrence, self.Transform).Gradient(None, data)
            check(lib().kmerlr_select_from_gradient(_p(g), nt, self.N, _p(ai), _p(at), len(ai), self.tie, self.Epsilon,
                                                    float(lambda_prev), _p(mask), lam, c, ok))
        else:
            g = np.zeros(nt) if want_gradient else None
            check(lib().kmerlr_select(data.h, _p(self.ClassWeights), int(self.Cooccurrence), self.N, float(theta0),
                                      _p(ai), _p(at), len(ai), self.tie, self.Epsilon, float(lambda_prev), _p(mask), nt,
                                      lam, c, ok, _p(g)))
        s = featureSelection(self, mask.astype(bool), c.value, t)
        s.g = g
        return s, lam.value, bool(ok.value)


# ---------------------------------------------------------------------------------------------------
# estimator (kmerLr_estimator.go:209-255 control loop; kmerLr_estimator_proximal.go solver)
# ---------------------------------------------------------------------------------------------------
class KmerLrEstimator:
    """State the Go estimator keeps between leapfrog targets: theta, active coefficient indices,
    L1Reg, the hook's loss_old / loss_new."""

    def __init__(self, Cooccurrence=False, Epsilon=0.0, EpsilonLoss=1e-8, EpsilonLambda=0.0, L2Reg=0.0,
                 StepSizeFactor=1.0, MaxIterations=100000, MaxEpochs=0, tie=TIE_GO118, Accelerated=False):
        self.Cooccurrence, self.Epsilon, self.EpsilonLoss = Cooccurrence, Epsilon, EpsilonLoss
        self.EpsilonLambda, self.L2Reg, self.StepSizeFactor = EpsilonLambda, L2Reg, StepSizeFactor
        self.MaxIterations, self.MaxEpochs, self.tie = MaxIterations, MaxEpochs, tie
        self.Theta = np.zeros(1)
        self.active_idx = np.zeros(0, dtype=np.int64)
        self.L1Reg = 0.0
        self.ClassWeights = np.ones(2)
        self.hook_state = np.array([np.nan, np.nan])
        self.path = []
        self.Transform = None            # the selected transform of the last estimate (r.Transform of the reference's KmerLr)
        # Accelerated: estimate_proximal runs FISTA with gradient restart (kmerlr_proxgrad_accel_full; every one-GPU
        # matrix: reduced ones of any width, and the whole feature space of a fixed-lambda fit; with Cooccurrence and a
        # Theta of every pair coefficient of the raw matrix, kmerlr_proxgrad_pairs_accel).  accel_state = (handle of the data, y, t, restarts of the last call): the momentum carried between calls
        # on the same reduced data, so that a run cut into slices of MaxIterations resumes exactly.
        self.Accelerated = Accelerated
        self.accel_state = None

    def estimate_proximal(self, data_train, lam):
        """estimate_proximal (kmerLr_estimator_proximal.go:78-120) on the (reduced) data set."""
        theta = np.ascontiguousarray(self.Theta, dtype=np.float64).copy()
        iters, delta = C.c_int64(), C.c_double()
        # pair mode on the whole data set (estimate_fixed): theta holds every pair coefficient of the raw matrix
        pairs = bool(self.Cooccurrence) and len(theta) == lib().kmerlr_coeff_dim(data_train.m) != data_train.m + 1
        if self.Accelerated:
            return self._estimate_accelerated(data_train, lam, theta, iters, delta, pairs)
        entry = lib().kmerlr_proxgrad_pairs if pairs else lib().kmerlr_proxgrad
        check(entry(data_train.h, _p(theta), len(theta), _p(self.ClassWeights), float(lam),
                                    self.L2Reg, self.StepSizeFactor, self.Epsilon, self.EpsilonLoss,
                                    self.MaxIterations, _p(self.hook_state), iters, delta))
        self.Theta = theta
        return iters.value, delta.value

    def _estimate_accelerated(self, data_train, lam, theta, iters, delta, pairs=False):
        st = self.accel_state
        if st is None or st[0] != data_train.h or len(st[1]) != len(theta):
            st = (data_train.h, theta.copy(), 1.0, 0)         # fresh start: y = theta, t = 1
        y, t, restarts = st[1].copy(), C.c_double(st[2]), C.c_int64()
        entry = lib().kmerlr_proxgrad_pairs_accel if pairs else lib().kmerlr_proxgrad_accel_full
        check(entry(data_train.h, _p(theta), _p(y), t, len(theta), _p(self.ClassWeights), float(lam), self.L2Reg,
                    self.StepSizeFactor, self.Epsilon, self.EpsilonLoss, self.MaxIterations, _p(self.hook_state), iters,
                    delta, restarts))
        self.Theta = theta
        self.accel_state = (data_train.h, y, t.value, restarts.value)
        return iters.value, delta.value

    def estimate_coordinate(self, data_train):
        """estimate_coordinate (kmerLr_estimator_coordinate.go:86-139) on a reduced data set: IRLS outer
        iterations, cyclic coordinate descent on the dense Gram matrix inside (theta slices de-aliased).
        L1Reg / L2Reg are the estimator's (sum scale, as the reference applies them).  Returns (sweeps, delta)."""
        theta = np.ascontiguousarray(self.Theta, dtype=np.float64).copy()
        sweeps, delta = C.c_int64(), C.c_double()
        check(lib().kmerlr_coordinate(data_train.h, _p(theta), len(theta), _p(self.ClassWeights), float(self.L1Reg),
                                      self.L2Reg, self.Epsilon, self.EpsilonLoss, self.MaxIterations,
                                      _p(self.hook_state), sweeps, delta))
        self.Theta = theta
        return sweeps.value, delta.value

    def estimate_loop(self, data, lambdaAuto, balance=False, transform=None):
        """estimate_loop (kmerLr_estimator.go:209-255): leapfrog epochs until Select returns !ok.  transform: the
        TransformFull fitted on `data` (or None): the selection gradient is taken under it, and every reduced data
        set goes through Transform.Apply before the solver sees it, as estimate() does (kmerLr_estimator.go:148);
        self.Theta is then the coefficient vector of the TRANSFORMED features, as in the reference's model."""
        n = data.n_global                # len(data.Data) of the whole set: the same L1Reg on every rank
        self.ClassWeights = data.class_weights() if balance else np.ones(2)
        s = featureSelector(self.ClassWeights, self.Cooccurrence, lambdaAuto, data.m, self.EpsilonLambda, self.tie,
                            Transform=transform)
        r = False
        epoch = 0
        while self.MaxEpochs == 0 or epoch < self.MaxEpochs:
            selection, lam, ok = s.Select(data, self.Theta[0], self.active_idx, self.Theta[1:], self.L1Reg)
            if not ok and r:
                break
            self.L1Reg = lam * n
            self.active_idx = selection.sel[1:].copy()
            self.Theta = selection.Theta()
            reduced = selection.Data(data)
            reduced.SetLabels(data.Labels)
            if transform is not None and not transform.Nil():
                self.Transform = transform.Select(selection.sel)        # selection.Transform()
                tdata = self.Transform.Apply(reduced)
                reduced.free()
                reduced = tdata
            self.accel_state = None          # the momentum restarts at every epoch: y = theta of the new reduced matrix, t = 1
            iters, _ = self.estimate_proximal(reduced, lam)
            reduced_nnz = reduced.nnz
            reduced.free()
            self.path.append((lam, iters, len(self.active_idx), reduced_nnz))
            r = True
            epoch += 1
        return epoch

    def Estimate(self, data, LambdaAuto, balance=False, transform=None):
        """Estimate (kmerLr_estimator.go:257-270): one warm-started loop per target."""
        out = []
        for n in LambdaAuto:
            self.estimate_loop(data, n, balance, transform)
            out.append((self.active_idx.copy(), self.Theta.copy()))
        return out


# ---------------------------------------------------------------------------------------------------
# cross-validation (kmerLr_crossvalidation.go:56-211)
# ---------------------------------------------------------------------------------------------------
def cv_groups(n, k):
    """getCvGroups (kmerLr_crossvalidation.go:56) without its math/rand shuffle: row i goes to fold i mod k.  Go's
    generator cannot be reproduced here (SURVEY §2), so a caller that needs the reference's folds passes its fold ids
    to crossvalidation instead."""
    if k < 1:
        raise KmerLrError(_lib.ERR_ARG, "cv_groups: k must be at least 1")
    return np.arange(n, dtype=np.int64) % k


def cv_scatter(fold_ids, held_out):
    """the held-out results of every fold back at the rows' original positions: held_out[f] lists fold f's rows in
    ascending row order (the order crossvalidation takes its test subset in), folds in ascending order of their id"""
    fold_ids = np.asarray(fold_ids)
    out = np.zeros(len(fold_ids))
    for f, v in zip(np.unique(fold_ids), held_out):
        out[np.nonzero(fold_ids == f)[0]] = v
    return out


class CrossValidation:
    """what crossvalidation returns.  Folds: the fold ids in ascending order; Models[f][j] = (active_idx, Theta,
    Transform) of fold f's estimator after target LambdaAuto[j]; Predictions[j] = the held-out LogPdf of every row
    under the model of target j that was fitted without the row's fold, at the row's original position (the
    reference's CV .table); Loss[f][j] = the held-out Loss of fold f at target j (its _loss.table)."""

    def __init__(self, folds, models, predictions, loss):
        self.Folds, self.Models, self.Predictions, self.Loss = folds, models, predictions, loss


def crossvalidation(data, fold_ids, make_estimator, LambdaAuto, balance=False, transform_kind=None):
    """crossvalidation / learn_cv (kmerLr_crossvalidation.go:167-211) on one resident data set with labels.  Every
    fold is a row subset of `data` (same columns and class numbering): its training rows are all rows of the other
    folds.  Per fold, one after the other: make_estimator() gives a fresh KmerLrEstimator; the transform of
    `transform_kind` is fitted on the training rows (TransformFull.Fit); Estimate runs over LambdaAuto, warm-started
    from target to target; after each target the held-out rows are reduced to the model's features (SelectData) and
    scored (LogPdf, and Loss with the estimator's class weights and no penalty), kmerLr_classifier.go:107-147.  The
    tables are written by the caller."""
    fold_ids = np.asarray(fold_ids, dtype=np.int64).reshape(-1)
    if len(fold_ids) != data.n:
        raise KmerLrError(_lib.ERR_ARG, "crossvalidation: one fold id per row is needed")
    folds = np.unique(fold_ids)
    if len(folds) < 2:
        raise KmerLrError(_lib.ERR_ARG, "crossvalidation: at least two folds are needed")
    models, held_out, losses = [], [], []
    for f in folds:
        train, test = data.subset(np.nonzero(fold_ids != f)[0]), data.subset(np.nonzero(fold_ids == f)[0])
        try:
            est = make_estimator()
            transform = TransformFull().Fit(train, transform_kind, est.Cooccurrence) if transform_kind else None
            fm, fp, fl = [], [], []
            for n in LambdaAuto:
                est.Estimate(train, [n], balance, transform)
                fm.append((est.active_idx.copy(), est.Theta.copy(), est.Transform))
                sel = select_data(test, np.concatenate([[0], est.active_idx]))
                try:
                    lr = logisticRegression(est.Theta, est.ClassWeights, 0.0, False, est.Transform)
                    fp.append(lr.LogPdf(sel))
                    fl.append(lr.Loss(sel))
                finally:
                    sel.free()
            models.append(fm)
            held_out.append(fp)
            losses.append(fl)
        finally:
            train.free()
            test.free()
    predictions = [cv_scatter(fold_ids, [p[j] for p in held_out]) for j in range(len(LambdaAuto))]
    return CrossValidation(folds, models, predictions, losses)


# ---------------------------------------------------------------------------------------------------
# genomic scoring (kmerLr_predict_genomic.go:116-171)
# ---------------------------------------------------------------------------------------------------
class genomicKmerLr:
    """models: list of dict(counter=Config, class_k, class_code, features, theta, summary)"""

    def __init__(self, classifiers):
        self.classifiers = classifiers
        self._keep = []
        self._arr = (_lib.Model * len(classifiers))()
        for i, md in enumerate(classifiers):
            ck = np.ascontiguousarray(md["class_k"], dtype=np.int32)
            cc = np.ascontiguousarray(md["class_code"], dtype=np.uint64)
            ft = np.ascontiguousarray(md["features"], dtype=np.int32).reshape(-1, 2)
            th = np.ascontiguousarray(md["theta"], dtype=np.float64).reshape(-1, ft.shape[0] + 1)
            self._keep += [ck, cc, ft, th]
            self._arr[i] = _lib.Model(md["counter"], len(ck), ck.ctypes.data_as(C.POINTER(C.c_int32)),
                                      cc.ctypes.data_as(C.POINTER(C.c_uint64)), ft.shape[0],
                                      ft.ctypes.data_as(C.POINTER(C.c_int32)), th.shape[0],
                                      th.ctypes.data_as(C.POINTER(C.c_double)), _lib.SUMMARY[md.get("summary", "")])

    def predict_window_genomic(self, sequences, window_size, window_step):
        """predict_window_genomic (:147-171): returns predictions[i] per region (log scale)"""
        L = lib()
        if isinstance(sequences, Sequences):
            raise KmerLrError(_lib.ERR_ARG, "use predict_resident for resident sequences")
        buf, off = flatten(sequences)
        slots = [L.kmerlr_window_slots(int(off[i + 1] - off[i]), window_size, window_step)
                 for i in range(len(off) - 1)]
        out = np.zeros(max(sum(slots), 1))
        check(L.kmerlr_score_windows(self._arr, len(self.classifiers), _p(buf), _p(off), len(off) - 1, window_size,
                                     window_step, _p(out)))
        res, p = [], 0
        for s in slots:
            res.append(out[p:p + s].copy())
            p += s
        return res

    def predict_window(self, sequences, window_size, window_step):
        """predict_window (kmerLr_predict.go:89-124), first classifier: predictions[i][j] for the window at j"""
        buf, off = flatten(sequences)
        slots = [max(int(off[i + 1] - off[i]) - window_size, 0) for i in range(len(off) - 1)]
        out = np.zeros(max(sum(slots), 1))
        check(lib().kmerlr_predict_windows(self._arr, _p(buf), _p(off), len(off) - 1, window_size, window_step, _p(out)))
        res, p = [], 0
        for s in slots:
            res.append(out[p:p + s].copy())
            p += s
        return res

    def predict_resident(self, sequences, window_size, window_step, fetch=False, total_slots=0):
        """scores of a resident set (Sequences, import_fasta, Sequences.regions); fetch: the total_slots scores"""
        out = np.zeros(max(total_slots, 1)) if fetch else None
        check(lib().kmerlr_score_windows_resident(self._arr, len(self.classifiers), sequences.h, window_size,
                                                  window_step, _p(out), None))
        return out


# ---------------------------------------------------------------------------------------------------
# on-disk formats either side of the path (SURVEY 8f-4)
# ---------------------------------------------------------------------------------------------------
def wiggle_records(predictions):
    """the "%0.15f\n" records of exp(prediction), formatted on the device: (bytes, number of irregular records)"""
    pred = np.ascontiguousarray(predictions, dtype=np.float64)
    out = np.zeros(max(18 * len(pred), 1), dtype=np.uint8)
    irr = C.c_int64(0)
    check(lib().kmerlr_wiggle_records(_p(pred), len(pred), _p(out), C.byref(irr)))
    return out[:18 * len(pred)].tobytes(), irr.value


def saveWindowPredictionsWiggle(filename, regions, predictions, track_name, window_size, window_step, scores=None):
    """saveWindowPredictionsWiggle (kmerLr_predict_genomic.go:37-60).  regions = [(seqname, from), ...];
    predictions = one array per region (what predict_window_genomic returns), or None with `scores` = the handle
    of device-resident scores and predictions replaced by the number of slots per region."""
    names = (C.c_char_p * max(len(regions), 1))(*[r[0].encode() for r in regions])
    frm = np.array([r[1] for r in regions], dtype=np.int64)
    if scores is None:
        lens = [len(p) for p in predictions]
        pred = np.ascontiguousarray(np.concatenate([np.asarray(p, dtype=np.float64) for p in predictions])
                                    if len(predictions) else np.zeros(0))
    else:
        lens, pred = list(predictions), None
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    dummy = np.zeros(1)                       # (kept alive over the call; never read when there are no slots)
    if scores is None:
        parg = _p(pred) if len(pred) else _p(dummy)
    else:
        parg = None
    check(lib().kmerlr_save_wiggle(filename.encode(), track_name.encode(), len(regions), names, _p(frm), _p(off), parg,
                                   0 if scores is None else scores, window_size, window_step))


def class_name(counter, k, code):
    """printed name of a class (gonetics KmerClass.String): "aaaatt|aatttt" """
    buf = C.create_string_buffer(256)
    check(lib().kmerlr_class_name(C.byref(counter), int(k), int(code), buf, 256))
    return buf.value.decode()


def export_kmers(counter, filename, data, transformed=False):
    """export_kmers (kmerLr_data.go:127-174); transformed = the data went through Transform.Apply ("%e" rows)"""
    check(lib().kmerlr_export_kmers(data.h, C.byref(counter), filename.encode(), 1 if transformed else 0))


class KmerRegularizationPath:
    """the table of KmerRegularizationPath.Export (kmerLr_estimator_path.go:29-73)"""

    def __init__(self):
        self.Estimator, self.Lambda, self.Norm, self.Theta = [], [], [], []

    def Export(self, filename):
        off = np.concatenate([[0], np.cumsum([len(t) for t in self.Theta])]).astype(np.int64)
        th = np.ascontiguousarray(np.concatenate([np.asarray(t, dtype=np.float64) for t in self.Theta])
                                  if len(self.Theta) else np.zeros(0))
        est = np.asarray(self.Estimator, dtype=np.int64) if len(self.Estimator) else None
        check(lib().kmerlr_export_path(filename.encode(), len(self.Lambda), _p(est), _p(np.asarray(self.Lambda, dtype=np.float64)),
                                       _p(np.asarray(self.Norm, dtype=np.float64)), _p(off), _p(th) if len(th) else _p(np.zeros(1))))


class Trace:
    """the table of Trace.Export (kmerLr_estimator_trace.go:39-80); Duration in nanoseconds"""

    def __init__(self):
        self.Iteration, self.Nonzero, self.Change, self.Lambda, self.Loss, self.Duration = [], [], [], [], [], []

    def Export(self, filename):
        i64 = lambda v: np.asarray(v, dtype=np.int64)
        f64 = lambda v: np.asarray(v, dtype=np.float64)
        check(lib().kmerlr_export_trace(filename.encode(), len(self.Iteration), _p(i64(self.Duration)), _p(i64(self.Iteration)),
                                        _p(f64(self.Change)), _p(i64(self.Nonzero)),
                                        _p(f64(self.Lambda)) if len(self.Lambda) else None,
                                        _p(f64(self.Loss)) if len(self.Loss) else None))
