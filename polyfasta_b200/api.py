"""Host-side objects over the C ABI: Context (one GPU), Fasta (one parsed file), Alignment (packed planes in HBM).

Everything that computes runs in libpolyfasta_b200.so on the GPU; this module only moves pointers."""
import ctypes

import numpy as np

from . import _lib
from ._lib import FinalIn, FinalOut, PFA_CDS_LEN, PolyFastaError, check, lib

_default_ctx = {}


class Context:
    """one CUDA device + stream (pfa_ctx)"""

    def __init__(self, device=0):
        self._h = ctypes.c_void_p()
        check(lib().pfa_ctx_create(int(device), ctypes.byref(self._h)))
        self.device = int(device)

    @property
    def handle(self):
        if not self._h:
            raise PolyFastaError(_lib.PFA_ERR_ARG, "context is closed")
        return self._h

    def close(self):
        if self._h:
            lib().pfa_ctx_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        check(lib().pfa_ctx_sync(self.handle), self.handle)

    def trim(self):
        """return the library's cached device memory to the driver"""
        check(lib().pfa_ctx_trim(self.handle), self.handle)

    def set_stream(self, cuda_stream):
        """run the library's kernels on a caller-owned stream (int / torch.cuda.Stream.cuda_stream); None restores"""
        check(lib().pfa_ctx_set_stream(self.handle, ctypes.c_void_p(cuda_stream or 0)), self.handle)

    def set_host_threads(self, threads):
        """host threads the ingest may use to pack column chunks (0 = PFA_HOST_THREADS or all hardware threads)"""
        check(lib().pfa_ctx_set_host_threads(self.handle, int(threads)), self.handle)

    def ingest_stats(self):
        """the last upload: dict(raw_chunks, packed_chunks, dirty_chunks, threads, h2d_text_bytes, h2d_packed_bytes)"""
        out = (ctypes.c_int64 * 8)()
        check(lib().pfa_ctx_ingest_stats(self.handle, out), self.handle)
        return {"raw_chunks": out[0], "packed_chunks": out[1], "dirty_chunks": out[2], "threads": out[3],
                "h2d_text_bytes": out[4], "h2d_packed_bytes": out[5], "packed_chunks_with_validity": out[6]}

    @property
    def last_kernel(self):
        """the scan kernel of the last K2 / K4 launch as instantiated, with its grid and, for the TMA kernels, passes and
        validity records per slot, e.g. 'pfa_site_scan_tma_kernel<LPS=16,ITER=5,...> grid=148 block=512 passes_per_slot=1 ...'"""
        return lib().pfa_ctx_last_kernel(self.handle).decode()

    @property
    def launch_count(self):
        return int(lib().pfa_ctx_launch_count(self.handle))

    def finalize(self, items):
        """items: iterable of (n, S, H, seqlen, jc) -> list of (S, pi_site, theta_site, D | "NA"), the tuple
        polymorphism returns (PolyFastA.py:502-520); S == 0 gives (0, 0, 0, "NA").  fp64 on the device (K5)."""
        items = list(items)
        if not items:
            return []
        inp = (FinalIn * len(items))()
        for i, (n, S, H, seqlen, jc) in enumerate(items):
            inp[i] = FinalIn(int(n), int(S), int(H), float(seqlen), int(bool(jc)), 0)
        out = (FinalOut * len(items))()
        check(lib().pfa_finalize(self.handle, inp, out, len(items)), self.handle)
        res = []
        for (n, S, H, seqlen, jc), o in zip(items, out):
            if o.no_var:
                res.append((0, 0, 0, "NA"))
            else:
                res.append((int(S), o.pi_site, o.theta_site, "NA" if o.D_is_NA else o.D))
        return res

    def cds_ssites(self, cds_rows):
        """[k][PFA_CDS_LEN] int64 -> synonymous-site counts (fp64 on the device)"""
        arr = np.ascontiguousarray(cds_rows, dtype=np.int64).reshape(-1, PFA_CDS_LEN)
        out = np.zeros(arr.shape[0], dtype=np.float64)
        check(lib().pfa_cds_ssites(self.handle, arr.ctypes.data, out.ctypes.data, arr.shape[0]), self.handle)
        return out


def synth_text_device(ctx, d_ptr, ld, n, seed, p_seg_ppm=50000, tri_ppm=10000, col_begin=0, col_end=0):
    """fill device memory with the synthetic alignment as text (benchmark input)"""
    check(lib().pfa_synth_text_device(ctx.handle, ctypes.c_void_p(d_ptr), ld, n, seed, p_seg_ppm, tri_ppm, col_begin, col_end),
          ctx.handle)


def default_context(device=0):
    ctx = _default_ctx.get(device)
    if ctx is None or not ctx._h:
        ctx = _default_ctx[device] = Context(device)
    return ctx


class NotFasta(Exception):
    """the reference would print '# file ... is not FASTA!' (PolyFastA.py:246-248)"""


class Fasta:
    """one parsed FASTA file on the host (pfa_fasta); parsing follows readfasta (PolyFastA.py:227-250)"""

    def __init__(self, handle):
        self._h = handle
        L = lib()
        self.nseq = int(L.pfa_fasta_nseq(handle))
        self.seqlen = int(L.pfa_fasta_seqlen(handle))  # -1 when rows differ in length
        self._headers = None

    @classmethod
    def from_file(cls, path):
        h = ctypes.c_void_p()
        rc = lib().pfa_fasta_parse_file(str(path).encode(), ctypes.byref(h))
        return cls._wrap(rc, h, path)

    @classmethod
    def from_bytes(cls, data):
        if isinstance(data, str):
            data = data.encode("utf-8", "surrogateescape")
        h = ctypes.c_void_p()
        buf = ctypes.create_string_buffer(data, len(data)) if data else None
        rc = lib().pfa_fasta_parse_buffer(buf, len(data), ctypes.byref(h))
        return cls._wrap(rc, h, "<buffer>")

    @classmethod
    def _wrap(cls, rc, h, what):
        if rc == _lib.PFA_ERR_NOT_FASTA:
            raise NotFasta(what)
        if rc == _lib.PFA_ERR_IO:
            raise OSError("cannot read %s" % what)
        if rc == _lib.PFA_ERR_NON_ASCII:
            raise ValueError("%s: non-ASCII bytes in sequence lines are not supported" % what)
        check(rc)
        return cls(h)

    def export_layout(self):
        """where the rows of a large file parsed in place are (bytes), for the other ranks of a column-sharded run; None when
        this file is not mapped in place"""
        n = int(lib().pfa_fasta_layout_bytes(self._h))
        if n == 0:
            return None
        buf = ctypes.create_string_buffer(n)
        check(lib().pfa_fasta_export_layout(self._h, buf, n))
        return buf.raw

    @classmethod
    def from_layout(cls, path, blob):
        """map `path` and adopt the row layout another rank exported: no line scan, no byte of the file is read"""
        h = ctypes.c_void_p()
        rc = lib().pfa_fasta_import_layout(str(path).encode(), blob, len(blob), ctypes.byref(h))
        return cls._wrap(rc, h, path)

    @property
    def handle(self):
        return self._h

    @property
    def headers(self):
        if self._headers is None:
            L = lib()
            out = []
            n = ctypes.c_int64()
            for i in range(self.nseq):
                ptr = L.pfa_fasta_header(self._h, i, ctypes.byref(n))
                out.append(ctypes.string_at(ptr, n.value).decode("utf-8", "surrogateescape") if n.value else "")
            self._headers = out
        return self._headers

    def row_lengths(self):
        L = lib()
        return [int(L.pfa_fasta_row_len(self._h, i)) for i in range(self.nseq)]

    def row(self, i):
        """upper-cased sequence i as str"""
        n = int(lib().pfa_fasta_row_len(self._h, i))
        buf = ctypes.create_string_buffer(max(n, 1))
        check(lib().pfa_fasta_copy_row(self._h, i, buf, n))
        return buf.raw[:n].decode("latin-1")

    def as_dict(self):
        """{header: SEQUENCE}, what readfasta returns"""
        return {h: self.row(i) for i, h in enumerate(self.headers)}

    def close(self):
        if self._h:
            lib().pfa_fasta_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def rows_to_masks(wn, row_lists):
    """list of row-index lists -> uint32 [k][wn] bit masks for pfa_aln_set_pops (wn = pfa_aln_mask_words)"""
    m = np.zeros((len(row_lists), max(wn, 1)), dtype=np.uint32)
    for q, rows in enumerate(row_lists):
        r = np.asarray(list(rows), dtype=np.int64)
        if r.size:
            np.bitwise_or.at(m[q], r >> 5, (np.uint32(1) << (r & 31).astype(np.uint32)))
    return m


class Alignment:
    """one alignment, or one column shard of it, packed in HBM (pfa_aln)"""

    def __init__(self, ctx, handle):
        self.ctx = ctx
        self._h = handle
        L = lib()
        self.n = int(L.pfa_aln_nseq(handle))
        self.nsites = int(L.pfa_aln_nsites(handle))

    # ---- constructors ----
    @classmethod
    def from_fasta(cls, ctx, fasta, col_begin=0, col_end=None):
        if fasta.seqlen < 0:
            raise PolyFastaError(_lib.PFA_ERR_RAGGED, "sequences do not have the same length")
        col_end = fasta.seqlen if col_end is None else col_end
        h = ctypes.c_void_p()
        check(lib().pfa_aln_from_fasta(ctx.handle, fasta.handle, col_begin, col_end, ctypes.byref(h)), ctx.handle)
        return cls(ctx, h)

    @classmethod
    def from_rows(cls, ctx, mat, col_begin=0, col_end=None):
        """mat: uint8 [n][L] row-major host matrix (numpy array, or anything with __array_interface__)"""
        mat = np.asarray(mat)
        if mat.dtype != np.uint8 or mat.ndim != 2:
            raise ValueError("expected a 2-D uint8 matrix")
        if mat.shape[1] and mat.strides[1] != 1:
            mat = np.ascontiguousarray(mat)
        n, L = mat.shape
        ld = mat.strides[0] if n > 1 else max(L, 1)
        col_end = L if col_end is None else col_end
        h = ctypes.c_void_p()
        check(lib().pfa_aln_from_rows(ctx.handle, mat.ctypes.data, n, L, ld, col_begin, col_end, ctypes.byref(h)), ctx.handle)
        a = cls(ctx, h)
        return a

    @classmethod
    def from_host_ptr(cls, ctx, ptr, n, L, ld, col_begin=0, col_end=None):
        """raw host pointer (e.g. a pinned torch tensor's data_ptr())"""
        col_end = L if col_end is None else col_end
        h = ctypes.c_void_p()
        check(lib().pfa_aln_from_rows(ctx.handle, ctypes.c_void_p(ptr), n, L, ld, col_begin, col_end, ctypes.byref(h)), ctx.handle)
        return cls(ctx, h)

    @classmethod
    def from_device_ptr(cls, ctx, ptr, n, L, ld, col_begin=0, col_end=None):
        col_end = L if col_end is None else col_end
        h = ctypes.c_void_p()
        check(lib().pfa_aln_from_device_rows(ctx.handle, ctypes.c_void_p(ptr), n, L, ld, col_begin, col_end, ctypes.byref(h)),
              ctx.handle)
        return cls(ctx, h)

    @classmethod
    def from_strings(cls, ctx, seqs, col_begin=0, col_end=None):
        """list of equal-length str/bytes (any case)"""
        n = len(seqs)
        L = len(seqs[0]) if n else 0
        mat = np.zeros((n, max(L, 1)), dtype=np.uint8)
        for i, s in enumerate(seqs):
            b = s.encode("latin-1") if isinstance(s, str) else bytes(s)
            if len(b) != L:
                raise PolyFastaError(_lib.PFA_ERR_RAGGED, "sequences do not have the same length")
            if L:
                mat[i, :L] = np.frombuffer(b, dtype=np.uint8)
        return cls.from_rows(ctx, mat[:, :L] if L else mat[:, :0], col_begin, col_end)

    @classmethod
    def synthetic(cls, ctx, n, L, seed, p_seg_ppm=50000, tri_ppm=10000, col_begin=0, col_end=None):
        col_end = L if col_end is None else col_end
        h = ctypes.c_void_p()
        check(lib().pfa_aln_synthetic(ctx.handle, n, L, seed, p_seg_ppm, tri_ppm, col_begin, col_end, ctypes.byref(h)), ctx.handle)
        return cls(ctx, h)

    # ---- housekeeping ----
    @property
    def handle(self):
        if not self._h:
            raise PolyFastaError(_lib.PFA_ERR_ARG, "alignment is freed")
        return self._h

    def free(self):
        if self._h:
            lib().pfa_aln_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    @property
    def num_escapes(self):
        return int(lib().pfa_aln_num_escapes(self.handle))

    @property
    def has_invalid(self):
        return bool(lib().pfa_aln_has_invalid(self.handle))

    def poke_gaps(self, seed, gap_ppm):
        """turn gap_ppm cells per million into '-' (synth.poke_gaps is the numpy twin)"""
        check(lib().pfa_aln_poke_gaps(self.handle, int(seed), int(gap_ppm)), self.ctx.handle)

    def force_validity(self, flag=True):
        """benchmarking: make the scans read the validity plane even for a pure-ACGT shard"""
        check(lib().pfa_aln_force_validity(self.handle, int(bool(flag))), self.ctx.handle)

    @property
    def plane_alloc(self):
        """where the planes live: "pool", "vmm" or "compressible" (PFA_PLANE_ALLOC at the time of the upload)"""
        return ("pool", "vmm", "compressible")[lib().pfa_aln_plane_alloc(self.handle)]

    @property
    def packed_bytes(self):
        return int(lib().pfa_aln_packed_bytes(self.handle))

    def read_probe(self, planes=2, reps=5):
        """ms per pass of a kernel that only reads the first `planes` planes (the read-only ceiling for these bytes)"""
        ms = ctypes.c_double()
        check(lib().pfa_aln_read_probe(self.handle, planes, reps, ctypes.byref(ms)), self.ctx.handle)
        return ms.value

    def plane(self, which):
        """uint32 [nsites][4*Wq] copy of plane 0 (b0), 1 (b1) or 2 (v)"""
        out = np.zeros((self.nsites, self.mask_words), dtype=np.uint32)
        check(lib().pfa_aln_copy_plane(self.handle, which, out.ctypes.data, out.nbytes), self.ctx.handle)
        return out

    # ---- populations ----
    def set_pops(self, row_lists):
        """row_lists: list of row-index iterables (one per population, in output order); None/[] = all rows"""
        if not row_lists:
            check(lib().pfa_aln_set_pops(self.handle, None, 0), self.ctx.handle)
            return
        m = rows_to_masks(self.mask_words, row_lists)
        check(lib().pfa_aln_set_pops(self.handle, m.ctypes.data, len(row_lists)), self.ctx.handle)

    @property
    def mask_words(self):
        return int(lib().pfa_aln_mask_words(self.handle))

    @property
    def num_pops(self):
        return int(lib().pfa_aln_num_pops(self.handle))

    def pop_sizes(self):
        return [int(lib().pfa_aln_pop_size(self.handle, q)) for q in range(self.num_pops)]

    # ---- scans ----
    def site_len(self):
        return int(lib().pfa_site_len(self.handle))

    def site_offsets(self):
        return [int(lib().pfa_site_offset(self.handle, q)) for q in range(self.num_pops + 1)]

    def unpack_site(self, vec):
        """int64 result vector -> list of dict(n, S, H, sfs) per population"""
        off = self.site_offsets()
        sizes = self.pop_sizes()
        return [{"n": sizes[q], "S": int(vec[off[q]]), "H": int(vec[off[q] + 1]),
                 "sfs": [int(x) for x in vec[off[q] + 2: off[q + 1]]]} for q in range(len(sizes))]

    def site_stats(self, want_isvar=False):
        """K2 -> list of dict(n, S, H, sfs[, isvar]) per population"""
        out = np.zeros(max(self.site_len(), 1), dtype=np.int64)
        k = self.num_pops
        isvar = np.zeros((k, max(self.nsites, 1)), dtype=np.uint8) if want_isvar else None
        check(lib().pfa_site_stats(self.handle, out.ctypes.data, isvar.ctypes.data if want_isvar else None), self.ctx.handle)
        res = self.unpack_site(out)
        if want_isvar:
            flat = isvar.reshape(-1)[: k * self.nsites].reshape(k, self.nsites) if self.nsites else isvar[:, :0]
            for q in range(k):
                res[q]["isvar"] = flat[q]
        return res

    def site_stats_device(self, d_out_ptr, d_isvar_ptr=None):
        """asynchronous K2 into caller device memory (int64[site_len]); for the multi-GPU all-reduce"""
        check(lib().pfa_site_stats_device(self.handle, ctypes.c_void_p(d_out_ptr), ctypes.c_void_p(d_isvar_ptr or 0)),
              self.ctx.handle)

    def site_stats_xchg(self, xchg, d_out_ptr, d_isvar_ptr=None):
        """K2 fused with the sum over the column shards of all ranks (one launch): d_out gets the whole alignment's vector"""
        check(lib().pfa_site_stats_xchg(self.handle, xchg.handle, ctypes.c_void_p(d_out_ptr), ctypes.c_void_p(d_isvar_ptr or 0)),
              self.ctx.handle)

    def cds_stats_xchg(self, xchg, d_out_ptr, d_labels_ptr=None):
        """K4 fused with the sum over the column shards of all ranks"""
        check(lib().pfa_cds_stats_xchg(self.handle, xchg.handle, ctypes.c_void_p(d_out_ptr), ctypes.c_void_p(d_labels_ptr or 0)),
              self.ctx.handle)

    def site_cds_stats_xchg(self, xchg, d_out_ptr, d_isvar_ptr=None, d_labels_ptr=None):
        """K2 + K4 with ONE exchange: d_out (device int64[site_len + 71 k]) = the site vector, then the codon vectors"""
        check(lib().pfa_site_cds_stats_xchg(self.handle, xchg.handle, ctypes.c_void_p(d_out_ptr), ctypes.c_void_p(d_isvar_ptr or 0),
                                            ctypes.c_void_p(d_labels_ptr or 0)), self.ctx.handle)

    @staticmethod
    def unpack_cds(row):
        return {"nstops": int(row[0]), "missing": int(row[1]), "S_s": int(row[2]), "H_s": int(row[3]), "S_n": int(row[4]),
                "H_n": int(row[5]), "sum3_by_len": {l: int(row[6 + l]) for l in range(65) if row[6 + l]}}

    def cds_stats(self, want_labels=False):
        """K4 -> list of dict(nstops, missing, S_s, H_s, S_n, H_n, sum3_by_len, ssites[, labels]) per population"""
        k = self.num_pops
        out = np.zeros((k, PFA_CDS_LEN), dtype=np.int64)
        labels = np.zeros((k, max(self.nsites, 1)), dtype=np.uint8) if want_labels else None
        check(lib().pfa_cds_stats(self.handle, out.ctypes.data, labels.ctypes.data if want_labels else None), self.ctx.handle)
        ss = self.ctx.cds_ssites(out)
        res = []
        for q in range(k):
            d = self.unpack_cds(out[q])
            d["ssites"] = float(ss[q])
            d["raw"] = out[q].copy()
            if want_labels:
                d["labels"] = labels.reshape(-1)[: k * self.nsites].reshape(k, self.nsites)[q] if self.nsites else labels[q, :0]
            res.append(d)
        return res

    def cds_stats_device(self, d_out_ptr, d_labels_ptr=None):
        check(lib().pfa_cds_stats_device(self.handle, ctypes.c_void_p(d_out_ptr), ctypes.c_void_p(d_labels_ptr or 0)),
              self.ctx.handle)

    def pairwise_xchg(self, xchg, d_out_ptr):
        """K3 on this rank's column shard + the sum over all ranks: d_out (device int64[k]) = sums of the whole alignment"""
        check(lib().pfa_pairwise_xchg(self.handle, xchg.handle, ctypes.c_void_p(d_out_ptr)), self.ctx.handle)

    def pairwise(self, want_matrix=False):
        """K3 -> (list of sum_{i<j} d_ij per population, optional int32 [n][n] matrix over all rows)"""
        k = self.num_pops
        out = np.zeros(k, dtype=np.int64)
        mat = np.zeros((self.n, self.n), dtype=np.int32) if want_matrix else None
        check(lib().pfa_pairwise(self.handle, out.ctypes.data, mat.ctypes.data if want_matrix else None), self.ctx.handle)
        return ([int(x) for x in out], mat) if want_matrix else [int(x) for x in out]


class Exchange:
    """sum of the per-shard vectors over NVLink peer memory, fused into the scan kernels (pfa_xchg).  One per rank;
    polyfasta_b200.parallel.connect_exchange builds and connects it across the ranks of a torch.distributed group."""

    HANDLE_BYTES = 64

    def __init__(self, ctx, cap_words):
        self.ctx = ctx
        self._h = ctypes.c_void_p()
        check(lib().pfa_xchg_create(ctx.handle, int(cap_words), ctypes.byref(self._h)), ctx.handle)
        self.rank, self.world = 0, 0

    @property
    def handle(self):
        if not self._h:
            raise PolyFastaError(_lib.PFA_ERR_ARG, "exchange is closed")
        return self._h

    @property
    def capacity(self):
        return int(lib().pfa_xchg_capacity(self.handle))

    def export(self):
        """the CUDA IPC handle of this rank's buffer (bytes), to be all-gathered by the host"""
        buf = ctypes.create_string_buffer(self.HANDLE_BYTES)
        check(lib().pfa_xchg_export(self.handle, buf), self.ctx.handle)
        return buf.raw

    def connect(self, rank, world, handles):
        """handles: the exported handles of all ranks, in rank order"""
        blob = b"".join(handles)
        if len(blob) != world * self.HANDLE_BYTES:
            raise ValueError("expected %d handles of %d bytes" % (world, self.HANDLE_BYTES))
        check(lib().pfa_xchg_connect(self.handle, rank, world, ctypes.create_string_buffer(blob, len(blob))), self.ctx.handle)
        self.rank, self.world = rank, world

    @staticmethod
    def connect_local(exchanges):
        """several ranks inside ONE process (tests): exchanges[r] is rank r; the buffers must be addressable from every
        device involved (same device, or peer access enabled)"""
        world = len(exchanges)
        bases = (ctypes.c_void_p * world)(*[lib().pfa_xchg_base(x.handle) for x in exchanges])
        for r, x in enumerate(exchanges):
            check(lib().pfa_xchg_connect_ptrs(x.handle, r, world, bases), x.ctx.handle)
            x.rank, x.world = r, world

    def timed_out(self):
        """True when a wait gave up because a rank never arrived (synchronises the stream)"""
        st = ctypes.c_int()
        check(lib().pfa_xchg_status(self.handle, ctypes.byref(st)), self.ctx.handle)
        return bool(st.value)

    def set_timeout_ms(self, ms):
        """how long an exchange waits for a missing rank before it reports a timeout (default 4 s / PFA_XCHG_TIMEOUT_MS)"""
        check(lib().pfa_xchg_set_timeout_ms(self.handle, int(ms)), self.ctx.handle)

    def stamps(self):
        """ns between the stages of the last exchange on this rank: dict(scan, push, fence, wait, copy); scan = first block's start to the last block's arrival (K2 only)"""
        t = (ctypes.c_uint64 * 8)()
        check(lib().pfa_xchg_stamps(self.handle, t), self.ctx.handle)
        return {"scan": t[0] - t[5] if t[5] else None, "push": t[1] - t[0], "fence": t[2] - t[1], "wait": t[3] - t[2], "copy": t[4] - t[3]}

    def allreduce(self, d_ptr, length):
        """in-place sum over ranks of an int64 device vector produced elsewhere (K3 pairwise sums)"""
        check(lib().pfa_xchg_allreduce(self.handle, ctypes.c_void_p(d_ptr), int(length)), self.ctx.handle)

    def close(self):
        if self._h:
            lib().pfa_xchg_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def parse_files(paths, threads=0):
    """parse many FASTA files with host threads -> list of Fasta | NotFasta | OSError | ValueError instances, in order"""
    n = len(paths)
    if n == 0:
        return []
    arr = (ctypes.c_char_p * n)(*[str(x).encode() for x in paths])
    out = (ctypes.c_void_p * n)()
    status = (ctypes.c_int * n)()
    check(lib().pfa_fasta_parse_files(arr, n, threads, out, status))
    res = []
    for i in range(n):
        rc = status[i]
        if rc == _lib.PFA_OK:
            res.append(Fasta(ctypes.c_void_p(out[i])))
        elif rc == _lib.PFA_ERR_NOT_FASTA:
            res.append(NotFasta(paths[i]))
        elif rc == _lib.PFA_ERR_IO:
            res.append(OSError("cannot read %s" % paths[i]))
        elif rc == _lib.PFA_ERR_NON_ASCII:
            res.append(ValueError("%s: non-ASCII bytes in sequence lines are not supported" % paths[i]))
        else:
            res.append(PolyFastaError(rc, "parse failed: %s" % paths[i]))
    return res


def match_mask(fasta, key):
    """(mask uint32[mask_words_for(n)], number of rows) of the headers containing `key` (PolyFastA.py:125)"""
    words = int(lib().pfa_mask_words_for(fasta.nseq))
    m = np.zeros(max(words, 1), dtype=np.uint32)
    kb = key.encode("utf-8", "surrogateescape")
    hits = int(lib().pfa_fasta_match_mask(fasta.handle, kb, len(kb), m.ctypes.data, words))
    return m, hits


class Batch:
    """many small loci, one upload + a few segmented launches + one synchronisation (pfa_batch): the site scan and, with
    cds=True, the codon scan of every locus"""

    MAX_ROWS = 16384          # Wq <= 128: the batched site kernel keeps a site record in registers
    MAX_LOCUS_BYTES = 64 << 20

    def __init__(self, ctx):
        self.ctx = ctx
        self._h = ctypes.c_void_p()
        check(lib().pfa_batch_create(ctx.handle, ctypes.byref(self._h)), ctx.handle)

    def close(self):
        if self._h:
            lib().pfa_batch_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def clear(self):
        check(lib().pfa_batch_clear(self._h), self.ctx.handle)

    def __len__(self):
        return int(lib().pfa_batch_size(self._h))

    @property
    def text_bytes(self):
        return int(lib().pfa_batch_text_bytes(self._h))

    @classmethod
    def fits(cls, fasta):
        return fasta.seqlen >= 0 and fasta.nseq <= cls.MAX_ROWS and fasta.nseq * max(fasta.seqlen, 1) <= cls.MAX_LOCUS_BYTES

    def add(self, fasta, masks=None):
        """masks: None (all rows) or uint32 [k][mask_words_for(n)]; returns the locus index"""
        idx = ctypes.c_int64()
        if masks is None:
            check(lib().pfa_batch_add(self._h, fasta.handle, None, 0, ctypes.byref(idx)), self.ctx.handle)
        else:
            m = np.ascontiguousarray(masks, dtype=np.uint32)
            check(lib().pfa_batch_add(self._h, fasta.handle, m.ctypes.data, m.shape[0], ctypes.byref(idx)), self.ctx.handle)
        return idx.value

    def add_rows(self, mat, row_lists=None):
        mat = np.ascontiguousarray(mat, dtype=np.uint8)
        n, L = mat.shape
        idx = ctypes.c_int64()
        if row_lists:
            m = rows_to_masks(int(lib().pfa_mask_words_for(n)), row_lists)
            check(lib().pfa_batch_add_rows(self._h, mat.ctypes.data, n, L, max(L, 1), m.ctypes.data, len(row_lists), ctypes.byref(idx)),
                  self.ctx.handle)
        else:
            check(lib().pfa_batch_add_rows(self._h, mat.ctypes.data, n, L, max(L, 1), None, 0, ctypes.byref(idx)), self.ctx.handle)
        return idx.value

    def add_synthetic(self, n, L, seed, p_seg_ppm=50000, tri_ppm=10000, row_lists=None):
        """a locus of the synthetic generator, produced on the device when the batch is staged (benchmarks)"""
        idx = ctypes.c_int64()
        if row_lists:
            m = rows_to_masks(int(lib().pfa_mask_words_for(n)), row_lists)
            check(lib().pfa_batch_add_synthetic(self._h, n, L, seed, p_seg_ppm, tri_ppm, m.ctypes.data, len(row_lists), ctypes.byref(idx)),
                  self.ctx.handle)
        else:
            check(lib().pfa_batch_add_synthetic(self._h, n, L, seed, p_seg_ppm, tri_ppm, None, 0, ctypes.byref(idx)), self.ctx.handle)
        return idx.value

    def add_files(self, paths, keys=(), threads=0):
        """read + parse + population split + append of many files in one native call (host threads).
        -> list of dict(status, n, L, locus, hits[list per key, or [n] without keys])"""
        n = len(paths)
        if n == 0:
            return []
        nk = max(len(keys), 1)
        parr = (ctypes.c_char_p * n)(*[str(x).encode() for x in paths])
        karr = (ctypes.c_char_p * max(len(keys), 1))(*[k.encode("utf-8", "surrogateescape") for k in keys]) if keys else None
        status = (ctypes.c_int * n)()
        shape = (ctypes.c_int64 * (2 * n))()
        locus = (ctypes.c_int64 * n)()
        hits = (ctypes.c_int64 * (n * nk))()
        check(lib().pfa_batch_add_files(self._h, parr, n, karr, len(keys), threads, status, shape, locus, hits), self.ctx.handle)
        return [{"status": status[i], "n": shape[2 * i], "L": shape[2 * i + 1], "locus": locus[i],
                 "hits": [hits[i * nk + j] for j in range(nk)]} for i in range(n)]

    def run(self, jc=False, cds=False):
        if cds:
            check(lib().pfa_batch_run_cds(self._h, int(bool(jc))), self.ctx.handle)
        else:
            check(lib().pfa_batch_run(self._h, int(bool(jc))), self.ctx.handle)

    def stage(self):
        """upload + encode: the planes of every locus stay resident until release() / clear()"""
        check(lib().pfa_batch_stage(self._h), self.ctx.handle)

    def scan(self, jc=False, cds=False):
        """the segmented scans over the staged batch (may be repeated)"""
        check(lib().pfa_batch_scan(self._h, int(bool(jc)), int(bool(cds))), self.ctx.handle)

    def release(self):
        check(lib().pfa_batch_release(self._h), self.ctx.handle)

    def kernel_ms(self):
        """(site scan ms, codon scan ms) of the last scan, device time"""
        a, b = ctypes.c_double(), ctypes.c_double()
        check(lib().pfa_batch_kernel_ms(self._h, ctypes.byref(a), ctypes.byref(b)), self.ctx.handle)
        return a.value, b.value

    def shape(self):
        """(bases, bytes of one plane) of the batch"""
        a, b = ctypes.c_int64(), ctypes.c_int64()
        check(lib().pfa_batch_shape(self._h, ctypes.byref(a), ctypes.byref(b)), self.ctx.handle)
        return a.value, b.value

    def result_cds(self, locus, pop=0):
        """dict(nstops, missing, S_s, H_s, S_n, H_n, sum3_by_len, ssites, raw, poly_s, poly_n) of the codon scan"""
        raw = np.zeros(PFA_CDS_LEN, dtype=np.int64)
        ss = ctypes.c_double()
        fin = (FinalOut * 2)()
        check(lib().pfa_batch_result_cds(self._h, locus, pop, raw.ctypes.data, ctypes.byref(ss), fin), self.ctx.handle)
        d = Alignment.unpack_cds(raw)
        d["ssites"], d["raw"] = ss.value, raw

        def poly(S, o):
            return (0, 0, 0, "NA") if o.no_var else (int(S), o.pi_site, o.theta_site, "NA" if o.D_is_NA else o.D)
        d["poly_s"], d["poly_n"] = poly(d["S_s"], fin[0]), poly(d["S_n"], fin[1])
        return d

    def result(self, locus, pop=0, want_sfs=False):
        """dict(n, S, H[, sfs], poly) with poly = the tuple polymorphism returns"""
        counts = (ctypes.c_int64 * 3)()
        fin = FinalOut()
        check(lib().pfa_batch_result(self._h, locus, pop, counts, None, ctypes.byref(fin)), self.ctx.handle)
        res = {"n": counts[0], "S": counts[1], "H": counts[2]}
        if want_sfs:
            sfs = np.zeros(max(counts[0] // 2, 1), dtype=np.int64)
            check(lib().pfa_batch_result(self._h, locus, pop, counts, sfs.ctypes.data, None), self.ctx.handle)
            res["sfs"] = sfs[: counts[0] // 2].tolist()
        res["poly"] = (0, 0, 0, "NA") if fin.no_var else (counts[1], fin.pi_site, fin.theta_site, "NA" if fin.D_is_NA else fin.D)
        return res
