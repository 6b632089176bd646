"""B200 drop-in for ``mixemt.preprocess.build_em_matrix``.

Mirrors the reference interface (mixemt/preprocess.py:23-96, :151-160,
:177-198): same function name, arguments, return value and exceptions; the
N x H x K Python loop is replaced by the bitset kernel in csrc/build.cu behind
the C-ABI of include/mixemt_b200.h.
"""
import ctypes
import itertools
import math
import sys

import numpy as np

from . import _lib
from ._lib import lib, check, ptr
from . import sharding
from .runtime import DeviceMatrix, RowShard, get_context, remember_resident, resident_mode


def pos_from_var(var):
    """0-based position of a SNP string such as ``'A73G'``, ``'(C16519T)'`` or
    ``'T152C!'`` (same contract as reference phylotree.py:338-350)."""
    core = var[1:-1] if var.startswith('(') else var
    core = core.rstrip('!')
    return int(core[1:-1]) - 1


def der_allele(var):
    """Upper-cased derived base of a SNP string (reference phylotree.py:353-363)."""
    return var.rstrip(')!')[-1].upper()


class HapVarBaseMatrix(object):
    """Host-side tables behind the device bitsets.

    Same construction rules as the reference class of the same name
    (preprocess.py:39-67): ``mut_prob[pos] = min(mut_max, mut_wt * (number of
    Phylotree mutations at pos))`` read from ``phylo.variants`` *as is*
    (SURVEY.md F3), and ``markers[hap][pos] = derived base`` wherever it differs
    from ``refseq[pos]``.  On top of that it lays the tables out for the GPU:

    * ``positions``  sorted variant positions, ``pos2idx`` the inverse map;
    * ``hit[p] = log(1 - mut_prob)``, ``miss[p] = log(mut_prob / 3)`` computed
      with ``math.log`` exactly like preprocess.py:75-95 does per cell;
    * a symbol alphabet (normally ``ACGT``) and, per haplotype column, the
      markers as CSR ``(position index, symbol code)``.
    """

    def __init__(self, refseq, phylo, haplogroups=None, mut_wt=0.01, mut_max=0.5):
        self.refseq = refseq
        self.phylo = phylo
        self.mut_wt = mut_wt
        self.mut_max = mut_max
        self.mut_prob = {}
        for pos in phylo.variants:
            self.mut_prob[pos] = min(mut_max, mut_wt * sum(phylo.variants[pos].values()))
        self.markers = {}
        self.add_hap_markers(phylo.hap_var)
        self.haplogroups = list(phylo.hap_var) if haplogroups is None else list(haplogroups)
        self._device = None

    def add_hap_markers(self, hap_var):
        refseq = self.refseq
        # a variant string sits on every haplogroup below its branch (Build 17: 263 826
        # entries, 10 k distinct strings): decode each string once
        decoded = {}
        for hap, variants in hap_var.items():
            table = {}
            for var in variants:
                hit = decoded.get(var)
                if hit is None:
                    pos = pos_from_var(var)
                    der = der_allele(var)
                    hit = decoded[var] = (pos, der if der != refseq[pos] else None)
                if hit[1] is not None:
                    table[hit[0]] = hit[1]
            self.markers[hap] = table

    # -- reference-compatible scalar probes (used by tests) -------------------
    def _prob(self, hap_pos, pos, base):
        expected = hap_pos[pos] if pos in hap_pos else self.refseq[pos]
        if expected == base:
            return 1.0 - self.mut_prob[pos]
        return self.mut_prob[pos] / 3.0

    # -- packing ---------------------------------------------------------------
    def pack(self):
        """Build the flat numpy tables handed to ``mxb_phylo_pack``."""
        positions = sorted(self.mut_prob)
        n_pos = len(positions)
        self.positions = np.asarray(positions, dtype=np.int64)
        pos_index = {pos: i for i, pos in enumerate(positions)}
        max_pos = (max(positions) + 1) if positions and max(positions) >= 0 else 0
        self.pos2idx = np.full(max_pos, -1, dtype=np.int32)
        for pos, i in pos_index.items():
            if pos >= 0:
                self.pos2idx[pos] = i

        def _log(x):
            return math.log(x) if x > 0.0 else float("-inf")
        self.hit = np.array([_log(1.0 - self.mut_prob[p]) for p in positions], dtype=np.float64)
        self.miss = np.array([_log(self.mut_prob[p] / 3.0) for p in positions], dtype=np.float64)

        hap_tables = [self.markers[hap] for hap in self.haplogroups]  # KeyError like :93
        symbols = {self.refseq[p] for p in positions}
        for table in hap_tables:
            symbols.update(table.values())
        symbols = sorted(symbols)
        if len(symbols) > 254:
            raise ValueError("more than 254 distinct base symbols")
        self.symbols = symbols
        code_of = {s: i for i, s in enumerate(symbols)}
        self.sym2code = np.full(256, 255, dtype=np.uint8)
        for s, i in code_of.items():
            raw = s.encode("utf-8")
            if len(raw) == 1:
                self.sym2code[raw[0]] = i
        self.ref_code = np.array([code_of[self.refseq[p]] for p in positions], dtype=np.uint8)

        # markers as CSR over the haplotype columns, in the tables' own order; markers off the
        # variant table are dead data (F8).  263 826 entries at Build 17: flattened and looked up
        # with numpy (the per-entry Python loop below remains for exotic tables)
        n_tab = len(hap_tables)
        lens = np.fromiter(map(len, hap_tables), dtype=np.int64, count=n_tab)
        total = int(lens.sum())
        all_pos = np.fromiter(itertools.chain.from_iterable(hap_tables), dtype=np.int64, count=total)
        all_der = "".join(itertools.chain.from_iterable(map(dict.values, hap_tables)))
        if len(all_der) == total and all_der.isascii() and (total == 0 or all_pos.min() >= 0):
            inside = all_pos < max_pos
            idx = np.full(total, -1, dtype=np.int32)
            idx[inside] = self.pos2idx[all_pos[inside]]
            keep = idx >= 0
            code_lut = np.full(256, 255, dtype=np.uint8)
            for sym, i in code_of.items():
                if len(sym) == 1 and sym.isascii():
                    code_lut[ord(sym)] = i
            codes = code_lut[np.frombuffer(all_der.encode("ascii"), dtype=np.uint8)]
            kept_before = np.concatenate(([0], np.cumsum(keep, dtype=np.int64)))
            bounds = np.concatenate(([0], np.cumsum(lens)))
            self.marker_ptr = kept_before[bounds]
            self.marker_pos_idx = idx[keep]
            self.marker_code = codes[keep]
        else:
            ptrs = np.zeros(n_tab + 1, dtype=np.int64)
            m_pos, m_code = [], []
            for j, table in enumerate(hap_tables):
                for pos, der in table.items():
                    i = pos_index.get(pos)
                    if i is not None:
                        m_pos.append(i)
                        m_code.append(code_of[der])
                ptrs[j + 1] = len(m_pos)
            self.marker_ptr = ptrs
            self.marker_pos_idx = np.asarray(m_pos, dtype=np.int32)
            self.marker_code = np.asarray(m_code, dtype=np.uint8)
        self.n_pos, self.n_hap, self.n_sym = n_pos, len(hap_tables), max(1, len(symbols))
        return self

    def to_device(self, ctx=None):
        if self._device is not None:
            return self._device
        if not hasattr(self, "marker_ptr"):
            self.pack()
        ctx = ctx or get_context()
        handle = ctypes.c_void_p()
        check(lib.mxb_phylo_pack(ctx.handle, self.n_pos, self.n_hap, self.n_sym,
                                 ptr(self.hit), ptr(self.miss), ptr(self.ref_code),
                                 ptr(self.marker_ptr), ptr(self.marker_pos_idx),
                                 ptr(self.marker_code), ctypes.byref(handle)))
        self._device = _PhyloHandle(ctx, handle)
        return self._device


class _PhyloHandle(object):
    def __init__(self, ctx, handle):
        self.ctx, self.handle = ctx, handle

    def __del__(self):
        try:
            if self.handle:
                lib.mxb_phylo_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class SignatureCSR(object):
    """Observations of N signatures: ``row_ptr[N+1]``, ``pos_idx``, ``base_code``."""

    def __init__(self, row_ptr, pos_idx, base_code):
        self.row_ptr, self.pos_idx, self.base_code = row_ptr, pos_idx, base_code

    @property
    def n_rows(self):
        return len(self.row_ptr) - 1


_utf8_and_size = ctypes.pythonapi.PyUnicode_AsUTF8AndSize
_utf8_and_size.argtypes = [ctypes.py_object, ctypes.POINTER(ctypes.c_ssize_t)]
_utf8_and_size.restype = ctypes.c_void_p


def _flatten_signatures(reads):
    """All signatures as one byte buffer + row offsets.  Returns ``(buf, offsets)`` with ``buf``
    a ``ctypes.c_char_p`` that keeps its memory alive.  An ASCII ``str`` is its own UTF-8 form
    (CPython compact strings), so the joined text is handed to C where it lies: no second
    80 MB copy at config 2."""
    joined = "".join(reads)
    if joined.isascii():
        lens = np.fromiter(map(len, reads), dtype=np.int64, count=len(reads))
        size = ctypes.c_ssize_t(0)
        buf = ctypes.c_char_p(_utf8_and_size(joined, ctypes.byref(size)))
        if size.value != len(joined):
            raise RuntimeError("unexpected UTF-8 length of an ASCII string")
        buf._owner = joined
    else:
        enc = [r.encode("utf-8") for r in reads]
        lens = np.fromiter(map(len, enc), dtype=np.int64, count=len(enc))
        raw = b"".join(enc)
        buf = ctypes.c_char_p(raw)
        buf._owner = raw
    offsets = np.zeros(len(reads) + 1, dtype=np.int64)
    np.cumsum(lens, out=offsets[1:])
    return buf, offsets


def parse_signatures(reads, tables):
    """``pos_obs_from_sig`` (preprocess.py:151-160) for all rows at once, in C.

    Returns ``(csr, error)``; ``error`` is ``None`` or ``(row, kind, pos)`` with
    kind ``'value'`` (malformed signature -> ValueError in the reference) or
    ``'key'`` (position outside ``phylo.variants`` -> KeyError)."""
    n = len(reads)
    cbuf, offsets = _flatten_signatures(reads)
    row_ptr = np.zeros(n + 1, dtype=np.int64)
    check(lib.mxb_sig_count(cbuf, ptr(offsets), n, ptr(row_ptr)))
    total = int(row_ptr[-1])
    pos_idx = np.empty(total, dtype=np.int32)
    base_code = np.empty(total, dtype=np.uint8)
    bad_row, bad_pos = ctypes.c_int64(-1), ctypes.c_int64(0)
    rc = lib.mxb_sig_parse(cbuf, ptr(offsets), n, ptr(tables.pos2idx), len(tables.pos2idx),
                           ptr(tables.sym2code), ptr(row_ptr), ptr(pos_idx), ptr(base_code),
                           ctypes.byref(bad_row), ctypes.byref(bad_pos))
    error = None
    if rc == _lib.MXB_ERR_VALUE:
        error = (bad_row.value, "value", None)
    elif rc == _lib.MXB_ERR_KEY:
        error = (bad_row.value, "key", bad_pos.value)
    else:
        check(rc)
    return SignatureCSR(row_ptr, pos_idx, base_code), error


def build_matrix_from_csr(tables, csr, ctx=None, want_host=True, want_counts=False,
                          keep_device=False, routes_out=None):
    """Run kernel 1 on packed inputs.  Returns ``(host_matrix|None,
    match_counts|None, DeviceMatrix|None, kernel_ms)``.  ``routes_out``: an int32
    array of one entry per row, filled in place with the path that finished each row
    (``mxb_build_matrix``'s ``route_host``)."""
    ctx = ctx or get_context()
    dev = tables.to_device(ctx)
    n, h = csr.n_rows, tables.n_hap
    out = _lib.result_empty((n, h)) if want_host else None
    counts = np.empty((n, h), dtype=np.int32) if want_counts else None
    handle = ctypes.c_void_p()
    ms = ctypes.c_float(0.0)
    if routes_out is not None and (routes_out.dtype != np.int32 or routes_out.shape != (n,)):
        raise ValueError("routes_out must be an int32 array of %d entries" % n)
    check(lib.mxb_build_matrix(ctx.handle, dev.handle, n, ptr(csr.row_ptr), ptr(csr.pos_idx),
                               ptr(csr.base_code), ptr(out), ptr(counts), ptr(routes_out),
                               ctypes.byref(handle) if keep_device else None,
                               ctypes.byref(ms)))
    dmat = DeviceMatrix(ctx, handle) if keep_device else None
    return out, counts, dmat, ms.value


def _raise_like_reference(error, tables, reads):
    row, kind, pos = error
    if kind == "value":
        raise ValueError("malformed read signature in row %d: %r" % (row, reads[row][:80]))
    raise KeyError(pos)


def build_em_matrix(refseq, phylo, reads, haplogroups, args):
    """
    Returns the matrix that describes the probability of each read
    originating in each haplotype: float64, shape (len(reads), len(haplogroups)),
    C-contiguous -- the contract of reference preprocess.py:177-198.

    Raises ``KeyError`` for a haplogroup that is not in ``phylo.hap_var`` or a
    signature position that is not in ``phylo.variants``, ``ValueError`` for a
    malformed signature, in the order the reference's loops would hit them.
    """
    verbose = getattr(args, "verbose", False)
    n, h = len(reads), len(haplogroups)
    tables = HapVarBaseMatrix(refseq, phylo, haplogroups=[])
    if verbose:
        sys.stderr.write('Building EM input matrix...\n')
    if n == 0:
        if verbose:
            sys.stderr.write('Done.\n\n')
        return np.empty((0, h))

    known = [hap in tables.markers for hap in haplogroups]
    first_unknown = known.index(False) if not all(known) else None
    tables.haplogroups = [hap for hap, ok in zip(haplogroups, known) if ok]
    tables.pack()
    csr, error = parse_signatures(list(reads), tables)

    # Replay the reference's failure order: row 0 is parsed, then column 0's
    # marker table is looked up, then row 0's positions, then column 1 ...
    if error is not None and error[0] == 0 and error[1] == "value":
        _raise_like_reference(error, tables, reads)
    if first_unknown == 0:
        raise KeyError(haplogroups[0])
    if error is not None and error[0] == 0 and h > 0:
        _raise_like_reference(error, tables, reads)
    if first_unknown is not None:
        raise KeyError(haplogroups[first_unknown])
    if error is not None and (error[1] == "value" or h > 0):
        _raise_like_reference(error, tables, reads)

    keep = resident_mode(args)
    out, _, dmat, _ = build_matrix_from_csr(tables, csr, want_host=True, keep_device=keep)
    if keep and dmat is not None:
        # The device copy stays valid only while the host array is untouched:
        # hand it out read-only and let run_em reuse the HBM-resident matrix.
        out.flags.writeable = False
        remember_resident(out, dmat)
    if verbose:
        for done in range(500, n + 1, 500):
            sys.stderr.write('  processed %d fragments...\n' % done)
        sys.stderr.write('Done.\n\n')
    return out


def build_em_matrix_device(refseq, phylo, reads, haplogroups, args=None, want_counts=False):
    """Same inputs as :func:`build_em_matrix`; keeps the matrix in HBM and
    returns ``(DeviceMatrix, match_counts|None, kernel_ms)`` (no N x H copy to
    the host) for pipelines that feed ``run_em`` directly."""
    tables = HapVarBaseMatrix(refseq, phylo, haplogroups=haplogroups).pack()
    csr, error = parse_signatures(list(reads), tables)
    if error is not None:
        _raise_like_reference(error, tables, reads)
    _, counts, dmat, ms = build_matrix_from_csr(tables, csr, want_host=False,
                                                want_counts=want_counts, keep_device=True)
    return dmat, counts, ms


# ---- fragments -> signatures on binary observations (SURVEY.md 8f N1) ------------
class ReducedReads(object):
    """Unique signatures of a set of fragments, rows in the reference's order
    (``sorted(read_sigs)``, preprocess.py:219).

    ``row_ptr`` / ``pos`` / ``base`` are the rows' observations (0-based
    reference positions, ASCII bases); ``weights[r]`` the number of fragments
    carrying row ``r`` (preprocess.py:220); ``sig_of_frag[f]`` the row of fragment
    ``f``; ``frag_order`` the fragment indexes grouped by row (fragment order
    inside a row, like the id lists ``reduce_reads`` builds, :172-173)."""

    def __init__(self, row_ptr, pos, base, weights, first_frag, sig_of_frag, frag_order,
                 str_buf, str_off):
        self.row_ptr, self.pos, self.base = row_ptr, pos, base
        self.weights, self.first_frag = weights, first_frag
        self.sig_of_frag, self.frag_order = sig_of_frag, frag_order
        self._str_buf, self._str_off = str_buf, str_off
        self._signatures = None

    @property
    def n_rows(self):
        return len(self.weights)

    @property
    def signatures(self):
        """The rows as the reference's signature strings (preprocess.py:142-148)."""
        if self._signatures is None:
            text = self._str_buf.tobytes().decode("ascii")
            off = self._str_off.tolist()
            self._signatures = [text[off[i]:off[i + 1]] for i in range(self.n_rows)]
        return self._signatures

    def fragments_of_rows(self):
        """List (per row) of arrays of fragment indexes, fragment order."""
        return np.split(self.frag_order, np.cumsum(self.weights)[:-1]) if self.n_rows else []

    def csr(self, tables):
        """``SignatureCSR`` against a packed ``HapVarBaseMatrix``; raises
        ``KeyError(pos)`` for the first row holding a position that is not a
        variant site, like ``mut_prob[pos]`` does (preprocess.py:79-84)."""
        pos = self.pos.astype(np.int64)
        ok = (pos >= 0) & (pos < len(tables.pos2idx))
        idx = np.full(len(pos), -1, dtype=np.int32)
        idx[ok] = tables.pos2idx[pos[ok]]
        if (idx < 0).any():
            raise KeyError(int(pos[int(np.argmax(idx < 0))]))
        return SignatureCSR(self.row_ptr, idx, tables.sym2code[self.base])


def reduce_reads_arrays(frag_ptr, pos, base):
    """``reduce_reads`` + the ordering of ``build_em_input`` (preprocess.py:163-174,
    :218-220) for fragments given as arrays: ``frag_ptr[F+1]`` delimits each
    fragment's observations, ``pos`` (0-based, ascending inside a fragment) and
    ``base`` (ASCII codes or a bytes object).  Returns :class:`ReducedReads`."""
    frag_ptr = np.ascontiguousarray(frag_ptr, dtype=np.int64)
    pos = np.ascontiguousarray(pos, dtype=np.int32)
    if isinstance(base, (bytes, bytearray)):
        base = np.frombuffer(bytes(base), dtype=np.uint8)
    base = np.ascontiguousarray(base, dtype=np.uint8)
    n_frag = len(frag_ptr) - 1
    if n_frag < 0 or (n_frag >= 0 and len(frag_ptr) and frag_ptr[0] != 0) or \
            (n_frag > 0 and (np.diff(frag_ptr) < 0).any()) or \
            (len(frag_ptr) and frag_ptr[-1] != len(pos)) or len(pos) != len(base):
        raise ValueError("inconsistent fragment arrays")
    handle = ctypes.c_void_p()
    check(lib.mxb_reduce_reads(ptr(frag_ptr), ptr(pos), ptr(base), n_frag, ctypes.byref(handle)))
    try:
        n_sig, n_obs, n_chars = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64()
        check(lib.mxb_sigset_sizes(handle, ctypes.byref(n_sig), ctypes.byref(n_obs),
                                   ctypes.byref(n_chars)))
        n_sig, n_obs, n_chars = n_sig.value, n_obs.value, n_chars.value
        row_ptr = np.zeros(n_sig + 1, dtype=np.int64)
        r_pos = np.empty(n_obs, dtype=np.int32)
        r_base = np.empty(n_obs, dtype=np.uint8)
        weights = np.empty(n_sig, dtype=np.int64)
        first = np.empty(n_sig, dtype=np.int64)
        sig_of_frag = np.empty(n_frag, dtype=np.int64)
        frag_order = np.empty(n_frag, dtype=np.int64)
        str_buf = np.empty(n_chars, dtype=np.uint8)
        str_off = np.zeros(n_sig + 1, dtype=np.int64)
        check(lib.mxb_sigset_export(handle, ptr(row_ptr), ptr(r_pos), ptr(r_base), ptr(weights),
                                    ptr(first), ptr(sig_of_frag), ptr(frag_order), ptr(str_buf),
                                    ptr(str_off)))
    finally:
        lib.mxb_sigset_destroy(handle)
    return ReducedReads(row_ptr, r_pos, r_base, weights, first, sig_of_frag, frag_order, str_buf,
                        str_off)


def flatten_read_obs(read_obs):
    """``{read_id: {pos: base}}`` (what process_reads returns, preprocess.py:99-139)
    -> ``(ids, frag_ptr, pos, base)``; ``None`` for the arrays when an observation
    is not a single ASCII character (the caller then keeps the string route)."""
    ids = list(read_obs)
    lens, pos, bases = [], [], []
    for rid in ids:
        obs = read_obs[rid]
        keys = sorted(obs)
        lens.append(len(keys))
        pos.extend(keys)
        bases.extend(map(obs.__getitem__, keys))
    joined = "".join(bases)
    if len(joined) != len(bases) or not joined.isascii() or \
            (pos and (min(pos) < -2**31 or max(pos) >= 2**31)):
        return ids, None, None, None
    frag_ptr = np.zeros(len(ids) + 1, dtype=np.int64)
    np.cumsum(np.asarray(lens, dtype=np.int64), out=frag_ptr[1:])
    return ids, frag_ptr, np.asarray(pos, dtype=np.int32), \
        np.frombuffer(joined.encode("ascii"), dtype=np.uint8)


def reduce_reads(read_obs):
    """
    Drop-in for reference preprocess.reduce_reads (preprocess.py:163-174):
    signature string -> list of the read ids carrying it, signatures in order of
    first appearance and ids in input order, like the reference's defaultdict.
    """
    ids, frag_ptr, pos, base = flatten_read_obs(read_obs)
    if frag_ptr is None:     # exotic observations (multi-character / non-ASCII bases)
        read_sigs = {}
        for rid in ids:
            obs = read_obs[rid]
            sig = ','.join(["%d:%s" % (p, obs[p]) for p in sorted(obs)])
            read_sigs.setdefault(sig, []).append(rid)
        return read_sigs
    red = reduce_reads_arrays(frag_ptr, pos, base)
    sigs = red.signatures
    groups = red.fragments_of_rows()
    read_sigs = {}
    for row in np.argsort(red.first_frag, kind="stable").tolist():
        read_sigs[sigs[row]] = [ids[f] for f in groups[row].tolist()]
    return read_sigs


def build_em_input_arrays(frag_ptr, pos, base, refseq, phylo, args=None, keep_device=False):
    """``build_em_input`` (preprocess.py:201-227) from binary observations, without
    signature strings.  Returns ``(em_matrix, weights, haplogroups, reduced)``:
    the matrix is a host ndarray (or a ``DeviceMatrix`` with ``keep_device``),
    rows ordered like the reference's ``sorted(read_sigs)``; ``reduced`` is the
    :class:`ReducedReads` that maps rows back to fragments.

    Rows mode (``args.b200_shard == "rows"`` under torchrun with more than one
    rank): every rank passes all fragments and reduces them all (the reduction is
    deterministic, so every rank gets the same rows), then builds only its rows
    ``sharding.row_shard(N, rank, world)`` on its GPU.  The matrix is then the
    shard (a ``DeviceMatrix`` marked as one with ``keep_device``) and ``weights``
    its slice; ``haplogroups`` and ``reduced`` are whole, so the global row indexes
    of ``consumers.assign_read_indexes`` map to fragments through
    ``reduced.fragments_of_rows()``.  The repeated host reduction costs every rank
    about 1.3 s per million fragments on 8 cores."""
    red = reduce_reads_arrays(frag_ptr, pos, base)
    haplogroups = sorted(phylo.hap_var)
    tables = HapVarBaseMatrix(refseq, phylo, haplogroups=haplogroups).pack()
    if red.n_rows and (np.diff(red.row_ptr) == 0).any():
        raise ValueError("empty read signature")        # ''.split(':') in preprocess.py:158
    csr = red.csr(tables)
    ctx = get_context()
    rows_mode = getattr(args, "b200_shard", None) == "rows"
    if rows_mode:
        ctx.init_comm_from_torch()
    weights = red.weights
    if rows_mode and ctx.world > 1:
        lo, hi = sharding.row_shard(red.n_rows, ctx.rank, ctx.world)
        a, b = int(csr.row_ptr[lo]), int(csr.row_ptr[hi])
        csr = SignatureCSR(csr.row_ptr[lo:hi + 1] - a, csr.pos_idx[a:b], csr.base_code[a:b])
        weights = red.weights[lo:hi]
    out, _, dmat, _ = build_matrix_from_csr(tables, csr, ctx=ctx, want_host=not keep_device,
                                            keep_device=keep_device)
    if dmat is not None and rows_mode and ctx.world > 1:
        dmat.row_shard = RowShard(lo, red.n_rows)
    return (dmat if keep_device else out), weights, haplogroups, red
