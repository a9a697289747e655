"""ctypes binding of include/dnastore_b200.h (one class per opaque handle).

Names mirror the reference's: ``Machine.from_file`` / ``Machine.compose`` /
``Machine.to_json`` (reference src/trans.h:83-126), ``ErrorFlags`` = the CLI's
error-model flags (reference t/dnastore.cpp:69-75), ``Decoder.decode_fasta`` =
``decodeFastSeqs`` (reference src/viterbi.h:108).
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
lib_path = os.environ.get("DNAB_LIB") or os.path.join(_HERE, "libdnastore_b200.so")  # DNAB_LIB: A/B builds

if not os.path.exists(lib_path):
    raise ImportError(
        f"{lib_path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(or `make -C dnastore_b200/csrc`). There is no Python/CPU fallback."
    )
lib = C.CDLL(lib_path)

READ_OK, READ_NO_DECODING, READ_OVERFLOW, READ_TRACEBACK_FAILED = 0, 1, 2, 3


class DnabError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"dnab error {code}: {msg}")
        self.code = code


class Tables(C.Structure):
    """struct dnab_tables (include/dnab_tables.h)."""
    _fields_ = [
        ("n_states", C.c_uint32), ("k", C.c_uint32), ("local", C.c_uint32), ("n_emit", C.c_uint32), ("n_null", C.c_uint32),
        ("emit_off", C.POINTER(C.c_uint32)), ("emit_src", C.POINTER(C.c_uint32)), ("emit_score", C.POINTER(C.c_double)),
        ("emit_base", C.POINTER(C.c_uint8)), ("emit_in", C.POINTER(C.c_uint8)),
        ("null_off", C.POINTER(C.c_uint32)), ("null_src", C.POINTER(C.c_uint32)), ("null_score", C.POINTER(C.c_double)),
        ("null_in", C.POINTER(C.c_uint8)),
        ("ctx", C.POINTER(C.c_uint8)), ("mdl", C.POINTER(C.c_uint8)),
        ("noGap", C.c_double), ("delOpen", C.c_double), ("delExtend", C.c_double), ("delEnd", C.c_double), ("tanDup", C.c_double),
        ("sub", C.c_double * 16),
        ("len", C.POINTER(C.c_double)),
    ]


class ErrorFlags(C.Structure):
    """struct dnab_error_flags: the CLI's error-model flags with the reference's defaults."""
    _fields_ = [("length", C.c_int32), ("global_", C.c_int32), ("sub_prob", C.c_double), ("iv_ratio", C.c_double),
                ("dup_prob", C.c_double), ("del_open", C.c_double), ("del_ext", C.c_double)]

    def __init__(self, length=12, global_=False, sub_prob=.01, iv_ratio=10., dup_prob=.001, del_open=.001, del_ext=.01):
        super().__init__(int(length), int(bool(global_)), sub_prob, iv_ratio, dup_prob, del_open, del_ext)


class DecoderInfo(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in ("n_states", "k", "local", "cluster_size", "states_per_cta", "threads_per_cta",
                                          "smem_bytes_per_cta", "t_in_smem", "table_in_smem", "s_prev_in_smem", "n_clusters", "sm_count")]


class BatchInfo(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in ("enabled", "reads_per_group", "team_size", "states_per_cta", "warps_per_cta",
                                          "smem_bytes_per_cta", "n_teams", "wide_states")] + [("cross_cta_transition_fraction", C.c_double)]


class PipelineStats(C.Structure):
    _fields_ = [("reads", C.c_int64), ("chunks", C.c_int64), ("overflow_reruns", C.c_int64), ("parse_seconds", C.c_double),
                ("decode_busy_seconds", C.c_double), ("wall_seconds", C.c_double)]


class DecoderStats(C.Structure):
    _fields_ = [("kernel_launches", C.c_uint64), ("fill_launches", C.c_uint64), ("traceback_launches", C.c_uint64),
                ("reads", C.c_uint64), ("cells", C.c_uint64), ("last_fill_ms", C.c_double), ("last_traceback_ms", C.c_double),
                ("timed_fill_ms", C.c_double), ("timed_traceback_ms", C.c_double), ("timed_fill_launches", C.c_uint64)]


class MutatorParams(C.Structure):
    """struct dnab_mutator_params (reference MutatorParams, src/mutator.h:9-31)."""
    _fields_ = [("p_del_open", C.c_double), ("p_del_extend", C.c_double), ("p_tan_dup", C.c_double),
                ("p_transition", C.c_double), ("p_transversion", C.c_double), ("p_len", C.c_double * 16),
                ("max_dup_len", C.c_int32), ("local", C.c_int32)]

    @classmethod
    def from_flags(cls, flags):
        p = cls()
        lib.dnab_mutator_params_from_flags(C.byref(flags), C.byref(p))
        return p

    def probs(self):
        return np.array([self.p_del_open, self.p_del_extend, self.p_tan_dup, self.p_transition, self.p_transversion])

    def plen(self):
        return np.array(list(self.p_len)[:self.max_dup_len])

    def to_json(self):
        ptr = lib.dnab_mutator_params_json(C.byref(self))
        try:
            return C.string_at(ptr).decode()
        finally:
            lib.dnab_free(ptr)


class MutatorCounts(C.Structure):
    """struct dnab_mutator_counts (reference MutatorCounts, src/mutator.h:43-67)."""
    _fields_ = [("n_del_open", C.c_double), ("n_tan_dup", C.c_double), ("n_no_gap", C.c_double),
                ("n_del_extend", C.c_double), ("n_del_end", C.c_double), ("n_len", C.c_double * 16),
                ("n_sub", C.c_double * 16), ("max_dup_len", C.c_int32), ("reserved", C.c_int32)]

    def flat(self):
        """[nDelOpen, nTanDup, nNoGap, nDelExtend, nDelEnd, nLen[k], nSub[16]] -- the oracle's order."""
        return np.array([self.n_del_open, self.n_tan_dup, self.n_no_gap, self.n_del_extend, self.n_del_end]
                        + list(self.n_len)[:self.max_dup_len] + list(self.n_sub))

    def to_json(self):
        ptr = lib.dnab_mutator_counts_json(C.byref(self))
        try:
            return C.string_at(ptr).decode()
        finally:
            lib.dnab_free(ptr)


def _sig(name, restype, *argtypes):
    fn = getattr(lib, name)
    fn.restype = restype
    fn.argtypes = list(argtypes)
    return fn


_vp = C.c_void_p
_sig("dnab_last_error", C.c_char_p)
_sig("dnab_version", C.c_char_p)
_sig("dnab_free", None, _vp)
_sig("dnab_machine_load", _vp, C.c_char_p)
_sig("dnab_machine_from_json", _vp, C.c_char_p)
_sig("dnab_machine_compose", _vp, _vp, _vp)
_sig("dnab_machine_to_json", _vp, _vp)
_sig("dnab_machine_n_states", C.c_uint32, _vp)
_sig("dnab_machine_max_left_context", C.c_uint32, _vp)
_sig("dnab_machine_input_alphabet", C.c_int, _vp, C.c_int, C.c_char_p, C.c_size_t)
_sig("dnab_machine_free", None, _vp)
_sig("dnab_error_flags_default", None, C.POINTER(ErrorFlags))
_sig("dnab_compile", _vp, _vp, C.POINTER(ErrorFlags))
_sig("dnab_compile_with_error_file", _vp, _vp, C.c_char_p)
_sig("dnab_compiled_tables", C.POINTER(Tables), _vp)
_sig("dnab_compiled_free", None, _vp)
_sig("dnab_decoder_create", _vp, C.POINTER(Tables), C.c_int)
_sig("dnab_decoder_destroy", None, _vp)
_sig("dnab_decoder_get_info", C.c_int, _vp, C.POINTER(DecoderInfo))
_sig("dnab_decoder_configure", C.c_int, _vp, C.c_uint32, C.c_uint32, C.c_uint32)
_sig("dnab_decoder_get_stats", C.c_int, _vp, C.POINTER(DecoderStats))
_sig("dnab_decoder_set_timing", C.c_int, _vp, C.c_int)
_sig("dnab_decoder_reset_timing", C.c_int, _vp)
_sig("dnab_posterior_classes", C.c_int, _vp, C.c_char_p, C.c_size_t)
_sig("dnab_posterior_batch", C.c_int, _vp, C.c_int64, _vp, _vp, _vp, C.c_int32, _vp, _vp, _vp, _vp, _vp)
_sig("dnab_decoder_set_option", C.c_int, _vp, C.c_char_p, C.c_int64)
_sig("dnab_decoder_get_batch_info", C.c_int, _vp, _vp)
_sig("dnab_decoder_set_debug", C.c_int, _vp, C.c_int)
_sig("dnab_decoder_debug_counters", C.c_int, _vp, _vp)
_sig("dnab_packed_size", C.c_size_t, _vp, C.c_int64)
_sig("dnab_pack_reads", C.c_int, C.c_char_p, _vp, C.c_int64, _vp, _vp, _vp)
_sig("dnab_viterbi_batch", C.c_int, _vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, C.c_int32, _vp, _vp, _vp, C.c_int32, _vp)
_sig("dnab_viterbi_batch_device", C.c_int, _vp, C.c_int64, C.c_int32, _vp, _vp, _vp, _vp, _vp, C.c_int32, _vp, _vp, _vp)
_sig("dnab_viterbi_cells", C.c_int, _vp, _vp, C.c_int32, _vp, _vp)
_sig("dnab_forward_batch", C.c_int, _vp, C.c_int64, _vp, _vp, _vp, C.c_int32, _vp, _vp, _vp, _vp)
_sig("dnab_fwdback_counts_batch", C.c_int, _vp, C.c_int64, _vp, _vp, _vp, C.c_int32, _vp, _vp, _vp, _vp)
_sig("dnab_mutator_params_from_flags", None, C.POINTER(ErrorFlags), C.POINTER(MutatorParams))
_sig("dnab_mutator_params_json", _vp, C.POINTER(MutatorParams))
_sig("dnab_mutator_counts_json", _vp, C.POINTER(MutatorCounts))
_sig("dnab_lse_table", C.POINTER(C.c_double), C.POINTER(C.c_int32))
_sig("dnab_pair_db_load", _vp, C.c_char_p)
_sig("dnab_pair_db_count", C.c_int64, _vp)
_sig("dnab_pair_db_in_len", C.c_int32, _vp, C.c_int64)
_sig("dnab_pair_db_out_len", C.c_int32, _vp, C.c_int64)
_sig("dnab_pair_db_in", C.POINTER(C.c_uint8), _vp, C.c_int64)
_sig("dnab_pair_db_out", C.POINTER(C.c_uint8), _vp, C.c_int64)
_sig("dnab_pair_db_env_a", C.POINTER(C.c_int32), _vp, C.c_int64)
_sig("dnab_pair_db_env_b", C.POINTER(C.c_int32), _vp, C.c_int64)
_sig("dnab_pair_db_free", None, _vp)
_sig("dnab_pairhmm_set_chunk_cells", C.c_int, C.c_int64)
_sig("dnab_pairhmm_fb_batch", C.c_int, C.c_int, C.POINTER(MutatorParams), C.c_int, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp,
     _vp, _vp, _vp, C.POINTER(C.c_double))
_sig("dnab_expected_counts", C.c_int, C.c_int, C.POINTER(MutatorParams), _vp, C.c_int, C.POINTER(MutatorCounts),
     C.POINTER(C.c_double))
_sig("dnab_baum_welch", C.c_int, C.c_int, C.POINTER(MutatorParams), _vp, C.c_int, C.POINTER(MutatorParams),
     C.POINTER(C.c_int32))
_sig("dnab_decode_fasta", _vp, _vp, C.c_char_p)
_sig("dnab_multi_decoder_create", _vp, _vp, _vp, C.c_int)
_sig("dnab_multi_decoder_destroy", None, _vp)
_sig("dnab_multi_decoder_count", C.c_int, _vp)
_sig("dnab_multi_decoder_at", _vp, _vp, C.c_int)
_sig("dnab_multi_decoder_set_option", C.c_int, _vp, C.c_char_p, C.c_int64)
_sig("dnab_viterbi_batch_multi", C.c_int, _vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, C.c_int32, _vp, _vp)
_sig("dnab_decode_fasta_multi", _vp, _vp, C.c_char_p)
_sig("dnab_multi_decoder_last_stats", C.c_int, _vp, _vp)
_sig("dnab_decoded_count", C.c_int64, _vp)
_sig("dnab_decoded_name", C.c_char_p, _vp, C.c_int64)
_sig("dnab_decoded_seq", C.c_char_p, _vp, C.c_int64)
_sig("dnab_decoded_loglike", C.c_double, _vp, C.c_int64)
_sig("dnab_decoded_status", C.c_int32, _vp, C.c_int64)
_sig("dnab_decoded_free", None, _vp)
_sig("dnab_exact_decoder_create", _vp, _vp)
_sig("dnab_exact_decoder_feed", C.c_int, _vp, C.c_char_p, C.c_size_t)
_sig("dnab_exact_decoder_close", C.c_int, _vp)
_sig("dnab_exact_decoder_take_symbols", _vp, _vp)
_sig("dnab_exact_decoder_warnings", _vp, _vp)
_sig("dnab_exact_decoder_hypotheses", C.c_int64, _vp)
_sig("dnab_exact_decoder_destroy", None, _vp)
_sig("dnab_pack_decoded_symbols", C.c_int64, C.c_char_p, C.c_size_t, _vp, C.c_size_t, C.c_char_p, C.POINTER(_vp))
_sig("dnab_exact_decode_fasta", C.c_int, _vp, C.c_char_p, C.POINTER(_vp), C.POINTER(C.c_size_t), C.POINTER(_vp))


def _err(code=-1):
    return DnabError(code, lib.dnab_last_error().decode(errors="replace"))


def _ptr(a):
    return a.ctypes.data_as(_vp)


class Machine:
    """dnastore transducer handle (reference src/trans.h:83-126)."""

    def __init__(self, handle):
        if not handle:
            raise _err()
        self._h = handle

    @classmethod
    def from_file(cls, path):
        return cls(lib.dnab_machine_load(os.fspath(path).encode()))

    @classmethod
    def from_json(cls, text):
        return cls(lib.dnab_machine_from_json(text.encode()))

    @classmethod
    def compose(cls, first, second):
        """Machine::compose(first, second): first's output feeds second's input."""
        return cls(lib.dnab_machine_compose(first._h, second._h))

    @classmethod
    def load_composed(cls, base, composes=()):
        """--load-machine BASE --compose-machine C1 --compose-machine C2 ...:
        applied right to left, so the first listed is outermost (reference t/dnastore.cpp:159-165)."""
        m = cls.from_file(base)
        for c in reversed(list(composes)):
            m = cls.compose(cls.from_file(c), m)
        return m

    def to_json(self):
        p = lib.dnab_machine_to_json(self._h)
        if not p:
            raise _err()
        try:
            return C.string_at(p).decode()
        finally:
            lib.dnab_free(p)

    @property
    def n_states(self):
        return lib.dnab_machine_n_states(self._h)

    @property
    def max_left_context(self):
        return lib.dnab_machine_max_left_context(self._h)

    def input_alphabet(self, flags=2 | 8 | 16):
        buf = C.create_string_buffer(256)
        rc = lib.dnab_machine_input_alphabet(self._h, flags, buf, 256)
        if rc:
            raise _err(rc)
        return buf.value.decode()

    def compile(self, flags=None, error_file=None):
        return Compiled(self, flags, error_file)

    def __del__(self):
        if getattr(self, "_h", None):
            lib.dnab_machine_free(self._h)
            self._h = None



def _take_string(p):
    if not p:
        raise _err()
    try:
        return C.string_at(p).decode()
    finally:
        lib.dnab_free(p)


class ExactDecoder:
    """Error-free decoding on the host: the reference's ``Decoder<Writer>`` (src/decoder.h:7-190), i.e. what
    ``--decode-string`` / ``--decode-bits`` / ``-d`` drive.  ``feed`` = ``decodeString``, ``close`` = ``close``;
    ``take_symbols`` returns the input symbols resolved so far ('0', '1', '^', '$', control letters)."""

    def __init__(self, machine):
        self._machine = machine  # the C++ decoder keeps a reference to it
        self._h = lib.dnab_exact_decoder_create(machine._h)
        if not self._h:
            raise _err()

    def feed(self, bases):
        b = bases.encode()
        rc = lib.dnab_exact_decoder_feed(self._h, b, len(b))
        if rc:
            raise _err(rc)
        return self

    def close(self):
        rc = lib.dnab_exact_decoder_close(self._h)
        if rc:
            raise _err(rc)
        return self

    def take_symbols(self):
        return _take_string(lib.dnab_exact_decoder_take_symbols(self._h))

    @property
    def warnings(self):
        return _take_string(lib.dnab_exact_decoder_warnings(self._h)).splitlines()

    @property
    def hypotheses(self):
        return lib.dnab_exact_decoder_hypotheses(self._h)

    def __del__(self):
        if getattr(self, "_h", None):
            lib.dnab_exact_decoder_destroy(self._h)
            self._h = None


def exact_decode_bits(machine, dna):
    """``--decode-bits DNA`` (reference t/dnastore.cpp:205-211): the input-symbol string, e.g. ``^0001...0$``."""
    dec = ExactDecoder(machine).feed(dna).close()
    return dec.take_symbols()


def pack_decoded_symbols(symbols):
    """``BinaryWriter`` (reference src/decoder.h:193-240). Returns (bytes, leftover bits as the reference's warning
    prints them, warnings)."""
    s = symbols.encode()
    buf = C.create_string_buffer(len(s) // 8 + 1)
    left = C.create_string_buffer(16)
    warn = _vp()
    n = lib.dnab_pack_decoded_symbols(s, len(s), buf, len(s) // 8 + 1, left, C.byref(warn))
    if n < 0:
        raise _err(n)
    return buf.raw[:n], left.value.decode(), _take_string(warn.value).splitlines()


def exact_decode_string(machine, dna):
    """``--decode-string DNA`` (reference t/dnastore.cpp:199-202): the decoded bytes."""
    return pack_decoded_symbols(exact_decode_bits(machine, dna))[0]


def exact_decode_fasta(machine, path):
    """``-d/--decode-file FASTA`` (reference t/dnastore.cpp:185-190): every record through one decoder, bytes out.
    Returns (bytes, warnings)."""
    out, n, warn = _vp(), C.c_size_t(0), _vp()
    rc = lib.dnab_exact_decode_fasta(machine._h, os.fspath(path).encode(), C.byref(out), C.byref(n), C.byref(warn))
    if rc:
        raise _err(rc)
    try:
        data = C.string_at(out.value, n.value)
    finally:
        lib.dnab_free(out)
    return data, _take_string(warn.value).splitlines()

class Compiled:
    """Flat tables in host memory (include/dnab_tables.h)."""

    def __init__(self, machine, flags=None, error_file=None):
        self._machine = machine
        if error_file is not None:
            h = lib.dnab_compile_with_error_file(machine._h, os.fspath(error_file).encode())
        else:
            self.flags = flags if flags is not None else ErrorFlags()
            h = lib.dnab_compile(machine._h, C.byref(self.flags))
        if not h:
            raise _err()
        self._h = h
        self.tables = lib.dnab_compiled_tables(h)

    @property
    def t(self):
        return self.tables.contents

    def arrays(self):
        """numpy views of the tables (for tests)."""
        t = self.t
        n, k = t.n_states, t.k

        def arr(p, count, dt):
            if count == 0:
                return np.zeros(0, dtype=dt)
            return np.ctypeslib.as_array(p, shape=(count,)).astype(dt, copy=True)

        return dict(
            n_states=n, k=k, local=t.local,
            emit_off=arr(t.emit_off, n + 1, np.uint32), emit_src=arr(t.emit_src, t.n_emit, np.uint32),
            emit_score=arr(t.emit_score, t.n_emit, np.float64), emit_base=arr(t.emit_base, t.n_emit, np.uint8),
            emit_in=arr(t.emit_in, t.n_emit, np.uint8),
            null_off=arr(t.null_off, n + 1, np.uint32), null_src=arr(t.null_src, t.n_null, np.uint32),
            null_score=arr(t.null_score, t.n_null, np.float64), null_in=arr(t.null_in, t.n_null, np.uint8),
            ctx=arr(t.ctx, n * k, np.uint8), mdl=arr(t.mdl, n, np.uint8),
            noGap=t.noGap, delOpen=t.delOpen, delExtend=t.delExtend, delEnd=t.delEnd, tanDup=t.tanDup,
            sub=np.array(list(t.sub)), len=arr(t.len, k, np.float64),
        )

    def __del__(self):
        if getattr(self, "_h", None):
            lib.dnab_compiled_free(self._h)
            self._h = None


class PairDb:
    """Database of 2-row Stockholm alignments prepared for the pair-HMM lattice."""

    def __init__(self, path):
        h = lib.dnab_pair_db_load(os.fspath(path).encode())
        if not h:
            raise _err()
        self._h = h

    def __len__(self):
        return lib.dnab_pair_db_count(self._h)

    def alignment(self, i):
        """(in tokens, out tokens, env_a, env_b) as numpy arrays."""
        n_in, n_out = lib.dnab_pair_db_in_len(self._h, i), lib.dnab_pair_db_out_len(self._h, i)

        def arr(p, n, dt):
            return np.ctypeslib.as_array(p, shape=(n,)).astype(dt, copy=True) if n else np.zeros(0, dtype=dt)
        return (arr(lib.dnab_pair_db_in(self._h, i), n_in, np.uint8), arr(lib.dnab_pair_db_out(self._h, i), n_out, np.uint8),
                arr(lib.dnab_pair_db_env_a(self._h, i), n_in + 1, np.int32),
                arr(lib.dnab_pair_db_env_b(self._h, i), n_out + 1, np.int32))

    def __del__(self):
        if getattr(self, "_h", None):
            lib.dnab_pair_db_free(self._h)
            self._h = None


def pairhmm_set_chunk_cells(cells):
    """Cap on the envelope cells one pair-HMM launch keeps on the device (0 = automatic); results do not depend on it."""
    lib.dnab_pairhmm_set_chunk_cells(int(cells))


def pairhmm_fb_batch(params, aligns, strict=False, device=0):
    """aligns: list of (in_tok, out_tok, env_a, env_b). Returns (fwd_ll, back_ll, [MutatorCounts], kernel_ms)."""
    n = len(aligns)
    in_off = np.zeros(n + 1, dtype=np.int64)
    out_off = np.zeros(n + 1, dtype=np.int64)
    np.cumsum([len(a[0]) for a in aligns], out=in_off[1:])
    np.cumsum([len(a[1]) for a in aligns], out=out_off[1:])
    cat = lambda k, dt: np.ascontiguousarray(np.concatenate([a[k] for a in aligns]).astype(dt)) if n else np.zeros(1, dtype=dt)
    in_tok, out_tok, env_a, env_b = cat(0, np.uint8), cat(1, np.uint8), cat(2, np.int32), cat(3, np.int32)
    if len(in_tok) == 0:
        in_tok = np.zeros(1, dtype=np.uint8)
    if len(out_tok) == 0:
        out_tok = np.zeros(1, dtype=np.uint8)
    fwd = np.zeros(n, dtype=np.float64)
    back = np.zeros(n, dtype=np.float64)
    counts = (MutatorCounts * max(n, 1))()
    ms = C.c_double(0)
    rc = lib.dnab_pairhmm_fb_batch(int(device), C.byref(params), int(bool(strict)), n, _ptr(in_tok), _ptr(in_off), _ptr(out_tok),
                                   _ptr(out_off), _ptr(env_a), _ptr(env_b), _ptr(fwd), _ptr(back),
                                   C.cast(counts, _vp), C.byref(ms))
    if rc:
        raise _err(rc)
    return fwd, back, [counts[i] for i in range(n)], ms.value


def expected_counts(params, db, strict=False, device=0):
    total = MutatorCounts()
    ll = C.c_double(0)
    rc = lib.dnab_expected_counts(int(device), C.byref(params), db._h, int(bool(strict)), C.byref(total), C.byref(ll))
    if rc:
        raise _err(rc)
    return total, ll.value


def baum_welch(params, db, strict=False, device=0):
    fitted = MutatorParams()
    iters = C.c_int32(0)
    rc = lib.dnab_baum_welch(int(device), C.byref(params), db._h, int(bool(strict)), C.byref(fitted), C.byref(iters))
    if rc:
        raise _err(rc)
    return fitted, iters.value


def pack_reads(reads):
    """ASCII reads -> (packed uint8, byte_off int64, read_len int32): 2 bits per base."""
    n = len(reads)
    joined = "".join(reads).encode()
    base_off = np.zeros(n + 1, dtype=np.int64)
    np.cumsum([len(r) for r in reads], out=base_off[1:])
    read_len = np.diff(base_off).astype(np.int32)
    packed = np.zeros(lib.dnab_packed_size(_ptr(read_len), n), dtype=np.uint8)
    byte_off = np.zeros(n, dtype=np.int64)
    rc = lib.dnab_pack_reads(joined, _ptr(base_off), n, _ptr(packed), _ptr(byte_off), _ptr(read_len))
    if rc:
        raise _err(rc)
    return packed, byte_off, read_len


class Decoder:
    """Tables resident on one GPU + the CUDA kernels. Raises without a CUDA device."""

    def __init__(self, compiled, device=0):
        self._compiled = compiled
        h = lib.dnab_decoder_create(compiled.tables, int(device))
        if not h:
            raise _err(-2)
        self._h = h
        self.device = int(device)

    def configure(self, cluster_size=0, threads_per_cta=0, t_in_smem_mode=0):
        """Placement overrides of the push kernel (0 = automatic); set_option has the others ("table", "s_prev", ...)."""
        rc = lib.dnab_decoder_configure(self._h, cluster_size, threads_per_cta, t_in_smem_mode)
        if rc:
            raise _err(rc)

    def set_option(self, key, value):
        """Named option (include/dnastore_b200.h dnab_decoder_set_option), e.g. kernel=1 (read-batched), 2 (push)."""
        rc = lib.dnab_decoder_set_option(self._h, key.encode(), int(value))
        if rc:
            raise _err(rc)

    def batch_info(self):
        i = BatchInfo()
        rc = lib.dnab_decoder_get_batch_info(self._h, C.byref(i))
        if rc:
            raise _err(rc)
        return {n: getattr(i, n) for n, _ in BatchInfo._fields_}

    def info(self):
        i = DecoderInfo()
        rc = lib.dnab_decoder_get_info(self._h, C.byref(i))
        if rc:
            raise _err(rc)
        return {n: getattr(i, n) for n, _ in DecoderInfo._fields_}

    def stats(self):
        s = DecoderStats()
        lib.dnab_decoder_get_stats(self._h, C.byref(s))
        return {n: getattr(s, n) for n, _ in DecoderStats._fields_}

    def set_timing(self, enabled=True):
        lib.dnab_decoder_set_timing(self._h, int(enabled))

    def set_debug(self, enabled=True):
        lib.dnab_decoder_set_debug(self._h, int(enabled))

    def debug_counters(self):
        out = np.zeros(16, dtype=np.uint64)
        lib.dnab_decoder_debug_counters(self._h, _ptr(out))
        names = ["columns", "sweeps", "work_rank0", "cyc_emit", "cyc_closure", "cyc_pred", "rounds", "cyc_dense", "dirty_first", "cyc_compact", "cyc_proc", "cyc_clusterwait", "cyc_pushwait", "hops_t0"]
        return {n: int(v) for n, v in zip(names, out)}

    def reset_timing(self):
        lib.dnab_decoder_reset_timing(self._h)

    def viterbi(self, reads, want_path=False, decoded_stride=None, path_stride=None):
        """Decode ASCII reads through host buffers. Returns dict(loglike, decoded, status[, path])."""
        packed, byte_off, read_len = pack_reads(reads)
        return self.viterbi_packed(packed, byte_off, read_len, want_path, decoded_stride, path_stride)

    def viterbi_packed(self, packed, byte_off, read_len, want_path=False, decoded_stride=None, path_stride=None):
        n = len(read_len)
        max_len = int(read_len.max()) if n else 0
        stride = int(decoded_stride or (8 * max_len + 1024))
        loglike = np.zeros(n, dtype=np.float64)
        decoded = np.zeros((n, stride), dtype=np.uint8)
        dec_len = np.zeros(n, dtype=np.int32)
        status = np.zeros(n, dtype=np.int32)
        path = path_len = None
        pstride = 0
        if want_path:
            pstride = int(path_stride or (16 * max_len + 4096))
            path = np.zeros((n, pstride, 3), dtype=np.int32)
            path_len = np.zeros(n, dtype=np.int32)
        rc = lib.dnab_viterbi_batch(self._h, n, _ptr(packed), _ptr(byte_off), _ptr(read_len), _ptr(loglike), _ptr(decoded),
                                    stride, _ptr(dec_len), _ptr(status), _ptr(path) if want_path else None, pstride,
                                    _ptr(path_len) if want_path else None)
        if rc:
            raise _err(rc)
        out = dict(loglike=loglike, status=status,
                   decoded=[bytes(decoded[r, :dec_len[r]]).decode("latin1") for r in range(n)])
        if want_path:
            out["path"] = [path[r, :min(path_len[r], pstride)].copy() for r in range(n)]
            out["path_len"] = path_len
        return out

    def viterbi_cells(self, read):
        """One read; returns (loglike, cells[(L+1), n_states, k+2]) in the reference's layout."""
        packed, byte_off, read_len = pack_reads([read])
        t = self._compiled.t
        L = int(read_len[0])
        cells = np.zeros((L + 1, t.n_states, t.k + 2), dtype=np.float64)
        ll = C.c_double(0)
        rc = lib.dnab_viterbi_cells(self._h, _ptr(packed), L, C.byref(ll), _ptr(cells))
        if rc:
            raise _err(rc)
        return ll.value, cells

    def forward(self, reads, max_sweeps=0, want_cells=False):
        """Forward (sum-product) log-likelihoods over the machine lattice (SURVEY.md 8a-12; not in the
        reference, specified by oracle/forward_oracle.c). Returns dict(loglike, sweeps, status[, cells of read 0])."""
        packed, byte_off, read_len = pack_reads(reads)
        n = len(read_len)
        t = self._compiled.t
        ll = np.zeros(n, dtype=np.float64)
        sweeps = np.zeros(n, dtype=np.int64)
        status = np.zeros(n, dtype=np.int32)
        cells = np.zeros((int(read_len[0]) + 1, t.n_states, t.k + 2), dtype=np.float64) if (want_cells and n) else None
        rc = lib.dnab_forward_batch(self._h, n, _ptr(packed), _ptr(byte_off), _ptr(read_len), int(max_sweeps), _ptr(ll),
                                    _ptr(sweeps), _ptr(status), _ptr(cells) if cells is not None else None)
        if rc:
            raise _err(rc)
        out = dict(loglike=ll, sweeps=sweeps, status=status)
        if cells is not None:
            out["cells"] = cells
        return out

    def fwdback_counts(self, reads, max_sweeps=0):
        """Forward + backward over the machine lattice and the posterior expected counts of the error-model
        events per read: dict(loglike, loglike_back, counts[n, 5+k+16], status). Not in the reference (8a-12)."""
        packed, byte_off, read_len = pack_reads(reads)
        n = len(read_len)
        t = self._compiled.t
        ll = np.zeros(n, dtype=np.float64)
        llb = np.zeros(n, dtype=np.float64)
        counts = np.zeros((n, 5 + t.k + 16), dtype=np.float64)
        status = np.zeros(n, dtype=np.int32)
        rc = lib.dnab_fwdback_counts_batch(self._h, n, _ptr(packed), _ptr(byte_off), _ptr(read_len), int(max_sweeps),
                                           _ptr(ll), _ptr(llb), _ptr(counts), _ptr(status))
        if rc:
            raise _err(rc)
        return dict(loglike=ll, loglike_back=llb, counts=counts, status=status)

    def posterior_classes(self):
        buf = C.create_string_buffer(64)
        n = lib.dnab_posterior_classes(self._h, buf, 64)
        if n < 0:
            raise _err(n)
        return buf.value.decode("latin1")

    def posterior(self, reads, max_sweeps=0):
        """Soft decoding (dnab_posterior_batch): per read an [L, n_classes] array of the posterior of the class of the move
        that emitted each base, the per-base most probable class as a string, the forward log-likelihood."""
        classes = self.posterior_classes()
        packed, byte_off, read_len = pack_reads(reads)
        n = len(read_len)
        off = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(read_len, out=off[1:])
        post = np.zeros((int(off[-1]), len(classes)), dtype=np.float64)
        dec = np.zeros(max(int(off[-1]), 1), dtype=np.uint8)
        ll = np.zeros(n, dtype=np.float64)
        status = np.zeros(n, dtype=np.int32)
        rc = lib.dnab_posterior_batch(self._h, n, _ptr(packed), _ptr(byte_off), _ptr(read_len), int(max_sweeps), _ptr(off),
                                      _ptr(ll), _ptr(post), _ptr(dec), _ptr(status))
        if rc:
            raise _err(rc)
        return dict(classes=classes, loglike=ll, status=status,
                    post=[post[off[r]:off[r + 1]] for r in range(n)],
                    decoded=[bytes(dec[off[r]:off[r + 1]]).decode("latin1") for r in range(n)])

    def viterbi_device(self, n_reads, max_read_len, d_packed, d_byte_off, d_read_len, d_loglike, d_decoded, decoded_stride,
                       d_decoded_len, d_status, stream=0):
        """All arguments are raw device pointers (ints), e.g. torch tensors' .data_ptr()."""
        rc = lib.dnab_viterbi_batch_device(self._h, n_reads, max_read_len, d_packed, d_byte_off, d_read_len, d_loglike,
                                           d_decoded, decoded_stride, d_decoded_len, d_status, stream)
        if rc:
            raise _err(rc)

    def decode_fasta(self, path):
        """decodeFastSeqs: [(name, decoded string, loglike, status)] in input order."""
        s = lib.dnab_decode_fasta(self._h, os.fspath(path).encode())
        if not s:
            raise _err()
        try:
            return [(lib.dnab_decoded_name(s, i).decode(), lib.dnab_decoded_seq(s, i).decode("latin1"),
                     lib.dnab_decoded_loglike(s, i), lib.dnab_decoded_status(s, i))
                    for i in range(lib.dnab_decoded_count(s))]
        finally:
            lib.dnab_decoded_free(s)

    def __del__(self):
        if getattr(self, "_h", None):
            lib.dnab_decoder_destroy(self._h)
            self._h = None


def _decoded_set(s):
    if not s:
        raise _err()
    try:
        return [(lib.dnab_decoded_name(s, i).decode(), lib.dnab_decoded_seq(s, i).decode("latin1"),
                 lib.dnab_decoded_loglike(s, i), lib.dnab_decoded_status(s, i))
                for i in range(lib.dnab_decoded_count(s))]
    finally:
        lib.dnab_decoded_free(s)


class MultiDecoder:
    """One decoder per listed device (a device may be listed twice), one host thread each; batches are cut into chunks
    handed out dynamically, results come back in input order (include/dnastore_b200.h dnab_multi_decoder)."""

    def __init__(self, compiled, devices):
        self._compiled = compiled
        devs = np.asarray(list(devices), dtype=np.int32)
        h = lib.dnab_multi_decoder_create(compiled.tables, _ptr(devs), len(devs))
        if not h:
            raise _err(-2)
        self._h = h
        self.devices = [int(x) for x in devs]

    def set_option(self, key, value):
        """"chunk_reads", "decoded_slot_bytes", or any decoder option (applied to every device)."""
        rc = lib.dnab_multi_decoder_set_option(self._h, key.encode(), int(value))
        if rc:
            raise _err(rc)

    def stats(self):
        s = PipelineStats()
        lib.dnab_multi_decoder_last_stats(self._h, C.byref(s))
        return {n: getattr(s, n) for n, _ in PipelineStats._fields_}

    def viterbi(self, reads, decoded_stride=None):
        packed, byte_off, read_len = pack_reads(reads)
        return self.viterbi_packed(packed, byte_off, read_len, decoded_stride)

    def viterbi_packed(self, packed, byte_off, read_len, decoded_stride=None, out=None):
        n = len(read_len)
        max_len = int(read_len.max()) if n else 0
        stride = int(decoded_stride or (8 * max_len + 1024))
        if out is None:
            out = dict(loglike=np.zeros(n, dtype=np.float64), raw=np.zeros((n, stride), dtype=np.uint8),
                       decoded_len=np.zeros(n, dtype=np.int32), status=np.zeros(n, dtype=np.int32))
        rc = lib.dnab_viterbi_batch_multi(self._h, n, _ptr(packed), _ptr(byte_off), _ptr(read_len), _ptr(out["loglike"]),
                                          _ptr(out["raw"]), stride, _ptr(out["decoded_len"]), _ptr(out["status"]))
        if rc:
            raise _err(rc)
        out["decoded"] = [bytes(out["raw"][i, :out["decoded_len"][i]]).decode("latin1") for i in range(n)]
        return out

    def decode_fasta(self, path):
        return _decoded_set(lib.dnab_decode_fasta_multi(self._h, os.fspath(path).encode()))

    def __del__(self):
        if getattr(self, "_h", None):
            lib.dnab_multi_decoder_destroy(self._h)
            self._h = None
