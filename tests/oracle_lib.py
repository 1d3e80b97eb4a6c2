"""ctypes loader for the CPU oracle (oracle/liboracle.so) — test infrastructure only."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")


class OrcStats(C.Structure):
    _fields_ = [("n_kmers", C.c_uint64),
                ("unitigs_before", C.c_uint64), ("links_before", C.c_uint64), ("length_before", C.c_uint64),
                ("unitigs_after", C.c_uint64), ("links_after", C.c_uint64), ("length_after", C.c_uint64),
                ("input_bases", C.c_uint64),
                ("t_load", C.c_double), ("t_kmer_graph", C.c_double), ("t_unitig_graph", C.c_double),
                ("t_simplify", C.c_double), ("t_gfa", C.c_double)]


class OracleError(RuntimeError):
    pass


_lib = None
_path = None
build_flags = "g++ -O3 -march=x86-64-v2 (oracle/Makefile, portable build)"


def build():
    subprocess.run(["make", "-s", "-C", ORACLE_DIR], check=True)


def use_native():
    """bench.py's CPU arm: build the oracle for THIS machine (-O3 -march=native) in a temporary directory, removed at exit, and use
    that library; the tree may be read-only.  Must be called before the first oracle call of the process.  Returns the compiler flags
    in use."""
    global _path, build_flags
    assert _lib is None, "use_native() must precede the first oracle call"
    out = tempfile.mkdtemp(prefix="autocycler_oracle_native_")
    atexit.register(shutil.rmtree, out, True)
    try:
        subprocess.run(["make", "-s", "-C", ORACLE_DIR, "native", f"NATIVE_DIR={out}"], check=True, capture_output=True, timeout=600)
        _path = os.path.join(out, "liboracle.so")
        build_flags = open(os.path.join(out, "flags.txt")).read().strip()
    except Exception as e:      # no compiler on this machine: the shipped portable build is used, and the line says so
        build_flags += f" [native build failed: {type(e).__name__}]"
    return build_flags


def lib():
    global _lib
    if _lib is None:
        path = _path or os.path.join(ORACLE_DIR, "liboracle.so")
        if not os.path.exists(path):
            build()
        _lib = C.CDLL(path)
        _lib.orc_last_error.restype = C.c_char_p
        _lib.orc_free.argtypes = [C.c_void_p]
        for name in ("orc_kmers_sorted", "orc_neighbour_kmers", "orc_find_best_match", "orc_load_sequences",
                     "orc_compress_dir", "orc_compress_seqs", "orc_gfa_roundtrip", "orc_gfa_unitig_seqs",
                     "orc_gfa_exclusive", "orc_gfa_common_seq", "orc_unitig_shift", "orc_unitig_from_kmers",
                     "orc_position_display", "orc_reverse_complement", "orc_gfa_merge_linear_paths",
                     "orc_gfa_merge_fixed_sets", "orc_pairwise_distances"):
            getattr(_lib, name).restype = C.c_void_p
    return _lib


def _take(ptr):
    if not ptr:
        raise OracleError(lib().orc_last_error().decode())
    s = C.string_at(ptr).decode()
    lib().orc_free(ptr)
    return s


def kmers_sorted(seq, k):
    return _take(lib().orc_kmers_sorted(seq.encode(), k)).splitlines()


def neighbour_kmers(seq, k, kmer, nxt):
    return _take(lib().orc_neighbour_kmers(seq.encode(), k, kmer.encode(), 1 if nxt else 0)).splitlines()


def find_best_match(matches):
    return _take(lib().orc_find_best_match("\n".join(matches).encode()))


def load_sequences(directory, k, max_contigs=25, threads=4):
    """-> (assembly_count, [(id, filename, header, length, padded_forward_seq)])"""
    lines = _take(lib().orc_load_sequences(directory.encode(), k, max_contigs, threads)).split("\n")
    count = int(lines[0].split("\t")[1])
    seqs = []
    for ln in lines[1:]:
        if not ln:
            continue
        i, fn, hd, length, fwd = ln.split("\t")
        seqs.append((int(i), fn, hd, int(length), fwd))
    return count, seqs


def compress_dir(directory, k, max_contigs=25, threads=4):
    """-> (gfa_text, yaml_text, OrcStats)"""
    st = OrcStats()
    y = C.c_void_p()
    g = lib().orc_compress_dir(directory.encode(), k, max_contigs, threads, C.byref(y), C.byref(st))
    gfa = _take(g)
    return gfa, _take(y.value), st


def compress_seqs(seqs, assembly_count, k, want_seed_dump=False):
    """seqs: [(id, filename, header, length, padded_forward_seq)] -> (gfa_text, OrcStats, seed_dump or None)"""
    n = len(seqs)
    arr = lambda xs: (C.c_char_p * n)(*[x.encode() for x in xs])
    fwd = arr([s[4] for s in seqs])
    fns = arr([s[1] for s in seqs])
    hds = arr([s[2] for s in seqs])
    ids = (C.c_uint16 * n)(*[s[0] for s in seqs])
    st = OrcStats()
    seed = C.c_void_p()
    g = lib().orc_compress_seqs(n, fwd, ids, fns, hds, assembly_count, k, C.byref(st),
                                C.byref(seed) if want_seed_dump else None)
    gfa = _take(g)
    return gfa, st, (_take(seed.value) if want_seed_dump else None)


def gfa_roundtrip(gfa_text):
    return _take(lib().orc_gfa_roundtrip(gfa_text.encode()))


def decompress(gfa_text, out_dir):
    if lib().orc_decompress(gfa_text.encode(), out_dir.encode()) != 0:
        raise OracleError(lib().orc_last_error().decode())


def pairwise_distances(gfa_text):   # cluster.rs:132-176 -> text of the distance matrix file
    return _take(lib().orc_pairwise_distances(gfa_text.encode()))


def gfa_merge_linear_paths(gfa_text, use_paths=True, renumber=False):
    return _take(lib().orc_gfa_merge_linear_paths(gfa_text.encode(), int(use_paths), int(renumber)))


def gfa_merge_fixed_sets(gfa_text):
    out = _take(lib().orc_gfa_merge_fixed_sets(gfa_text.encode())).split("\n")
    return [int(x) for x in out[0].split()], [int(x) for x in out[1].split()]


def gfa_unitig_seqs(gfa_text, simplify=False, use_paths=False):
    out = _take(lib().orc_gfa_unitig_seqs(gfa_text.encode(), int(simplify), int(use_paths)))
    return [tuple(ln.split("\t")) for ln in out.splitlines()]


def gfa_exclusive(gfa_text):
    out = _take(lib().orc_gfa_exclusive(gfa_text.encode()))
    return {int(a): (b, c) for a, b, c in (ln.split("\t") for ln in out.splitlines())}


def gfa_common_seq(gfa_text, spec, end):
    return _take(lib().orc_gfa_common_seq(gfa_text.encode(), spec.encode(), int(end)))


def unitig_shift(segment_line, op, amount=0, seq=""):
    return _take(lib().orc_unitig_shift(segment_line.encode(), op, amount, seq.encode())).split("\t")


def unitig_from_kmers(seq, k, first_fwd_start):
    return _take(lib().orc_unitig_from_kmers(seq.encode(), k, first_fwd_start)).split("\t")


def position_display(seq_id, strand, pos):
    return _take(lib().orc_position_display(seq_id, int(strand), pos))


def reverse_complement(s):
    return _take(lib().orc_reverse_complement(s.encode()))
