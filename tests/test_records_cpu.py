"""FASTA records reader (mb200_records_read, host only) and the bucketing of fragments into ragged stores."""
import numpy as np

from motifs_jl_b200 import records


def _write(tmp_path, text, name="r.fa"):
    p = tmp_path / name
    p.write_bytes(text.encode() if isinstance(text, str) else text)
    return str(p)


def _frags(r):
    off = r.frag_offsets
    return [(int(r.frag_record[f]), int(r.frag_start[f]), r.bases[off[f]:off[f + 1]].tobytes().decode()) for f in range(len(r.frag_len))]


def test_records_parsing(tmp_path):
    text = (">chr1 first record\r\nACGTNNac\r\ngtRYa\r\n"          # CRLF, wrapped lines, N run inside, lower case, IUPAC letters
            ">empty\n"                                             # empty record
            ">allN\nNNNN\nnn\n"                                    # all-N record
            ">ends\tx y\nNNACG\nT-AANN\n"                          # N runs at both ends, a gap symbol, a tab in the header
            ">last\nacgt")                                         # no newline at the end of the file
    r = records.read_records(_write(tmp_path, text))
    assert r.names == ["chr1", "empty", "allN", "ends", "last"]
    assert r.lengths.tolist() == [13, 0, 6, 11, 4]
    assert _frags(r) == [(0, 0, "ACGT"), (0, 6, "ACGT"), (0, 12, "A"),
                         (3, 2, "ACGT"), (3, 7, "AA"),
                         (4, 0, "ACGT")]
    assert r.bases.tobytes() == b"ACGTACGTAACGTAAACGT"


def test_records_no_filter_no_cap(tmp_path):
    rng = np.random.default_rng(3)
    seqs = ["".join(rng.choice(list("ACGT"), int(n))) for n in rng.integers(1, 300, 500)]
    text = "".join(f">r{i} description\n" + "\n".join(s[j:j + 60] for j in range(0, len(s), 60)) + "\n" for i, s in enumerate(seqs))
    r = records.read_records(_write(tmp_path, text))
    assert len(r.names) == 500 and r.names[7] == "r7"
    assert r.lengths.tolist() == [len(s) for s in seqs]
    assert [f[2] for f in _frags(r)] == seqs


def test_records_empty_file(tmp_path):
    r = records.read_records(_write(tmp_path, ""))
    assert r.names == [] and len(r.frag_len) == 0 and len(r.bases) == 0


def _check_buckets(L, minlen, buckets, max_padding=1 / 8):
    got = np.concatenate(buckets) if buckets else np.zeros(0, np.int64)
    assert sorted(got.tolist()) == np.nonzero(L >= minlen)[0].tolist()        # every eligible fragment exactly once
    for b in buckets:
        lb = L[b]
        assert lb.min() >= minlen
        assert len(b) * lb.max() - lb.sum() <= max_padding * len(b) * lb.max()


def test_bucketing():
    rng = np.random.default_rng(11)
    peaks = np.exp(rng.uniform(np.log(100), np.log(2000), 20000)).astype(np.int64)
    genome = np.concatenate([rng.integers(1, 50, 300), rng.integers(10_000, 5_000_000, 60), [248_000_000, 1]])
    for L, minlen in ((peaks, 8), (genome, 12), (np.array([5, 5, 5], np.int64), 6), (np.zeros(0, np.int64), 1)):
        b1 = records.bucket_fragments(L, minlen)
        _check_buckets(L, minlen, b1)
        b2 = records.bucket_fragments(L.copy(), minlen)
        assert len(b1) == len(b2) and all(np.array_equal(x, y) for x, y in zip(b1, b2))     # deterministic
    # padding 0: one bucket per distinct length
    L = np.array([7, 3, 7, 9, 3, 3, 1], np.int64)
    b0 = records.bucket_fragments(L, 2, max_padding=0)
    assert [sorted(x.tolist()) for x in b0] == [[3], [0, 2], [1, 4, 5]]
    _check_buckets(L, 2, b0, 0)
