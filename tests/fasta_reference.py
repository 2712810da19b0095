"""numpy FASTA formatter written from the definitions in include/pansim_b200.h, working on the one-hot rows of
download_core(): whole mode (every site a column) and SNP mode (the sites where two or more letters are present),
the constant-site counts by letter, and the closed form of a record's byte offset."""
import numpy as np

CODES = np.array([1, 2, 4, 8], np.uint8)
LETTERS = np.frombuffer(b"ACGT", np.uint8)


def fasta_columns(core, snps_only):
    """(column sites, const_counts[4]) of one-hot rows core [N, L]."""
    N, L = core.shape
    if not snps_only:
        return np.arange(L), np.zeros(4, np.int64)
    codes = np.searchsorted(CODES, core)
    present = np.stack([(codes == a).any(axis=0) for a in range(4)], axis=1)      # [L, 4]
    poly = present.sum(axis=1) >= 2
    const = present[~poly].sum(axis=0).astype(np.int64)                          # the one letter of each constant site
    return np.flatnonzero(poly), const


def fasta_letters(core, cols):
    """uint8 [N, len(cols)]: the ASCII letters of the columns."""
    return LETTERS[np.searchsorted(CODES, core[:, cols])]


def fasta_text(core, snps_only):
    """(file bytes, columns, const_counts) of one-hot rows core [N, L]."""
    cols, const = fasta_columns(core, snps_only)
    let = fasta_letters(core, cols)
    text = b"".join(b">ind_%d\n" % i + let[i].tobytes() + b"\n" for i in range(core.shape[0]))
    return text, len(cols), const


def record_offset(i, cols):
    """Byte offset of record i: i (7 + cols) plus the digits of every j < i."""
    o = i * (7 + cols) + i
    p = 10
    while p <= i:
        o += i - p
        p *= 10
    return o
