"""Synthetic FASTA builders shared by the tests (seeded, small, covering the edge cases that decide
bit-exactness: SURVEY.md section 4 / 7.3)."""
import numpy as np

ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


def random_bases(rng, n):
    return ACGT[rng.integers(0, 4, n)]


def to_fasta(records, width=60, newline=b"\n", final_newline=True):
    """records: list of (header bytes without '>', uint8 array of sequence characters)."""
    out = []
    for name, seq in records:
        out.append(b">" + name + newline)
        seq = np.asarray(seq, dtype=np.uint8).tobytes()
        for i in range(0, len(seq), width):
            out.append(seq[i:i + width] + newline)
    txt = b"".join(out)
    if not final_newline and txt.endswith(newline):
        txt = txt[:-len(newline)]
    return txt


def mutate(rng, seq, sub=0.01, indel=0.001):
    """Substitutions plus short indels (the config-2 mutation model, SURVEY.md 8d)."""
    s = np.array(seq, dtype=np.uint8, copy=True)
    hit = rng.random(s.size) < sub
    s[hit] = ACGT[rng.integers(0, 4, int(hit.sum()))]
    if indel > 0:
        pieces, pos = [], 0
        for at in np.flatnonzero(rng.random(s.size) < indel):
            if at < pos:
                continue
            pieces.append(s[pos:at])
            ln = int(rng.integers(1, 11))
            if rng.random() < 0.5:
                pieces.append(random_bases(rng, ln))   # insertion
                pos = at
            else:
                pos = min(s.size, at + ln)             # deletion
        pieces.append(s[pos:])
        s = np.concatenate(pieces)
    return s


def adversarial_fasta(rng, n=6000):
    """Multi-record FASTA with N runs, IUPAC codes, lower case, records shorter than k, blank
    lines, a '>' inside a sequence line, poly-T >= 32 and odd line widths."""
    recs = []
    a = random_bases(rng, n)
    a[100:140] = ord("N")
    a[500] = ord("R")
    a[900:905] = np.frombuffer(b"nnnnn", dtype=np.uint8)
    low = rng.random(n) < 0.5
    a = np.where(low, a | 0x20, a)
    recs.append((b"chr1 some description > with marker", a))
    recs.append((b"tiny", random_bases(rng, 7)))
    recs.append((b"empty", np.zeros(0, dtype=np.uint8)))
    b = random_bases(rng, 3000)
    b[1000:1040] = ord("T")          # poly-T of 40
    b[2000:2033] = ord("A")          # poly-A of 33
    b[2500] = ord(">")               # marker in the middle of a line: a plain invalid character
    recs.append((b"chr2", b))
    recs.append((b"chr3", random_bases(rng, 1)))
    txt = to_fasta(recs, width=61)
    return txt.replace(b">tiny", b"\n\n>tiny")  # blank lines between records


def kseq_fasta(rng, n=6000, fastq=False):
    """Text that exercises kseq's record rules (SURVEY.md A.1): '@' header lines between '>' ones,
    '@' / '+' / '>' in the middle of sequence lines, junk before the first marker; with fastq=True
    also FASTQ records -- single- and multi-line, quality lines that begin with '@' and '>'."""
    a = random_bases(rng, n)
    width = 67
    a[width * 3 + 5] = ord("@")          # columns 5, 7, 9: never the first byte of a line
    a[width * 7 + 7] = ord("+")
    b = a[n // 2:]
    b[width * 2 + 9] = ord(">")
    recs = [(b"r0 first", a[:n // 2]), (b"r1", b)]
    txt = to_fasta(recs, width=width).replace(b">r1", b"@r1")
    out = b"junk line\nmore junk " + txt
    if fastq:
        s1 = random_bases(rng, 150).tobytes()
        s2 = random_bases(rng, 301).tobytes()
        q2 = bytes(rng.integers(33, 74, 301).astype(np.uint8))
        q2 = b"@" + q2[1:100] + b"\n>" + q2[101:200] + b"\n+" + q2[201:]          # quality lines starting with @ > +
        out += (b"@read1 desc\n" + s1 + b"\n+\n" + b"I" * 150 + b"\n"
                b"@read2\n" + s2[:100] + b"\n" + s2[100:200] + b"\n" + s2[200:] + b"\n+read2\n" + q2 + b"\n"
                b"stray text >late record\n" + random_bases(rng, 200).tobytes() + b"\n")
    return out


def decode_packed(codes, invalid, nsym):
    """Packed stream (include/dandd_b200.h layout) -> oracle symbol stream (0..3, 4 = break)."""
    codes = np.asarray(codes, dtype=np.uint32)
    invalid = np.asarray(invalid, dtype=np.uint32)
    s = np.arange(nsym, dtype=np.int64)
    c = (codes[s >> 4] >> (30 - 2 * (s & 15)).astype(np.uint32)) & 3
    b = (invalid[s >> 5] >> (31 - (s & 31)).astype(np.uint32)) & 1
    return np.where(b == 1, 4, c).astype(np.uint8)


def kmask_of(ks):
    m = 0
    for k in ks:
        m |= 1 << (k - 1)
    return m


def reference_path(*parts):
    """A path inside the checkout of the reference project (github.com/jessicabonnie/dandd) that the
    DANDD_REFERENCE environment variable names, or None without one: the tests that run the reference
    beside the drop-in skip then, and the fixtures under tests/golden/ hold what it produced."""
    import os
    root = os.environ.get("DANDD_REFERENCE")
    return os.path.join(root, *parts) if root else None


def make_dataset(directory, n_genomes, length, seed, sub=0.03, indel=0.002, prefix="g"):
    """n mutated copies of one random ancestor, written as <prefix><i>.fasta (multi-record, odd line
    width).  Deterministic: the golden generator and the tests call this with the same arguments."""
    import os
    os.makedirs(directory, exist_ok=True)
    rng = np.random.default_rng(seed)
    anc = random_bases(rng, length)
    paths = []
    for g in range(n_genomes):
        r = np.random.default_rng(seed * 100 + g)
        seq = mutate(r, anc, sub=sub, indel=indel)
        cut = int(seq.size * (0.4 + 0.05 * g))
        seq[cut // 2:cut // 2 + 3] = ord("N")
        recs = [(b"%s%d_a len=%d" % (prefix.encode(), g, cut), seq[:cut]), (b"%s%d_b" % (prefix.encode(), g), seq[cut:])]
        path = os.path.join(directory, f"{prefix}{g}.fasta")
        with open(path, "wb") as fh:
            fh.write(to_fasta(recs, width=70))
        paths.append(path)
    return paths
