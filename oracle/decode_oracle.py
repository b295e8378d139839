"""Plain-Python restatement of `guidescan decode` (gsx_decode_database, include/gsx.h): the of:H: lists of a SAM complete database
back into enumerate's CSV rows.  No GPU, no CFD column; one site at a time.  Raises DecodeError where the library returns
GSX_ERR_ARG."""
import bisect


class DecodeError(ValueError):
    pass


COMP = {"A": "T", "T": "A", "C": "G", "G": "C", "a": "t", "t": "a", "c": "g", "g": "c"}


def revcomp(s):
    return "".join(COMP.get(c, c) for c in reversed(s))


def read_fasta(path):
    """(names, lengths, text) as the index builder reads a FASTA: name = first word of the header, text = the upper-cased lines"""
    names, lens, parts = [], [], []
    for line in open(path):
        line = line.rstrip("\n")
        if line.startswith(">"):
            names.append(line[1:].strip().split(" ")[0])
            lens.append(0)
            continue
        if lens:
            lens[-1] += len(line)
        parts.append(line.strip().upper())
    return names, lens, "".join(parts)


def hex_values(of):
    return [int.from_bytes(bytes.fromhex(of[i:i + 16]), "little", signed=True) for i in range(0, len(of), 16)]


def groups(vals, delim):
    """[(distance, [positions])] of one list; DecodeError unless it is [positions] d delim for d = 0, 1, ..."""
    out, cur = [], []
    for v in vals:
        if v != delim:
            cur.append(v)
            continue
        if not cur or cur[-1] != len(out):
            raise DecodeError("malformed of:H: group")
        out.append((len(out), cur[:-1]))
        cur = []
    if cur or not out:
        raise DecodeError("of:H: list does not end with a delimiter")
    return out


def ends(starts, lens):
    return [s + n for s, n in zip(starts, lens)]


def resolve(starts, lens, a, L):
    """resolve_abs (gsx_core.h): (chromosome index, pos1, strand) or None"""
    strand = "+"
    if a < 0:
        a, strand = -a, "-"
    i = bisect.bisect_right(ends(starts, lens), a)          # the first chromosome that ends after a
    if i >= len(lens):
        return None
    off = a - starts[i]
    start, end = (off + 2 - L, off + 1) if strand == "+" else (off + 1, off + L)
    if start < 0 or end > lens[i]:
        return None
    return i, start, strand


def decode(sam_path, fasta_path, pam_length=3, alt_pams=(), complete=True, regions=None):
    """CSV text.  regions: [(chrom, start, end)] (0-based, half-open) or None"""
    names, lens, text = read_fasta(fasta_path)
    G = sum(lens)
    starts = [sum(lens[:i]) for i in range(len(lens))]
    delim = -(G + 1)
    head = "id,sequence,match_chrm,match_position,match_strand,match_distance"
    out = [head + (",match_sequence,rna_bulges,dna_bulges" if complete else "") + ",specificity\n"]
    sq, prev = [], None
    for line in open(sam_path):
        line = line.rstrip("\n").rstrip("\r")
        if not line:
            continue
        if line.startswith("@"):
            if line.startswith("@SQ\t"):
                tags = dict(t.split(":", 1) for t in line.split("\t")[1:])
                sq.append((tags["SN"], int(tags["LN"])))
            continue
        if sq and sq != list(zip(names, lens)):
            raise DecodeError("@SQ lines differ from the FASTA records")
        f = line.split("\t")
        tags = {t[:5]: t[5:] for t in f[11:]}
        if "of:H:" not in tags:
            raise DecodeError("record %s has no of:H: tag (succinct database)" % f[0])
        of, sp = tags["of:H:"], tags["sp:f:"]
        if len(of) < 32 or len(of) % 16:
            raise DecodeError("record %s: truncated of:H:" % f[0])
        if prev is not None and prev[0] == f[0]:
            if prev[1] != of:
                raise DecodeError("record %s: of:H: differs from the previous record of the same QNAME" % f[0])
            continue
        prev = (f[0], of)
        seq = revcomp(f[9]) if int(f[1]) & 16 else f[9]
        L, q = len(seq), len(seq) - pam_length
        if regions is not None:
            a = int(f[3]) - 1
            if not (a >= 0 and any(c == f[2] and s <= a and a + L <= e for c, s, e in regions)):
                continue
        for d, positions in groups(hex_values(of), delim):
            for a in positions:
                r = resolve(starts, lens, a, q + pam_length) if -G <= a < G else None
                if r is None or (a >= 0 and a + 1 < L) or (a < 0 and -a + L > G):
                    raise DecodeError("record %s: off-target %d lies outside the genome" % (f[0], a))
                site = text[a - L + 1:a + 1] if a >= 0 else revcomp(text[-a:-a + L])
                match = "".join(c if i >= q or c == seq[i] else c.lower() for i, c in enumerate(site))
                if sum(1 for i in range(q) if site[i] != seq[i]) != d:
                    raise DecodeError("record %s: off-target %d is not at distance %d" % (f[0], a, d))
                if not any(all(p in ("N", c) for p, c in zip(pam, site[q:])) for pam in [seq[q:]] + list(alt_pams)):
                    raise DecodeError("record %s: off-target %d has another PAM" % (f[0], a))
                chrom, pos1, strand = r
                row = [f[0], seq, names[chrom], str(pos1), strand, str(d)]
                if complete:
                    row += [match, "0", "0"]
                out.append(",".join(row + [sp]) + "\n")
    return "".join(out)
