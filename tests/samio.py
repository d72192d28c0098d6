"""SAM text for the tests of the GPU SAM decoder (test infrastructure only): a writer whose arguments mirror
``oracle.bamio.write_bam``, and a Python restatement of the line rules of the product's decoder (csrc/k_sam.cuh,
csrc/sam_gpu.cu; SAM spec v1 section 1.4), which the host-compiled rules are checked against."""
import numpy as np

from oracle.bamio import CIGAR_OPS, CONSUMES_QRY, NT16


def write_sam(path, references, lengths, tid, pos, flag, mapq, cig_off, cig, l_seq=None, isize=None,
              names=None, seqs=None, text=None, with_index=True, aux=None, quals=None, mtid=None, mpos=None,
              crlf=False, final_newline=True):
    """Write the records ``write_bam`` writes for the same arguments as SAM text: names ``r<i>`` and all-'A' SEQ of the
    CIGAR's query length by default, QUAL '*' (the BAM writer's 0xff), RNEXT/PNEXT '*'/0 unless ``mtid``/``mpos`` are
    given.  ``aux``: per record the optional-field text (without the leading TAB); ``quals``: per record the QUAL
    string; ``crlf``: CRLF line ends; ``final_newline``: whether the last line ends in a newline.  ``with_index`` is
    accepted for symmetry with ``write_bam``; SAM has no index."""
    n = len(tid)
    if text is None:
        text = "@HD\tVN:1.4\tSO:coordinate\n" + "".join(
            "@SQ\tSN:%s\tLN:%d\n" % (r, l) for r, l in zip(references, lengths))
    nl = "\r\n" if crlf else "\n"
    lines = [l for l in text.split("\n") if l]
    ops_txt = np.array(list(CIGAR_OPS) + ["?"] * 7)
    out = []
    for i in range(n):
        ops = np.asarray(cig[int(cig_off[i]):int(cig_off[i + 1])], dtype=np.uint32)
        ls = int(l_seq[i]) if l_seq is not None else int(((ops >> 4).astype(np.int64) * CONSUMES_QRY[ops & 15]).sum())
        if seqs is None:
            seq = "A" * ls
        elif isinstance(seqs[i], str):                    # (letters as they are: lowercase, any byte)
            seq = seqs[i]
        else:
            seq = "".join(NT16[int(c)] for c in seqs[i])
        t = int(tid[i])
        rname = references[t] if t >= 0 else "*"
        if mtid is None or int(mtid[i]) < 0:
            rnext = "*"
        else:
            rnext = "=" if int(mtid[i]) == t else references[int(mtid[i])]
        pnext = int(mpos[i]) + 1 if mpos is not None else 0
        cigar = "".join("%d%s" % (c >> 4, ops_txt[c & 15]) for c in ops.tolist()) or "*"
        qual = quals[i] if quals is not None else "*"
        fields = [names[i] if names is not None else "r%d" % i, str(int(flag[i])), rname, str(int(pos[i]) + 1),
                  str(int(mapq[i])), cigar, rnext, str(pnext), str(int(isize[i]) if isize is not None else 0), seq or "*",
                  qual if (qual and seq) else "*"]
        if aux is not None and aux[i]:
            fields.append(aux[i].decode() if isinstance(aux[i], bytes) else aux[i])
        out.append("\t".join(fields))
    body = nl.join(lines + out)
    if final_newline and body:
        body += nl
    with open(path, "w", newline="") as fh:
        fh.write(body)
    return path


class SamError(ValueError):
    """A line that breaks a rule: ``line`` (1-based) and ``field`` (0-10 = QNAME..QUAL, 11 = fewer than 11 fields or an
    empty line, 12 = a header line after a record; None for a header error)."""

    def __init__(self, line, field, msg=""):
        self.line, self.field = line, field
        super().__init__("line %s: field %s %s" % (line, field, msg))


_NT16_OF = {c: i for i, c in enumerate(NT16)}
_NT16_OF.update({c.lower(): i for i, c in enumerate(NT16)})


def _udec(b, hi):
    if not b or not b.isdigit():
        return None
    v = int(b)
    return v if v <= hi else None


def parse_sam(data):
    """The SAM rules of the product's decoder over a whole file image -> (references, lengths, columns dict with
    tid/pos/flag/mapq/l_seq/isize/cig_off/cig, names (bytes), seqs (nt16 arrays)); raises SamError."""
    lines = data.split(b"\n")
    if lines and lines[-1] == b"":
        lines.pop()
    refs, lens = [], []
    k = 0
    while k < len(lines) and lines[k][:1] == b"@":
        ln = lines[k][:-1] if lines[k].endswith(b"\r") else lines[k]
        if ln.startswith(b"@SQ\t"):
            tags = {}
            for t in ln.split(b"\t")[1:]:
                if t[:3] in (b"SN:", b"LN:"):
                    tags[t[:2]] = t[3:]
            ln_v = _udec(tags.get(b"LN", b""), 2 ** 31 - 1)
            if not tags.get(b"SN") or not ln_v:
                raise SamError(k + 1, None, "@SQ")
            refs.append(tags[b"SN"].decode())
            lens.append(ln_v)
        k += 1
    if len(set(refs)) != len(refs):
        raise SamError(None, None, "duplicate @SQ")
    tid_of = {r: i for i, r in enumerate(refs)}
    cols = {c: [] for c in ("tid", "pos", "flag", "mapq", "l_seq", "isize")}
    cig, cig_off, names, seqs = [], [0], [], []
    for j in range(k, len(lines)):
        line_no = j + 1
        ln = lines[j][:-1] if lines[j].endswith(b"\r") else lines[j]
        if not ln:
            raise SamError(line_no, 11)
        if ln[:1] == b"@":
            raise SamError(line_no, 12)
        f = ln.split(b"\t")
        if len(f) < 11:
            raise SamError(line_no, 11)
        f = f[:11]
        qname, fl, rname, ps, mq, cg, rnext, pnext, tlen, seq, qual = f
        if not 1 <= len(qname) <= 254:
            raise SamError(line_no, 0)
        fl_v = _udec(fl, 65535)
        if fl_v is None:
            raise SamError(line_no, 1)
        if rname == b"*":
            t = -1
        elif rname.decode("latin-1") in tid_of:
            t = tid_of[rname.decode("latin-1")]
        else:
            raise SamError(line_no, 2)
        ps_v = _udec(ps, 2 ** 31 - 1)
        if ps_v is None:
            raise SamError(line_no, 3)
        mq_v = _udec(mq, 255)
        if mq_v is None:
            raise SamError(line_no, 4)
        ops = []
        if not cg:
            raise SamError(line_no, 5)
        if cg != b"*":
            num = b""
            for c in cg:
                ch = chr(c)
                if ch.isdigit() and c < 128:
                    num += bytes([c])
                elif ch in CIGAR_OPS:
                    if not num or int(num) > (1 << 28) - 1:
                        raise SamError(line_no, 5)
                    ops.append((int(num) << 4) | CIGAR_OPS.index(ch))
                    num = b""
                else:
                    raise SamError(line_no, 5)
            if num:
                raise SamError(line_no, 5)
        if not rnext:
            raise SamError(line_no, 6)
        if _udec(pnext, 2 ** 31 - 1) is None:
            raise SamError(line_no, 7)
        neg = tlen[:1] == b"-"
        tl = _udec(tlen[1:] if neg else tlen, 2 ** 31 if neg else 2 ** 31 - 1)
        if tl is None:
            raise SamError(line_no, 8)
        if not seq:
            raise SamError(line_no, 9)
        ls = 0 if seq == b"*" else len(seq)
        if not qual or (qual != b"*" and len(qual) != ls):
            raise SamError(line_no, 10)
        cols["tid"].append(t); cols["pos"].append(ps_v - 1); cols["flag"].append(fl_v); cols["mapq"].append(mq_v)
        cols["l_seq"].append(ls); cols["isize"].append(-tl if neg else tl)
        cig += ops
        cig_off.append(len(cig))
        names.append(bytes(qname))
        seqs.append(np.array([_NT16_OF.get(chr(c), 15) for c in (b"" if seq == b"*" else seq)], dtype=np.uint8))
    out = dict(tid=np.array(cols["tid"], np.int32), pos=np.array(cols["pos"], np.int32), flag=np.array(cols["flag"], np.uint16),
               mapq=np.array(cols["mapq"], np.uint8), l_seq=np.array(cols["l_seq"], np.int32),
               isize=np.array(cols["isize"], np.int64).astype(np.int32), cig_off=np.array(cig_off, np.uint32),
               cig=np.array(cig, np.uint32))
    return refs, lens, out, names, seqs
