"""BCF 2.2 genotypes in numpy: the CPU reference of the BCF input path, and a writer for test data (uncompressed, gzip
or BGZF).

A BCF means exactly the VCF that holds the same records (the text `bcftools view` prints), so everything vcf.py says
about the coding holds.  Its GT field is a typed integer vector per record: per sample `count` values of 1, 2 or 4
bytes, each (allele + 1) << 1 | phased, 0 or 1 for a missing allele, end-of-vector padding a shorter call.  `0/1` is
`02 04`, `0|1` is `02 05`, `./.` is `00 00` and a lone `.` is `00 81`; a record whose every sample is a lone `.` has
count 1 and value `00`.  csrc/bcf.cu decodes the GT vectors on the GPU by the rule of decode_gt
(csrc/bcf_gt.cuh:decode_gt).

GQ and DP (the call filter, --vcf-min-gq / --vcf-min-dp) are count-1 vectors of int8, int16, int32 or float; value_rule
restates csrc/bcf_gt.cuh:bcf_value, and call_values returns the vectors as the driver's loader copies them out.
"""
from __future__ import annotations

import gzip
import struct

import numpy as np

from . import vcf

MAGIC = b"BCF\x02\x02"
INT8, INT16, INT32, FLOAT, CHAR = 1, 2, 3, 5, 7
WIDTH = {INT8: 1, INT16: 2, INT32: 4, FLOAT: 4, CHAR: 1}
TYPE_OF_WIDTH = {1: INT8, 2: INT16, 4: INT32}
EOV = {1: -127, 2: -32767, 4: -2147483647}          # end-of-vector, sign-extended
INT_MISSING = {1: -128, 2: -32768, 4: -2147483648}   # missing value, sign-extended
FLOAT_MISSING, FLOAT_EOV = 0x7F800001, 0x7F800002     # the float sentinels' bits
_DT = {INT8: "<i1", INT16: "<i2", INT32: "<i4", FLOAT: "<f4", CHAR: "u1"}
_QUAL_MISSING = struct.pack("<I", 0x7F800001)
_FORMAT_LINES = {"GT": 'Number=1,Type=String,Description="Genotype"',
                 "AD": 'Number=R,Type=Integer,Description="Allelic depths"',
                 "DP": 'Number=1,Type=Integer,Description="Read depth"',
                 "GQ": 'Number=1,Type=Integer,Description="Genotype quality"',
                 "PL": 'Number=G,Type=Integer,Description="Phred-scaled genotype likelihoods"'}


def decode_gt(v0, v1, count, width):
    """The rule of csrc/bcf_gt.cuh:decode_gt.  v0, v1: one sample's first two values, sign-extended from `width` bytes
    (v1 unused when count == 1) → (a, b) allele index bytes (255 = missing), or None if the call is malformed."""
    M = vcf.MISSING
    if count < 1 or count > 2 or v0 < 0 or (v0 >> 1) - 1 > vcf.MAX_ALLELE:
        return None
    if count == 1 or v1 == EOV[width]:
        return (M, M) if v0 <= 1 else None
    if v1 < 0 or (v1 >> 1) - 1 > vcf.MAX_ALLELE:
        return None
    return ((v0 >> 1) - 1 if v0 > 1 else M, (v1 >> 1) - 1 if v1 > 1 else M)


def value_rule(raw, typ, thr):
    """The rule of csrc/bcf_gt.cuh:bcf_value: raw = an int8/16/32 value sign-extended, or a float's bits (as uint32 or
    int32) → 1 passes (>= thr, or a missing / end-of-vector sentinel), 0 is below thr, -1 is malformed (a float NaN that
    is not a sentinel, or an infinity)."""
    if typ == FLOAT:
        bits = int(raw) & 0xFFFFFFFF
        if bits in (FLOAT_MISSING, FLOAT_EOV):
            return 1
        f = float(np.array([bits], np.uint32).view(np.float32)[0])
        if not np.isfinite(f):
            return -1
        return int(f >= thr)
    w = WIDTH[typ]
    if raw in (INT_MISSING[w], EOV[w]):
        return 1
    return int(raw >= thr)


def value_array(values, typ):
    """float64 values (NaN = missing) → the vector of type typ (missing → the type's missing value)."""
    values = np.asarray(values, float)
    if typ == FLOAT:
        out = values.astype(np.float32).view(np.uint32).copy()
        out[np.isnan(values)] = FLOAT_MISSING
        return out.view("<f4")
    w = WIDTH[typ]
    return np.where(np.isnan(values), INT_MISSING[w], np.nan_to_num(values)).astype(_DT[typ])


def values_float(arr, typ):
    """A GQ / DP vector as read → float64, NaN for the sentinels."""
    if typ == FLOAT:
        bits = np.asarray(arr).view(np.uint32)
        with np.errstate(invalid="ignore"):                  # the sentinels are signalling NaNs
            out = np.asarray(arr, np.float32).astype(float)
        out[(bits == FLOAT_MISSING) | (bits == FLOAT_EOV)] = np.nan
        return out
    a = np.asarray(arr).astype(np.int64)
    w = WIDTH[typ]
    return np.where((a == INT_MISSING[w]) | (a == EOV[w]), np.nan, a.astype(float))


# ------------------------------------------------------------------------------------------------ typed values
def int_type(lo, hi):
    """The narrowest integer type for values in [lo, hi], as htslib picks it (the 8 lowest values of each width are
    reserved for the missing and end-of-vector markers)."""
    if -120 <= lo and hi <= 127:
        return INT8
    if -32760 <= lo and hi <= 32767:
        return INT16
    return INT32


def typed_desc(count, typ):
    """A typed descriptor: count << 4 | type, or 15 << 4 | type and the count as a typed int."""
    if count < 15:
        return bytes([count << 4 | typ])
    return bytes([0xF0 | typ]) + typed_int(count)


def typed_int(v):
    t = int_type(v, v)
    return bytes([0x10 | t]) + np.array([v], _DT[t]).tobytes()


def typed_str(s):
    b = s.encode() if s != "." else b""
    return typed_desc(len(b), CHAR) + b


def typed_ints(values, typ=None):
    """A typed int vector of values (1-d)."""
    values = np.asarray(values, np.int64)
    typ = typ or int_type(int(values.min()), int(values.max()))
    return typed_desc(len(values), typ) + values.astype(_DT[typ]).tobytes()


class _Cursor:
    """Reads typed values from data[i:end]; raises VcfError(what) past the end."""

    def __init__(self, data, i, end, what):
        self.d, self.i, self.end, self.what = data, i, end, what

    def take(self, n):
        if n < 0 or self.i + n > self.end:
            raise vcf.VcfError(self.what)
        self.i += n
        return self.d[self.i - n:self.i]

    def desc(self):
        b = self.take(1)[0]
        typ, count = b & 15, b >> 4
        if count == 15:
            count = self.typed_int()
        return count, typ

    def values(self, count, typ):
        if typ not in _DT:
            raise vcf.VcfError("typed value of unknown type %d" % typ)
        return np.frombuffer(self.take(count * WIDTH[typ]), _DT[typ])

    def typed_int(self):
        count, typ = self.desc()
        if count != 1 or typ not in (INT8, INT16, INT32):
            raise vcf.VcfError(self.what)
        return int(self.values(1, typ)[0])

    def typed_str(self):
        count, typ = self.desc()
        if count and typ != CHAR:
            raise vcf.VcfError(self.what)
        return bytes(self.take(count)).split(b"\0", 1)[0].decode()


# ------------------------------------------------------------------------------------------------ writer
def _header(v, keys, contigs, idx):
    def tail(i):
        return ",IDX=%d>" % i if idx else ">"
    lines = ["##fileformat=VCFv4.2", '##FILTER=<ID=PASS,Description="All filters passed"' + tail(0)]
    lines += ["##FORMAT=<ID=%s,%s%s" % (k, _FORMAT_LINES[k], tail(i + 1)) for i, k in enumerate(keys)]
    lines += ["##contig=<ID=%s%s" % (c, tail(i)) for i, c in enumerate(contigs)]
    lines.append("#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join(v.samples))
    return ("\n".join(lines) + "\n").encode() + b"\0"


def gt_width(idx):
    """Bytes per GT value: 1 while the largest allele index is at most 62, else 2, as htslib picks it."""
    present = np.asarray(idx)[np.asarray(idx) != vcf.MISSING]
    top = int(present.max()) if present.size else 0
    return 1 if top <= 62 else 2 if top <= 16382 else 4


def _gt_field(idx_s, lone_missing, width):
    """(count, values[N, count]) of one record's GT."""
    M = vcf.MISSING
    a, b = idx_s[:, 0].astype(np.int64), idx_s[:, 1].astype(np.int64)
    both = (a == M) & (b == M)
    if lone_missing and both.all():
        return 1, np.zeros((len(a), 1), np.int64)
    va = np.where(a == M, 0, (a + 1) << 1)
    vb = np.where(b == M, 0, (b + 1) << 1)
    if lone_missing:
        vb = np.where(both, EOV[width], vb)
    return 2, np.stack([va, vb], 1)


def bcf_bytes(v: vcf.Vcf, fmt="GT", lone_missing=False, width=None, idx=True, call_type=None) -> bytes:
    """The uncompressed BCF of v: fmt "GT" or "GT:AD:DP:GQ:PL" (the filler values of vcf.vcf_text), lone_missing writes
    a call with both alleles missing as a lone '.', width the GT value width (1, 2 or 4; None: gt_width), idx writes
    IDX= on every dictionary line (else the dictionaries are in order of appearance).  With v.gq / v.dp, fmt may be any
    ':'-list of GT (first), AD, DP, GQ and PL, and DP / GQ hold their values (NaN: missing) as call_type (INT8, INT16,
    INT32 or FLOAT; None: the narrowest integer type)."""
    keys = fmt.split(":")
    custom = v.gq is not None or v.dp is not None
    if fmt not in vcf.FORMATS and not (custom and keys[0] == "GT" and set(keys) <= set(vcf.FORMAT_KEYS)):
        raise ValueError("fmt must be one of %s" % (vcf.FORMATS,))
    contigs = list(dict.fromkeys(v.chrom))
    cidx = {c: i for i, c in enumerate(contigs)}
    idx_arr = np.asarray(v.idx, np.uint8)
    width = width or gt_width(idx_arr)
    if width < gt_width(idx_arr):
        raise ValueError("GT width %d cannot hold the allele indices" % width)
    text = _header(v, keys, contigs, idx)
    out = [MAGIC, struct.pack("<I", len(text)), text]
    N = len(v.samples)
    for s in range(len(v.chrom)):
        n_allele = 1 + len(v.alts[s])
        shared = struct.pack("<iii", cidx[v.chrom[s]], int(v.pos[s]) - 1, len(v.ref[s])) + _QUAL_MISSING
        shared += struct.pack("<II", n_allele, len(keys) << 24 | N)
        shared += typed_str(v.ids[s]) + b"".join(typed_str(a) for a in [v.ref[s]] + list(v.alts[s]))
        shared += typed_ints([0])                                  # FILTER: PASS
        indiv = []
        for k, key in enumerate(keys):
            val = v.gq if key == "GQ" else v.dp if key == "DP" else None
            if key == "GT":
                count, vals = _gt_field(idx_arr[s], lone_missing, width)
                body = typed_desc(count, TYPE_OF_WIDTH[width]) + vals.astype(_DT[TYPE_OF_WIDTH[width]]).tobytes()
            elif val is not None:
                row = np.asarray(val[s], float)
                present = row[~np.isnan(row)]
                t = call_type or (int_type(int(present.min()), int(present.max())) if present.size else INT8)
                body = typed_desc(1, t) + value_array(row, t).tobytes()
            else:
                per = {"AD": [3] * n_allele, "DP": [3 * n_allele], "GQ": [30],
                       "PL": [0] + [20] * (n_allele * (n_allele + 1) // 2 - 1)}[key]
                t = int_type(min(per), max(per))
                body = typed_desc(len(per), t) + np.tile(np.array(per, _DT[t]), N).tobytes()
            indiv.append(typed_int(k + 1) + body)
        indiv = b"".join(indiv)
        out += [struct.pack("<II", len(shared), len(indiv)), shared, indiv]
    return b"".join(out)


def write_bcf(path, v: vcf.Vcf, fmt="GT", lone_missing=False, width=None, compress="bgzf", idx=True, block_size=65280,
              call_type=None):
    """compress: "bgzf" (vcf.bgzf_compress, blocks of block_size input bytes), "gz" (one gzip member) or None."""
    data = bcf_bytes(v, fmt, lone_missing, width, idx, call_type)
    if compress == "bgzf":
        data = vcf.bgzf_compress(data, block_size)
    elif compress == "gz":
        data = gzip.compress(data, compresslevel=1)
    elif compress is not None:
        raise ValueError("compress must be 'bgzf', 'gz' or None")
    with open(path, "wb") as f:
        f.write(data)
    return path


# ------------------------------------------------------------------------------------------------ reader
def _inflate(path):
    with open(path, "rb") as f:
        data = f.read()
    return gzip.decompress(data) if data[:2] == b"\x1f\x8b" else data


def _meta_id(line):
    """(ID, IDX or None) of a structured header line ##KEY=<...> (values may be quoted)."""
    body = line[line.index("<") + 1:line.rindex(">")] if "<" in line and ">" in line else ""
    fields, i = {}, 0
    while i < len(body):
        j = i
        while j < len(body) and body[j] not in "=,":
            j += 1
        key, val = body[i:j], ""
        if j < len(body) and body[j] == "=":
            j += 1
            if j < len(body) and body[j] == '"':
                k = j + 1
                while k < len(body) and body[k] != '"':
                    k += 2 if body[k] == "\\" else 1
                val, j = body[j + 1:k], k + 1
            else:
                k = body.find(",", j)
                k = len(body) if k < 0 else k
                val, j = body[j:k], k
        fields[key] = val
        i = j + 1
    return fields.get("ID", ""), (int(fields["IDX"]) if "IDX" in fields else None)


def _dictionary(entries, first=()):
    """entries: [(ID, IDX or None)] → {index: ID} by IDX= on every line or by order of appearance."""
    with_idx = [e for e in entries if e[1] is not None]
    if with_idx and len(with_idx) != len(entries):
        raise vcf.VcfError("a header dictionary mixes lines with and without IDX=")
    if with_idx:
        d = {i: name for i, name in enumerate(first)}
        d.update({i: name for name, i in entries})
        return d
    names = list(dict.fromkeys(list(first) + [e[0] for e in entries]))
    return dict(enumerate(names))


def _parse(path):
    """→ (samples, records): per record a dict of every field; raises vcf.VcfError with the loader's checks."""
    data = _inflate(path)
    if data[:3] != b"BCF":
        raise vcf.VcfError("not a BCF file")
    if data[:5] != MAGIC:
        raise vcf.VcfError("BCF version %d.%d is not supported" % (data[3], data[4]) if len(data) >= 5 else "truncated header")
    if len(data) < 9:
        raise vcf.VcfError("truncated header")
    l_text = struct.unpack_from("<I", data, 5)[0]
    if 9 + l_text > len(data):
        raise vcf.VcfError("truncated header")
    text = data[9:9 + l_text].split(b"\0", 1)[0].decode()
    strings, contigs, samples = [], [], None
    for line in text.split("\n"):
        if line.startswith(("##FILTER=<", "##INFO=<", "##FORMAT=<")):
            e = _meta_id(line)
            if not (e[0] == "PASS" and e[1] is None):
                strings.append(e)
        elif line.startswith("##contig=<"):
            contigs.append(_meta_id(line))
        elif line.startswith("#CHROM"):
            cols = line.rstrip("\r").split("\t")
            if len(cols) < 9 or cols[8] != "FORMAT":
                raise vcf.VcfError("the #CHROM header has no FORMAT column")
            if len(cols) == 9:
                raise vcf.VcfError("the #CHROM header names no samples")
            samples = cols[9:]
            if len(set(samples)) != len(samples):
                raise vcf.VcfError("duplicate sample ID")
            break
    if samples is None:
        raise vcf.VcfError("no #CHROM header line")
    sdict, cdict = _dictionary(strings, ["PASS"]), _dictionary(contigs)
    N, i, recs = len(samples), 9 + l_text, []
    while i < len(data):
        no = len(recs) + 1
        if i + 8 > len(data):
            raise vcf.VcfError("record %d: truncated record" % no)
        l_shared, l_indiv = struct.unpack_from("<II", data, i)
        i += 8
        if i + l_shared + l_indiv > len(data):
            raise vcf.VcfError("record %d: truncated record" % no)
        if l_shared < 24:
            raise vcf.VcfError("record %d: l_shared is too small for its fields" % no)
        chrom, pos0, rlen = struct.unpack_from("<iii", data, i)
        qual = struct.unpack_from("<f", data, i + 12)[0]
        info_allele, fmt_sample = struct.unpack_from("<II", data, i + 16)
        if chrom not in cdict:
            raise vcf.VcfError("record %d: CHROM index %d is not in the contig dictionary" % (no, chrom))
        where = "record %d (%s:%d)" % (no, cdict[chrom], pos0 + 1)
        sh = _Cursor(data, i + 24, i + l_shared, where + ": l_shared is too small for its fields")
        rec = dict(chrom=cdict[chrom], pos=pos0 + 1, rlen=rlen, qual=qual, id=sh.typed_str() or ".")
        n_allele, n_info = info_allele & 0xFFFF, info_allele >> 16
        alleles = [sh.typed_str() for _ in range(n_allele)]
        rec.update(ref=alleles[0] if alleles else ".", alts=alleles[1:])
        count, typ = sh.desc()
        rec["filter"] = [sdict.get(int(k)) for k in sh.values(count, typ)]
        rec["info"] = {}
        for _ in range(n_info):
            key = sh.typed_int()
            count, typ = sh.desc()
            rec["info"][sdict.get(key)] = sh.values(count, typ)
        n_sample, n_fmt = fmt_sample & 0xFFFFFF, fmt_sample >> 24
        if n_sample != N:
            raise vcf.VcfError(where + ": %d samples, but the #CHROM header names %d samples" % (n_sample, N))
        ind = _Cursor(data, i + l_shared, i + l_shared + l_indiv, where + ": l_indiv is too small for its fields")
        rec["format"] = {}
        for k in range(n_fmt):
            key = ind.typed_int()
            if key not in sdict:
                raise vcf.VcfError(where + ": FORMAT key %d is not in the dictionary of strings" % key)
            count, typ = ind.desc()
            if k == 0:
                if sdict[key] != "GT":
                    raise vcf.VcfError(where + ": FORMAT does not start with GT (%s)" % sdict[key])
                if typ not in (INT8, INT16, INT32):
                    raise vcf.VcfError(where + ": the GT field is of type %d, not int8, int16 or int32" % typ)
                if count == 0:
                    raise vcf.VcfError(where + ": the GT field has a count of 0")
                rec["gt_type"] = min(count, 15) << 4 | typ
                rec["gt_raw"] = bytes(data[ind.i:ind.i + N * count * WIDTH[typ]])
            rec.setdefault("ftype", {}).setdefault(sdict[key], (count, typ, k))
            rec["format"][sdict[key]] = ind.values(N * count, typ).reshape(N, count)
        if n_fmt == 0:
            raise vcf.VcfError(where + ": FORMAT does not start with GT (no FORMAT fields)")
        rec["where"] = where
        recs.append(rec)
        i += l_shared + l_indiv
    return samples, recs


def read_bcf(path) -> vcf.Vcf:
    """Pure-Python reader (uncompressed, gzip or BGZF): every field is parsed; the GTs are decoded by decode_gt and
    checked as the driver checks them (malformed calls, allele indices above the ALT count)."""
    samples, recs = _parse(path)
    N = len(samples)
    idx = np.empty((len(recs), N, 2), np.uint8)
    for s, r in enumerate(recs):
        gt = r["format"]["GT"].astype(np.int64)
        count, width = gt.shape[1], WIDTH[r["gt_type"] & 15]
        for i in range(N):
            g = decode_gt(int(gt[i, 0]), int(gt[i, 1]) if count > 1 else 0, count, width)
            if g is None:
                raise vcf.VcfError(r["where"] + ": malformed GT of sample %s" % samples[i])
            if max((x for x in g if x != vcf.MISSING), default=-1) > len(r["alts"]):
                raise vcf.VcfError(r["where"] + ": allele index above the ALT count")
            idx[s, i] = g
    vals, bad = {}, None
    for j, key in enumerate(("GQ", "DP")):
        if any(key in r["format"] for r in recs):
            vals[key] = np.full((len(recs), N), np.nan)
            bad = np.zeros((len(recs), N, 2), bool) if bad is None else bad
            for s, r in enumerate(recs):
                if key in r["format"]:
                    count, typ, _ = r["ftype"][key]
                    if count != 1 or typ not in (INT8, INT16, INT32, FLOAT):     # refused only where filtered
                        bad[s, :, j] = True
                        continue
                    raw = r["format"][key][:, 0]
                    vals[key][s] = values_float(raw, typ)
                    if typ == FLOAT:                                  # a NaN that is not a sentinel, or an infinity
                        bad[s, :, j] = [value_rule(int(b), FLOAT, 1) < 0 for b in np.ascontiguousarray(raw).view(np.uint32)]
                        vals[key][s][bad[s, :, j]] = np.nan
    return vcf.Vcf(samples=samples, chrom=[r["chrom"] for r in recs], pos=np.array([r["pos"] for r in recs], np.int64),
                   ids=[r["id"] for r in recs], ref=[r["ref"] for r in recs], alts=[r["alts"] for r in recs], idx=idx,
                   gq=vals.get("GQ"), dp=vals.get("DP"), bad=bad)


def call_values(path, keys=("GQ", "DP")):
    """(bytes fv, int64 fv_off[L0+1], int32 fv_pos[L0, 2], uint8 fv_type[L0, 2], int32 fmt_index[L0, 2]): the GQ / DP
    vectors as the driver's loader copies them out (per record the present ones in FORMAT order, each at a multiple of
    4 bytes; -1 / 0 where absent) and their FORMAT indices."""
    _, recs = _parse(path)
    parts, off = [], [0]
    pos = np.full((len(recs), 2), -1, np.int32)
    types = np.zeros((len(recs), 2), np.uint8)
    fidx = np.full((len(recs), 2), -1, np.int32)
    for s, r in enumerate(recs):
        span = b""
        present = sorted((r["ftype"][k][2], j, k) for j, k in enumerate(("GQ", "DP")) if k in r["ftype"] and k in keys)
        for order, j, k in present:
            count, typ, _ = r["ftype"][k]
            pos[s, j], types[s, j], fidx[s, j] = len(span), 1 << 4 | typ, order
            raw = r["format"][k].tobytes()
            span += raw + b"\0" * (-len(raw) % 4)
        parts.append(span)
        off.append(off[-1] + len(span))
    return b"".join(parts), np.array(off, np.int64), pos, types, fidx


def gt_payload(path):
    """(bytes, int64 rec_off[L0+1], uint8 gt_type[L0]): the GT vectors as the driver uploads them, each record's at a
    multiple of 4 bytes (zero padding between), with its descriptor (the count capped at 15)."""
    _, recs = _parse(path)
    parts, off, types = [], [0], []
    for r in recs:
        raw = r["gt_raw"] + b"\0" * (-len(r["gt_raw"]) % 4)
        parts.append(raw)
        off.append(off[-1] + len(raw))
        types.append(r["gt_type"])
    return b"".join(parts), np.array(off, np.int64), np.array(types, np.uint8)
