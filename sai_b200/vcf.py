"""Host-side VCF ingest for the scoring path (GT only).

Stays on the host by design (the north star keeps VCF parsing off the GPU).
Produces what ``read_data(... is_phased=False, filter_*=False,
filter_missing=False)`` hands to the reference's ``WindowGenerator``
(sai/generators/window_generator.py:102-118): per population the positions and
the per-individual allele sums.  Follows

* ``parse_ind_file``        sai/utils/utils.py:31-75
* ``read_geno_data``        sai/utils/utils.py:78-186  (scikit-allel ``read_vcf``
  with ``numbers={"GT": ploidy}``, ``alt_number=1``, ``region``: GT is cut or
  padded with -1 to ``ploidy`` alleles, ``.`` = -1)
* ``read_anc_allele``       sai/utils/utils.py:435-489
* ``check_anc_allele`` / ``flip_snps``   sai/utils/utils.py:492-555
  (sites without ancestral allele or with one that is neither REF nor ALT are
  dropped; where ALT is ancestral every allele a becomes ``abs(a - 1)``, so a
  missing allele -1 becomes 2)
* ``reshape_genotypes(is_phased=False)``  sai/utils/utils.py:405-410
  (sum over the ploidy axis)

scikit-allel itself is a third-party dependency of the reference
(scikit-allel==1.3.7, pyproject.toml) and is not available here; this reader
covers plain-text and gzip/bgzip VCF.
"""

from __future__ import annotations

import gzip
import os
import warnings
from typing import Optional

import numpy as np

from .encode import PopData


def parse_ind_file(filename: str) -> dict[str, list[str]]:
    """``category sample`` lines -> ``{category: [samples]}``; lines that do
    not have exactly two fields are skipped."""
    try:
        samples: dict[str, list[str]] = {}
        with open(filename, "r") as f:
            for line in f:
                parts = line.strip().split()
                if len(parts) != 2:
                    continue
                samples.setdefault(parts[0], []).append(parts[1])
        if not samples:
            raise ValueError(f"No samples found in {filename}. Please check your data.")
    except FileNotFoundError:
        raise FileNotFoundError(f"File '{filename}' not found. Please check the file path.")
    return samples


def _open_text(path: str):
    with open(path, "rb") as f:
        magic = f.read(2)
    if magic == b"\x1f\x8b":
        return gzip.open(path, "rt")
    return open(path, "r")


def _parse_gt(field: str, ploidy: int, out: np.ndarray) -> None:
    gt = field.split(":", 1)[0]
    n = 0
    tok = ""
    for ch in gt:
        if ch == "|" or ch == "/":
            if n < ploidy:
                out[n] = -1 if tok in (".", "") else int(tok)
            n += 1
            tok = ""
        else:
            tok += ch
    if n < ploidy:
        out[n] = -1 if tok in (".", "") else int(tok)
    n += 1
    for k in range(n, ploidy):
        out[k] = -1


class VcfRegion:
    """All records of one chromosome region, parsed once; populations are then
    cut out by sample name with their own ploidy (the reference re-reads the
    file once per population, sai/utils/utils.py:716-734)."""

    def __init__(self, vcf_file: str, chr_name: str, start: Optional[int] = None, end: Optional[int] = None):
        self.samples: list[str] = []
        pos, ref, alt, rows = [], [], [], []
        try:
            with _open_text(vcf_file) as f:
                for line in f:
                    if line.startswith("##"):
                        continue
                    if line.startswith("#CHROM"):
                        self.samples = line.rstrip("\n").split("\t")[9:]
                        continue
                    tab = line.find("\t")
                    if line[:tab] != chr_name:
                        continue
                    cols = line.rstrip("\n").split("\t")
                    p = int(cols[1])
                    if start is not None and end is not None and not (start <= p <= end):
                        continue
                    pos.append(p)
                    ref.append(cols[3])
                    alt.append(cols[4].split(",")[0])
                    fmt = cols[8].split(":")
                    gi = fmt.index("GT") if "GT" in fmt else 0
                    rows.append([c.split(":")[gi] if gi else c for c in cols[9:]])
        except FileNotFoundError:
            raise
        except Exception as e:  # same wrapping as utils.py:136-137
            region = chr_name if start is None and end is None else f"{chr_name}:{start}-{end}"
            raise ValueError(f"Failed to read VCF file {vcf_file} from {region}: {e}") from e
        self.pos = np.asarray(pos, dtype=np.int32)
        self.ref = ref
        self.alt = alt
        self.rows = rows

    def genotypes(self, sample_names: list[str], ploidy: int) -> np.ndarray:
        """int8 ``(sites, individuals, ploidy)`` like ``calldata/GT``."""
        idx = [self.samples.index(s) for s in sample_names]
        gt = np.full((len(self.rows), len(idx), ploidy), -1, dtype=np.int8)
        for r, row in enumerate(self.rows):
            for c, i in enumerate(idx):
                _parse_gt(row[i], ploidy, gt[r, c])
        return gt


class AncAlleles:
    """Ancestral alleles of one chromosome as arrays: ``pos`` (int64, sorted, unique) and ``allele``
    (``str`` objects); ``.as_dict()`` gives the reference's ``{pos: allele}`` view."""

    def __init__(self, pos: np.ndarray, allele: np.ndarray):
        self.pos, self.allele = pos, allele

    def __len__(self) -> int:
        return int(self.pos.shape[0])

    def as_dict(self) -> dict[int, str]:
        return dict(zip(self.pos.tolist(), self.allele.tolist()))


def read_anc_arrays(anc_allele_file: str, chr_name: str, start=None, end=None) -> AncAlleles:
    """BED ``chrom start end allele`` of one chromosome (and region), vectorised: pandas' C reader
    instead of a Python line loop (6 M lines of a chromosome-scale table take a second, not ten).
    A position listed twice keeps its last allele, like the reference's dict (utils.py:435-489)."""
    import pandas as pd

    try:
        df = pd.read_csv(anc_allele_file, sep=r"\s+", header=None, usecols=[0, 2, 3], names=["chrom", "pos", "allele"],
                         dtype={"chrom": str, "pos": np.int64, "allele": str}, engine="c", comment=None,
                         keep_default_na=False)
    except FileNotFoundError as exc:
        raise FileNotFoundError(f"File {anc_allele_file} not found.") from exc
    except pd.errors.EmptyDataError:
        df = pd.DataFrame({"chrom": [], "pos": np.array([], dtype=np.int64), "allele": []})
    keep = df["chrom"].to_numpy() == chr_name
    pos = df["pos"].to_numpy()
    if start is not None:
        keep &= pos >= start
    if end is not None:
        keep &= pos <= end
    pos, allele = pos[keep], df["allele"].to_numpy()[keep]
    if pos.size == 0:
        if start is not None or end is not None:
            raise ValueError(
                f"No ancestral allele is found for chromosome {chr_name} in the region {start}-{end}."
            )
        raise ValueError(f"No ancestral allele is found for chromosome {chr_name}.")
    # last occurrence wins, then sorted by position
    _, first_of_reversed = np.unique(pos[::-1], return_index=True)
    idx = pos.size - 1 - first_of_reversed
    return AncAlleles(pos[idx], allele[idx])


def read_anc_allele(anc_allele_file: str, chr_name: str, start=None, end=None) -> dict[int, str]:
    """BED ``chrom start end allele`` -> ``{end: allele}`` for one chromosome."""
    return read_anc_arrays(anc_allele_file, chr_name, start, end).as_dict()


def _polarise(pos: np.ndarray, ref: list[str], alt: list[str], gt: np.ndarray, anc: dict[int, str]):
    """Keeps sites whose ancestral allele is REF or ALT; flips those where it is
    ALT (``abs(a - 1)`` on every allele, missing included)."""
    keep = np.zeros(pos.shape[0], dtype=bool)
    flip = np.zeros(pos.shape[0], dtype=bool)
    for i, p in enumerate(pos.tolist()):
        a = anc.get(p)
        if a is None or a not in (ref[i], alt[i]):
            continue
        keep[i] = True
        flip[i] = a == alt[i]  # utils.py:523-524
    gt = gt[keep].copy()
    f = flip[keep]
    gt[f] = np.abs(gt[f].astype(np.int16) - 1).astype(np.int8)
    return pos[keep], gt


def load_population_group(
    region: VcfRegion,
    sample_file: Optional[str],
    group: str,
    ploidy_config,
    anc: Optional[dict[int, str]],
):
    """``(data, samples)`` of one group like ``_load_population_data``
    (sai/utils/utils.py:649-761) with ``is_phased=False`` and no filtering."""
    if sample_file is None:
        return None, None
    samples = parse_ind_file(sample_file)
    if group not in ploidy_config.root:
        raise ValueError(f"Ploidy configuration missing group '{group}'.")
    ploidies = ploidy_config.root[group]
    for population in ploidies:
        if population not in samples:
            raise ValueError(
                f"Population '{population}' in ploidy_config[{group}] not found in sample file: {sample_file}"
            )
    data: dict[str, PopData] = {}
    for population, names in samples.items():
        if population not in ploidies:
            warnings.warn(
                f"Population '{population}' found in sample file but not in ploidy_config[{group}]; skipping.",
                RuntimeWarning,
            )
            continue
        if region.pos.size == 0:
            continue
        try:
            gt = region.genotypes(names, ploidies[population])
        except Exception as e:
            raise ValueError(f"Failed to read VCF data for {sample_file}, population '{population}': {e}")
        pos = region.pos
        if anc is not None:
            pos, gt = _polarise(pos, region.ref, region.alt, gt, anc)
        data[population] = PopData(pos.copy(), gt.sum(axis=2, dtype=np.int64).astype(np.int8))
    if not data:
        return None, samples
    return data, samples


def _scan_text(vcf_file, on_header, on_lines, n_threads=0, chunk_bytes=64 << 20, batch_bytes=256 << 20, on_size_hint=None,
               on_bgzf=None):
    """Feeds the text of a VCF (plain, bgzip or gzip) to ``on_lines(addr, length) -> bytes consumed``
    in large buffers of whole-or-partial lines (an incomplete last line is carried to the next
    buffer), after calling ``on_header(line)`` once with the ``#CHROM`` line.  Plain text is
    mapped read-only and handed over in place; bgzip blocks are inflated in parallel by the
    native library; plain gzip streams through Python's reader.  ``on_size_hint(total_text_bytes)``
    is called first when the total is known without reading the text (plain: the file size;
    bgzip: the sum of the blocks' ISIZE fields), so that the consumer can size its output once.
    ``on_bgzf(base_addr, block_off, out_off, n_blocks, skip)``, when given, receives a bgzip file
    as its block index instead of text (``skip`` = text offset of the first record): the fused
    inflate + parse of ``sai_bgzf_parse_gt``."""
    import ctypes as C

    from . import _cabi

    lib = _cabi.load()
    consumed = C.c_int64(0)
    seen_header = False
    if os.path.getsize(vcf_file) == 0:
        return
    if not _is_gzip(vcf_file):
        import mmap

        with open(vcf_file, "rb") as f, mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ) as mm:
            h = mm.find(b"#CHROM")
            he = mm.find(b"\n", h) if h >= 0 else -1
            if h >= 0 and he >= 0:
                on_header(mm[h:he])
                if on_size_hint is not None:
                    on_size_hint(len(mm) - he)
                view = np.frombuffer(mm, dtype=np.uint8)
                try:
                    body, length = he + 1, len(mm)
                    done = on_lines(view.ctypes.data + body, length - body) if length > body else 0
                    tail = bytes(mm[body + done :])
                finally:
                    del view
                if tail:  # last line without a newline
                    tail += b"\n"
                    buf = np.frombuffer(tail, dtype=np.uint8)
                    on_lines(buf.ctypes.data, len(tail))
    elif _is_bgzf(vcf_file):
        import mmap

        with open(vcf_file, "rb") as f, mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ) as mm:
            view = np.frombuffer(mm, dtype=np.uint8)
            try:
                base, total = view.ctypes.data, len(mm)
                max_blocks = 1 << 14
                block_off = np.empty(max_blocks, dtype=np.int64)
                out_off = np.empty(max_blocks + 1, dtype=np.int64)
                if on_bgzf is not None:
                    # index every block (18 header bytes each), find the #CHROM line in the first few, hand the rest over
                    offs, outs, p, text_total = [], [], 0, 0
                    while p < total:
                        n = int(lib.sai_bgzf_scan(base + p, total - p, max_blocks, 1 << 62, block_off.ctypes.data,
                                                  out_off.ctypes.data, C.byref(consumed)))
                        if n < 0:
                            _cabi.check(n)
                        if n == 0 or consumed.value == 0:
                            break
                        offs.append(block_off[:n] + p)
                        outs.append(out_off[1 : n + 1] + text_total)
                        text_total += int(out_off[n])
                        p += consumed.value
                    if not offs:
                        return
                    all_boff = np.ascontiguousarray(np.concatenate(offs))
                    all_ooff = np.ascontiguousarray(np.concatenate([np.zeros(1, dtype=np.int64)] + outs))
                    n_all, k, h, he = int(all_boff.shape[0]), 16, -1, -1
                    while True:
                        k = min(k, n_all)
                        head_buf = np.empty(int(all_ooff[k]) + 1, dtype=np.uint8)
                        _cabi.check(lib.sai_bgzf_inflate(base, all_boff.ctypes.data, all_ooff.ctypes.data, k, head_buf.ctypes.data, n_threads))
                        head = head_buf[: int(all_ooff[k])].tobytes()
                        h = head.find(b"#CHROM")
                        he = head.find(b"\n", h) if h >= 0 else -1
                        if (h >= 0 and he >= 0) or k == n_all:
                            break
                        k *= 8
                    if h < 0 or he < 0:
                        return
                    on_header(head[h:he])
                    if on_size_hint is not None:
                        on_size_hint(text_total - he)
                    on_bgzf(base, all_boff, all_ooff, n_all, he + 1)
                    return
                at, carry = 0, b""
                if on_size_hint is not None:  # the block headers alone give the size of the text
                    text_total, p = 0, 0
                    while p < total:
                        n = int(lib.sai_bgzf_scan(base + p, total - p, max_blocks, 1 << 62, block_off.ctypes.data,
                                                  out_off.ctypes.data, C.byref(consumed)))
                        if n <= 0 or consumed.value == 0:
                            break
                        text_total += int(out_off[n])
                        p += consumed.value
                    on_size_hint(text_total)
                buf = np.empty(0, dtype=np.uint8)  # reused from batch to batch: its pages are faulted in once
                while True:
                    n = int(lib.sai_bgzf_scan(base + at, total - at, max_blocks, batch_bytes, block_off.ctypes.data,
                                              out_off.ctypes.data, C.byref(consumed))) if at < total else 0
                    if n < 0:
                        _cabi.check(n)
                    last = n == 0 or at + consumed.value >= total
                    text_len = int(out_off[n]) if n else 0
                    if buf.size < len(carry) + text_len + 1:
                        buf = np.empty(max(len(carry) + text_len + 1, min(batch_bytes, total * 64) + (1 << 20)), dtype=np.uint8)
                    buf[: len(carry)] = np.frombuffer(carry, dtype=np.uint8)
                    if n:
                        _cabi.check(lib.sai_bgzf_inflate(base + at, block_off.ctypes.data, out_off.ctypes.data, n,
                                                         buf.ctypes.data + len(carry), n_threads))
                        at += consumed.value
                    length = len(carry) + text_len
                    start_at = 0
                    if not seen_header:
                        probe = 1 << 20  # the header is at the top of the file: do not copy a whole batch to find it
                        while True:
                            head = buf[: min(length, probe)].tobytes()
                            h = head.find(b"#CHROM")
                            he = head.find(b"\n", h) if h >= 0 else -1
                            if (h >= 0 and he >= 0) or probe >= length:
                                break
                            probe *= 16
                        if h < 0 or he < 0:
                            if last:
                                break
                            carry = buf[:length].tobytes()
                            continue
                        on_header(head[h:he])
                        seen_header = True
                        start_at = he + 1
                    if last and length > start_at and buf[length - 1] != 10:
                        buf[length] = 10  # last line without a newline
                        length += 1
                    done = start_at + (on_lines(buf.ctypes.data + start_at, length - start_at) if length > start_at else 0)
                    carry = buf[done:length].tobytes()
                    if last:
                        break
            finally:
                del view
    else:
        # a plain gzip file of moderate size: the whole text in one native call (sai_gzip_inflate: the
        # bgzip block decoder on a single-member file, ~8x Python's gzip reader); several members, very
        # large files or anything unexpected take the streaming reader below
        import mmap
        import struct

        size = os.path.getsize(vcf_file)
        if 18 <= size <= (1 << 30):
            with open(vcf_file, "rb") as f, mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ) as mm:
                isize = struct.unpack("<I", mm[size - 4 : size])[0]
                text = None
                if isize <= (3 << 30) and isize >= size // 2:  # (a wrapped ISIZE of a > 4 GB text would be implausibly small)
                    view = np.frombuffer(mm, dtype=np.uint8)
                    try:
                        text = np.empty(isize + 1, dtype=np.uint8)
                        if int(lib.sai_gzip_inflate(view.ctypes.data, size, text.ctypes.data, isize)) != isize:
                            text = None
                    except MemoryError:
                        text = None
                    finally:
                        del view
            if text is not None:
                head = text[: min(isize, 1 << 20)].tobytes()
                h = head.find(b"#CHROM")
                he = head.find(b"\n", h) if h >= 0 else -1
                if h < 0 or he < 0:  # an unusually long header: look through everything
                    head = text[:isize].tobytes()
                    h = head.find(b"#CHROM")
                    he = head.find(b"\n", h) if h >= 0 else -1
                if h < 0 or he < 0:
                    return
                on_header(head[h:he])
                if on_size_hint is not None:
                    on_size_hint(isize - he)
                length = isize
                if length > he + 1 and text[length - 1] != 10:
                    text[length] = 10  # last line without a newline
                    length += 1
                if length > he + 1:
                    on_lines(text.ctypes.data + he + 1, length - he - 1)
                return
        with gzip.open(vcf_file, "rb") as f:
            carry = b""
            while True:
                block = f.read(chunk_bytes)
                data = carry + block
                if not data:
                    break
                if not seen_header:
                    h = data.find(b"#CHROM")
                    he = data.find(b"\n", h) if h >= 0 else -1
                    if h < 0 or he < 0:
                        if not block:
                            break
                        carry = data
                        continue
                    on_header(data[h:he])
                    seen_header = True
                    data = data[he + 1 :]
                if not block and not data.endswith(b"\n"):
                    data += b"\n"  # last line without a newline
                buf = np.frombuffer(data, dtype=np.uint8)
                at = on_lines(buf.ctypes.data, len(data)) if len(data) else 0
                carry = data[at:]
                if not block:
                    break


def _span_from_ends(vcf_file: str, chr_name: str, tail_bytes: int = 1 << 20):
    """``(first POS, last POS, -1)`` when the first and the last record of a plain-text or bgzip
    file are both on ``chr_name`` (the usual one-file-per-chromosome layout; records of a
    chromosome are contiguous in a sorted VCF), else ``None``."""
    import ctypes as C
    import mmap

    from . import _cabi

    if os.path.getsize(vcf_file) == 0 or (_is_gzip(vcf_file) and not _is_bgzf(vcf_file)):
        return None

    def record_of(line: bytes):
        parts = line.rstrip(b"\r").split(b"\t", 2)
        if len(parts) < 3 or not parts[1].isdigit():
            return None
        return parts[0].decode(), int(parts[1])

    def first_record(text: bytes):
        at = 0
        while at < len(text):
            nl = text.find(b"\n", at)
            if nl < 0:
                return None  # incomplete line: not enough text
            if nl > at and text[at : at + 1] != b"#":
                return record_of(text[at:nl])
            at = nl + 1
        return None

    def last_record(text: bytes, complete_start: bool):
        body = text[:-1] if text.endswith(b"\n") else text
        nl = body.rfind(b"\n")
        if nl < 0 and not complete_start:
            return None
        line = body[nl + 1 :]
        return None if (not line or line.startswith(b"#")) else record_of(line)

    with open(vcf_file, "rb") as f, mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ) as mm:
        total = len(mm)
        if not _is_gzip(vcf_file):
            head = None
            for limit in (1 << 20, 64 << 20):
                head = first_record(mm[: min(total, limit)])
                if head is not None:
                    break
            tail = last_record(mm[max(0, total - tail_bytes) :], total <= tail_bytes)
        else:
            lib = _cabi.load()
            view = np.frombuffer(mm, dtype=np.uint8)
            try:
                base = view.ctypes.data
                nb = 1 << 12
                block_off, out_off = np.empty(nb, np.int64), np.empty(nb + 1, np.int64)
                used = C.c_int64(0)

                def inflate(at: int, length: int, limit: int):
                    n = int(lib.sai_bgzf_scan(base + at, length, nb, limit, block_off.ctypes.data, out_off.ctypes.data,
                                              C.byref(used)))
                    if n <= 0:
                        return None
                    buf = np.empty(int(out_off[n]), dtype=np.uint8)
                    if lib.sai_bgzf_inflate(base + at, block_off.ctypes.data, out_off.ctypes.data, n,
                                            buf.ctypes.data if buf.size else None, 0) != 0:
                        return None
                    return buf.tobytes()

                head = None
                for limit in (1 << 20, 64 << 20):  # the header usually fits the first megabyte of text
                    text = inflate(0, total, limit)
                    head = first_record(text) if text is not None else None
                    if head is not None:
                        break
                tail = None
                # the last blocks: look for a block boundary in the last ~256 KB of the file
                start = max(0, total - (256 << 10))
                magic = b"\x1f\x8b\x08\x04"
                while tail is None and start < total:
                    start = mm.find(magic, start)
                    if start < 0:
                        break
                    text = inflate(start, total - start, 1 << 40)
                    if text is not None and used.value == total - start:  # a true block chain up to the end of the file
                        tail = last_record(text, start == 0)
                        break
                    start += 1
            finally:
                del view
    if head is None or tail is None or head[0] != chr_name or tail[0] != chr_name:
        return None
    return head[1], tail[1], -1


def _scan_sorted_region(vcf_file, chr_name, start, end, on_header, on_lines, n_threads=0, batch_bytes=256 << 20,
                        on_bgzf=None):
    """Region read without an index, for the usual one-chromosome, position-sorted file (plain text or
    bgzip): bisection over line starts / bgzip blocks finds the byte range that holds every record with
    ``start <= POS <= end`` (plus a little slack; the parser still filters by POS), and only that range is
    inflated and parsed -- a chunk of a sharded run costs its share of the file, not the whole file.
    Returns False (nothing done) when the file does not qualify; the caller then scans everything.
    ``on_bgzf(base_addr, block_off, out_off, n_blocks, skip, at_eof)``, when given, receives a bgzip
    region as its blocks instead of text: ``block_off`` / ``out_off`` index the blocks found by the
    bisection (``out_off[0] = 0``), the records start at text offset ``skip``, and ``at_eof`` says the
    blocks end the file (else the last incomplete line is dropped, as the text path drops it)."""
    import ctypes as C
    import mmap

    from . import _cabi

    if _span_from_ends(vcf_file, chr_name) is None:  # not a single-chromosome file of a supported container
        return False
    lib = _cabi.load()

    def pos_of_line(text: bytes, at: int):
        t1 = text.find(b"\t", at)
        t2 = text.find(b"\t", t1 + 1) if t1 >= 0 else -1
        if t2 < 0 or not text[t1 + 1 : t2].isdigit():
            return None
        return int(text[t1 + 1 : t2])

    with open(vcf_file, "rb") as f, mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ) as mm:
        total = len(mm)
        if not _is_gzip(vcf_file):
            h = mm.find(b"#CHROM")
            he = mm.find(b"\n", h) if h >= 0 else -1
            if h < 0 or he < 0:
                return False
            body = he + 1

            class _Unparsable(Exception):
                pass

            def line_at(off: int):  # first line starting at or after `off`; POS None only past the last line
                ls = body if off <= body else (lambda nl: total if nl < 0 else nl + 1)(mm.find(b"\n", off - 1))
                if ls >= total:
                    return total, None
                # CHROM <TAB> POS <TAB>: probe to the second TAB (contig names can be long), not a fixed width
                t1 = mm.find(b"\t", ls)
                t2 = mm.find(b"\t", t1 + 1) if t1 >= 0 else -1
                if t2 < 0 or t2 - t1 > 12 or not mm[t1 + 1 : t2].isdigit():
                    raise _Unparsable  # not a data line we understand: let the full scan deal with the file
                return ls, int(mm[t1 + 1 : t2])

            def first_line(pred):  # start of the first line whose POS satisfies the monotone `pred`
                lo, hi = body, total
                while lo < hi:
                    mid = (lo + hi) // 2
                    ls, p = line_at(mid)
                    if p is None or pred(p):
                        hi = mid
                    else:
                        lo = ls + 1
                return line_at(lo)[0]

            try:
                lo, hi = first_line(lambda p: p >= start), first_line(lambda p: p > end)
            except _Unparsable:
                return False
            on_header(mm[h:he])
            if hi > lo:
                view = np.frombuffer(mm, dtype=np.uint8)
                try:
                    done = on_lines(view.ctypes.data + lo, hi - lo)
                    tail = bytes(mm[lo + done : hi])
                finally:
                    del view
                if tail:  # the file's last line without a newline
                    tail += b"\n"
                    buf = np.frombuffer(tail, dtype=np.uint8)
                    on_lines(buf.ctypes.data, len(tail))
            return True

        # bgzip: table of block offsets (headers only), then bisection on the first full line of a block
        view = np.frombuffer(mm, dtype=np.uint8)
        try:
            base = view.ctypes.data
            used = C.c_int64(0)
            offs, at = [], 0
            cap = 1 << 16
            b_off, o_off = np.empty(cap, np.int64), np.empty(cap + 1, np.int64)
            while at < total:
                n = int(lib.sai_bgzf_scan(base + at, total - at, cap, 1 << 62, b_off.ctypes.data, o_off.ctypes.data, C.byref(used)))
                if n <= 0:
                    break
                offs.append(b_off[:n] + at)
                at += used.value
            if at != total or not offs:
                return False
            boff = np.concatenate(offs + [np.array([total], dtype=np.int64)])
            n_blocks = boff.shape[0] - 1
            def inflate(b0: int, b1: int) -> bytes:
                n = int(lib.sai_bgzf_scan(base + int(boff[b0]), int(boff[b1] - boff[b0]), b1 - b0, 1 << 62,
                                          b_off.ctypes.data, o_off.ctypes.data, C.byref(used)))
                if n != b1 - b0:
                    raise ValueError("bgzip block table changed under the reader")
                buf = np.empty(max(1, int(o_off[n])), dtype=np.uint8)
                _cabi.check(lib.sai_bgzf_inflate(base + int(boff[b0]), b_off.ctypes.data, o_off.ctypes.data, n,
                                                 buf.ctypes.data, n_threads))
                return buf[: int(o_off[n])].tobytes()

            # the header: blocks from the start until the #CHROM line is complete
            hb, head = 0, b""
            while hb < n_blocks:
                head += inflate(hb, hb + 1)
                hb += 1
                h = head.find(b"#CHROM")
                he = head.find(b"\n", h) if h >= 0 else -1
                if he >= 0:
                    break
            else:
                return False
            first_data_block = hb - 1  # the block in which the records start

            def first_pos(b: int):  # POS of the first line that starts inside block b (None: no such line)
                if b <= first_data_block:
                    return -1
                text = inflate(b, b + 1)
                nl = text.find(b"\n")
                return None if nl < 0 else pos_of_line(text, nl + 1)

            def first_block(pred):  # first block > first_data_block whose first line satisfies the monotone pred
                lo, hi = first_data_block + 1, n_blocks
                while lo < hi:
                    mid = (lo + hi) // 2
                    p, probe = None, mid
                    while p is None and probe < hi:  # blocks without a line start: look further right
                        p = first_pos(probe)
                        probe += 1
                    if p is None or pred(p):
                        hi = mid
                    else:
                        lo = probe
                return lo

            b_lo = max(first_data_block, first_block(lambda p: p >= start) - 1)  # last block whose first line is < start
            # through the block whose first line is > end (it still holds the tail of the last wanted record);
            # blocks without a line start in between (or up to the end of the file) belong to the region
            probe, p_hi = first_block(lambda p: p > end), None
            while p_hi is None and probe < n_blocks:
                p_hi = first_pos(probe)
                probe += 1
            b_hi = n_blocks if p_hi is None else probe
            on_header(head[h:he])
            if on_bgzf is not None:
                blocks, texts = np.empty(b_hi - b_lo, np.int64), np.zeros(b_hi - b_lo + 1, np.int64)
                n = int(lib.sai_bgzf_scan(base + int(boff[b_lo]), int(boff[b_hi] - boff[b_lo]), b_hi - b_lo, 1 << 62,
                                          blocks.ctypes.data, texts.ctypes.data, C.byref(used))) if b_hi > b_lo else 0
                if n != b_hi - b_lo:
                    raise ValueError("bgzip block table changed under the reader")
                blocks += int(boff[b_lo])
                if b_lo == first_data_block:  # the records follow the header inside block b_lo
                    skip = max(0, he + 1 - (len(head) - int(texts[1] - texts[0])))
                else:  # behind the first newline from block b_lo on (a record that started before it)
                    skip = int(texts[n]) if n else 0
                    for b in range(b_lo, b_hi):
                        nl = inflate(b, b + 1).find(b"\n")
                        if nl >= 0:
                            skip = int(texts[b - b_lo]) + nl + 1
                            break
                on_bgzf(base, blocks, texts, n, skip, b_hi == n_blocks)
                return True
            # the records of the first data block follow the header inside `head`
            from_head = b_lo == first_data_block
            pending = head[he + 1 :] if from_head else b""
            b = hb if from_head else b_lo
            carry, first = b"", True
            per_batch = max(1, batch_bytes >> 16)  # a block inflates to at most 64 KB
            while True:
                e = max(b, min(b_hi, b + per_batch))
                # inflate the batch straight behind the carried bytes (no intermediate copies)
                n, text_len = 0, 0
                if e > b:
                    n = int(lib.sai_bgzf_scan(base + int(boff[b]), int(boff[e] - boff[b]), e - b, 1 << 62,
                                              b_off.ctypes.data, o_off.ctypes.data, C.byref(used)))
                    if n != e - b:
                        raise ValueError("bgzip block table changed under the reader")
                    text_len = int(o_off[n])
                prefix = len(carry) + (len(pending) if first else 0)
                buf = np.empty(prefix + text_len + 1, dtype=np.uint8)
                buf[: len(carry)] = np.frombuffer(carry, dtype=np.uint8)
                if first and pending:
                    buf[len(carry) : prefix] = np.frombuffer(pending, dtype=np.uint8)
                if n:
                    _cabi.check(lib.sai_bgzf_inflate(base + int(boff[b]), b_off.ctypes.data, o_off.ctypes.data, n,
                                                     buf.ctypes.data + prefix, n_threads))
                start_at, length = 0, prefix + text_len
                if first and not from_head:  # the tail of a record that started in the block before: POS < start
                    probe = buf[prefix : prefix + min(text_len, 4 << 20)].tobytes()
                    nl = probe.find(b"\n")
                    start_at = prefix + nl + 1 if nl >= 0 else length
                first = False
                b = e
                last = b >= b_hi
                if last and b_hi == n_blocks and length > start_at and buf[length - 1] != 10:
                    buf[length] = 10  # the file's last line without a newline
                    length += 1
                done = start_at + (on_lines(buf.ctypes.data + start_at, length - start_at) if length > start_at else 0)
                carry = buf[done:length].tobytes()
                if last:
                    break
            return True
        finally:
            del view


def chromosome_span(vcf_file: str, chr_name: str, n_threads: int = 0):
    """``(first POS, last POS, number of records)`` of ``chr_name`` in file order, or ``None`` when
    the chromosome does not occur -- what ``ChunkGenerator.__init__`` finds with pysam
    (sai/generators/chunk_generator.py:64-76).  A per-chromosome file (first and last record on
    ``chr_name``) is answered from its two ends without reading the middle (record count -1 =
    not counted); anything else takes one parallel native scan of the text."""
    import ctypes as C

    from . import _cabi

    lib = _cabi.load()
    quick = _span_from_ends(vcf_file, chr_name)
    if quick is not None:
        return quick
    first, last, n = None, None, 0
    f1, l1, n1, used = C.c_int64(0), C.c_int64(0), C.c_int64(0), C.c_int64(0)

    def on_lines(addr: int, length: int) -> int:
        nonlocal first, last, n
        _cabi.check(lib.sai_vcf_chrom_span(addr, length, chr_name.encode(), C.byref(f1), C.byref(l1), C.byref(n1),
                                           C.byref(used), n_threads))
        if n1.value:
            if first is None:
                first = int(f1.value)
            last = int(l1.value)
            n += int(n1.value)
        return int(used.value)

    _scan_text(vcf_file, lambda line: None, on_lines, n_threads)
    return None if first is None else (first, last, n)


def anc_table(anc):
    """The native parsers' form of an ancestral-allele table (``AncAlleles`` or ``{pos: allele}``):
    ``(pos int32, alleles as 8-byte NUL-padded records, n)``, or ``None`` when an allele is longer
    than 7 bytes (the native parsers' limit)."""
    if isinstance(anc, dict):
        keys = sorted(anc)
        anc = AncAlleles(np.asarray(keys, dtype=np.int64), np.asarray([anc[k] for k in keys], dtype=object))
    table = np.char.encode(anc.allele.astype(str), "utf-8")  # fixed-width bytes, NUL padded
    if table.dtype.itemsize > 7:
        return None
    return np.ascontiguousarray(anc.pos, dtype=np.int32), np.ascontiguousarray(table.astype("S8")).tobytes(), len(anc)


def _native_read(vcf_file, chr_name, start, end, requests, anc, n_threads=0, chunk_bytes=64 << 20,
                 batch_bytes=256 << 20, fused_bgzf=True, group_blocks=0):
    """One pass of the native parser (``sai_vcf_parse_gt``) over the file.
    ``requests`` = list of (sample_name, ploidy); returns ``(pos, gt)`` with one
    int8 column per request, or ``None`` for the sample names line missing."""
    import ctypes as C

    from . import _cabi

    lib = _cabi.load()
    anc_pos = anc_buf = None
    n_anc = 0
    if anc is not None:
        table = anc_table(anc)
        if table is None:
            return None  # long alleles: use the Python reader
        anc_pos, anc_buf, n_anc = table
    cols = ploidies = None
    n_out = len(requests)
    consumed = C.c_int64(0)
    region = (start, end) if (start is not None and end is not None) else (1, 0)
    # ONE output matrix for the whole file, sized from the text size when that is known up front
    # (np.empty commits no pages: an over-estimate costs address space only) and doubled otherwise:
    # no per-batch parts to concatenate at the end (a chromosome-sized copy)
    out = {"pos": np.empty(0, dtype=np.int32), "gt": np.empty((0, n_out), dtype=np.int8), "rows": 0}
    row_bytes = max(64, 2 * n_out)  # a record is never shorter: >= 2 characters per requested column

    def reserve(cap: int) -> None:
        if cap <= out["pos"].shape[0]:
            return
        try:
            pos_new, gt_new = np.empty(cap, dtype=np.int32), np.empty((cap, n_out), dtype=np.int8)
        except MemoryError:
            if out["rows"] == 0:
                raise
            cap = out["pos"].shape[0] + max(1024, out["pos"].shape[0] // 2)
            pos_new, gt_new = np.empty(cap, dtype=np.int32), np.empty((cap, n_out), dtype=np.int8)
        n = out["rows"]
        pos_new[:n] = out["pos"][:n]
        gt_new[:n] = out["gt"][:n]
        out["pos"], out["gt"] = pos_new, gt_new

    def on_size_hint(text_bytes: int) -> None:
        try:
            reserve(min(1 << 31, text_bytes // row_bytes + 1024))
        except MemoryError:
            pass  # grow on demand instead
    def header_columns(line: bytes):
        names = line.decode().rstrip("\r").split("\t")[9:]
        index = {n: i for i, n in enumerate(names)}
        return (np.ascontiguousarray([index[s] for s, _ in requests], dtype=np.int32),  # KeyError like list.index
                np.ascontiguousarray([p for _, p in requests], dtype=np.int32))

    def parse_buffer(addr: int, length: int) -> int:
        """Parses complete lines of ``length`` bytes at ``addr``; returns the bytes consumed."""
        at = 0
        while at < length:
            rows = out["rows"]
            want = (length - at) // row_bytes + 16  # upper bound of the records in the rest of this buffer
            if rows + want > out["pos"].shape[0]:
                reserve(max(rows + want, 2 * out["pos"].shape[0]))
            cap = out["pos"].shape[0] - rows
            n = lib.sai_vcf_parse_gt(
                addr + at, length - at, chr_name.encode(), region[0], region[1],
                cols.ctypes.data, ploidies.ctypes.data, n_out,
                anc_pos.ctypes.data if n_anc else None, anc_buf if n_anc else None, n_anc,
                out["pos"].ctypes.data + 4 * rows, out["gt"].ctypes.data + rows * n_out, n_out, cap, C.byref(consumed), n_threads,
            )
            if n < 0:
                _cabi.check(int(n))
            out["rows"] = rows + int(n)
            if consumed.value == 0:
                break
            at += consumed.value
        return at

    def parse_bgzf(base: int, block_off, out_off, n_blocks: int, skip: int) -> None:
        """Whole bgzip file: groups of blocks inflated and parsed by the same thread (no text buffer)."""
        text_bytes = int(out_off[n_blocks]) - skip
        reserve(text_bytes // row_bytes + 1024)
        while True:
            n = lib.sai_bgzf_parse_gt(
                base, block_off.ctypes.data, out_off.ctypes.data, n_blocks, skip, chr_name.encode(), region[0], region[1],
                cols.ctypes.data, ploidies.ctypes.data, n_out,
                anc_pos.ctypes.data if n_anc else None, anc_buf if n_anc else None, n_anc,
                out["pos"].ctypes.data, out["gt"].ctypes.data, n_out, out["pos"].shape[0], group_blocks, n_threads,
            )
            # records shorter than the header promises (truncated lines) can outnumber the estimate: the fused
            # read is not resumable, so repeat it with more room (a record is at least ~20 bytes of fixed columns)
            if n == _cabi.E_CAPACITY and out["pos"].shape[0] < text_bytes // 20 + 1024:
                reserve(min(text_bytes // 20 + 1024, 4 * out["pos"].shape[0]))
                continue
            break
        if n < 0:
            _cabi.check(int(n))
        out["rows"] = int(n)

    def on_header(line: bytes):
        nonlocal cols, ploidies, row_bytes
        cols, ploidies = header_columns(line)
        # a record holds every sample of the file, not just the requested ones: >= 2 characters per sample column
        row_bytes = max(row_bytes, 2 * (line.count(b"\t") - 8) + 18)

    handled = False
    if start is not None and end is not None:
        handled = _scan_sorted_region(vcf_file, chr_name, int(start), int(end), on_header, parse_buffer, n_threads, batch_bytes)
    if not handled:
        _scan_text(vcf_file, on_header, parse_buffer, n_threads, chunk_bytes, batch_bytes, on_size_hint,
                   parse_bgzf if fused_bgzf else None)
    if cols is None:
        return None
    n, cap = out["rows"], out["pos"].shape[0]
    if n == 0:
        return np.empty(0, dtype=np.int32), np.empty((0, n_out), dtype=np.int8)
    # rows beyond n were never touched: keeping the views costs address space only, unless the estimate was far off
    if n * 16 >= cap:
        return out["pos"][:n], out["gt"][:n]
    return out["pos"][:n].copy(), out["gt"][:n].copy()


def _is_bgzf(path: str) -> bool:
    """bgzip container (gzip members with a 'BC' extra subfield, SAM spec 4.1)?"""
    import ctypes as C

    from . import _cabi

    with open(path, "rb") as f:
        head = f.read(1 << 16)
    return bool(_cabi.load().sai_is_bgzf(head, len(head))) if len(head) >= 18 else False


def write_bgzf(path: str, data: bytes, block: int = 0xFF00, level: int = 6) -> None:
    """Writes ``data`` as a bgzip file (tests / tools; no htslib here)."""
    import struct
    import zlib

    with open(path, "wb") as f:
        for at in list(range(0, len(data), block)) + [None]:
            chunk = b"" if at is None else data[at : at + block]
            co = zlib.compressobj(level, zlib.DEFLATED, -15)
            payload = co.compress(chunk) + co.flush()
            bsize = 12 + 6 + len(payload) + 8
            f.write(struct.pack("<BBBBIBBH", 31, 139, 8, 4, 0, 0, 255, 6))
            f.write(b"BC" + struct.pack("<HH", 2, bsize - 1))
            f.write(payload)
            f.write(struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk)))


def _is_gzip(path: str) -> bool:
    with open(path, "rb") as f:
        return f.read(2) == b"\x1f\x8b"


def population_plan(groups, ploidy_config):
    """One output column per (population, sample) with the population's ploidy, for the groups
    ``((group, ind_file), ...)``: ``(plan, requests, out)`` with ``plan = [(group, samples,
    [(population, first request, end request), ...]), ...]``, ``requests = [(sample name, ploidy),
    ...]`` and ``out[group] = (None, None)`` for the groups without a sample file.  Raises and warns
    like ``_load_population_data`` (sai/utils/utils.py:649-761)."""
    plan, requests, out = [], [], {}
    for group, ind_file in groups:
        if ind_file is None or (group == "outgroup" and group not in ploidy_config.root):
            out[group] = (None, None)
            continue
        samples = parse_ind_file(ind_file)
        if group not in ploidy_config.root:
            raise ValueError(f"Ploidy configuration missing group '{group}'.")
        ploidies = ploidy_config.root[group]
        for population in ploidies:
            if population not in samples:
                raise ValueError(
                    f"Population '{population}' in ploidy_config[{group}] not found in sample file: {ind_file}"
                )
        pops = []
        for population, names in samples.items():
            if population not in ploidies:
                warnings.warn(
                    f"Population '{population}' found in sample file but not in ploidy_config[{group}]; skipping.",
                    RuntimeWarning,
                )
                continue
            a = len(requests)
            requests += [(n, ploidies[population]) for n in names]
            pops.append((population, a, len(requests)))
        plan.append((group, samples, pops))
    return plan, requests, out


def read_anc_or_error(anc_allele_file, chr_name, start, end):
    """``(table, error)``: the reference reads the VCF region first and returns None (-> NaN rows)
    when it holds no record, BEFORE it looks at the ancestral-allele table (utils.py:123-141 then
    :152-158), so an empty table is only an error once the region turns out to have records."""
    if not anc_allele_file:
        return None, None
    try:
        return read_anc_arrays(anc_allele_file, chr_name, start, end), None
    except ValueError as e:
        if "No ancestral allele is found" not in str(e):
            raise
        return None, e


def read_data(
    vcf_file: str,
    chr_name: str,
    ploidy_config,
    ref_ind_file: Optional[str],
    tgt_ind_file: Optional[str],
    src_ind_file: Optional[str],
    out_ind_file: Optional[str],
    anc_allele_file: Optional[str],
    start: Optional[int] = None,
    end: Optional[int] = None,
    native: bool = True,
):
    """``{"ref": (data, samples), "tgt": ..., "src": ..., "outgroup": ...}``
    (sai/utils/utils.py:215-356 with the WindowGenerator's fixed flags:
    ``is_phased=False``, no fixed-variant / missing filters).  ``native=True``
    parses the file once for all populations with ``sai_vcf_parse_gt``;
    ``native=False`` is the pure-Python reader kept as a cross-check."""
    # a chunk that falls into a gap (centromere) must not fail because the table is empty there too
    anc, anc_error = read_anc_or_error(anc_allele_file, chr_name, start, end)
    groups = (("ref", ref_ind_file), ("tgt", tgt_ind_file), ("src", src_ind_file), ("outgroup", out_ind_file))
    if not native:
        anc = anc.as_dict() if anc is not None else None
        region = VcfRegion(vcf_file, chr_name, start, end)
        if anc_error is not None and region.pos.size:
            raise anc_error
        out = {}
        for group, ind_file in groups:
            if ind_file is None or (group == "outgroup" and group not in ploidy_config.root):
                out[group] = (None, None)
                continue
            out[group] = load_population_group(region, ind_file, group, ploidy_config, anc)
        return out

    plan, requests, out = population_plan(groups, ploidy_config)
    if not requests:
        return out
    try:
        parsed = _native_read(vcf_file, chr_name, start, end, requests, anc)
    except (KeyError, OSError) as e:
        region = chr_name if start is None and end is None else f"{chr_name}:{start}-{end}"
        raise ValueError(f"Failed to read VCF file {vcf_file} from {region}: {e}") from e
    if parsed is None:
        return read_data(vcf_file, chr_name, ploidy_config, ref_ind_file, tgt_ind_file, src_ind_file, out_ind_file,
                         anc_allele_file, start, end, native=False)
    pos, gt = parsed
    if anc_error is not None and pos.size:  # records but no ancestral allele in the region: the reference raises
        raise anc_error
    for group, samples, pops in plan:
        if pos.size == 0 or not pops:
            out[group] = (None, samples)
            continue
        # column blocks of the one parsed matrix, as views: the packer takes a row stride
        out[group] = ({p: PopData(pos, gt[:, a:b]) for p, a, b in pops}, samples)
    return out
