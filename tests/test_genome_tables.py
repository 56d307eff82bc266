"""CPU checks of the tables a genome ingest (``vcf_device.read_genome``) hands to the device: the
chromosome table and the concatenated ancestral-allele table must equal their per-chromosome
equivalents (``anc_table(read_anc_arrays(file, c))``)."""

from __future__ import annotations

import numpy as np
import pytest


def _bed(tmp_path):
    rows = ["1\t9\t10\tA", "10\t19\t20\tC", "1\t4\t5\tG", "chr1\t0\t1\tT", "10\t19\t20\tG", "chr1_alt\t7\t8\tAC",
            "1\t9\t10\tT", "chrUn\t2\t3\tA", "10\t29\t30\tT"]
    p = tmp_path / "anc.bed"
    p.write_text("\n".join(rows) + "\n")
    return str(p)


def test_genome_tables_equal_per_chromosome_tables(tmp_path):
    from sai_b200.vcf import anc_table, read_anc_arrays
    from sai_b200.vcf_device import genome_tables

    bed = _bed(tmp_path)
    names_list = ["10", "1", "chrE", "chr1_alt", "chr1"]
    names, name_off, (anc_pos, anc_all, anc_off) = genome_tables(names_list, bed)
    assert [names[name_off[c] : name_off[c + 1]].decode() for c in range(len(names_list))] == names_list
    assert name_off.dtype == np.int32 and anc_off.dtype == np.int64 and anc_pos.dtype == np.int32
    assert anc_off[0] == 0 and anc_off[-1] == anc_pos.shape[0] == len(anc_all) // 8
    for c, name in enumerate(names_list):
        lo, hi = int(anc_off[c]), int(anc_off[c + 1])
        if name == "chrE":
            assert lo == hi
            with pytest.raises(ValueError, match="No ancestral allele"):
                read_anc_arrays(bed, name)
            continue
        want_pos, want_all, n = anc_table(read_anc_arrays(bed, name, None, None))
        assert hi - lo == n
        assert np.array_equal(anc_pos[lo:hi], want_pos)
        assert anc_all[8 * lo : 8 * hi] == want_all


def test_genome_tables_without_a_file_and_with_long_alleles(tmp_path):
    from sai_b200.vcf_device import genome_tables

    names, name_off, anc = genome_tables(["a", "bb"], None)
    assert names == b"abb" and name_off.tolist() == [0, 1, 3] and anc is None
    p = tmp_path / "long.bed"
    p.write_text("a\t0\t1\tACGTACGTA\n")
    assert genome_tables(["a"], str(p))[2] is None  # longer than 7 bytes: the one-pass read does not take it


def test_chromosome_table_limit_matches_header():
    import os
    import re

    from sai_b200 import _cabi

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    header = open(os.path.join(root, "include", "sai_b200.h")).read()
    assert int(re.search(r"#define SAI_VCF_MAX_CHROMS (\d+)", header).group(1)) == _cabi.MAX_CHROMS
    assert int(re.search(r"SAI_E_ORDER = (-\d+)", header).group(1)) == _cabi.E_ORDER
