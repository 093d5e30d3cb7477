"""The VCF dialect of include/v2p_vcf.h pinned on the reference binary: CRLF line ends, extra FORMAT fields before BCSQ
and extra meta lines give the files the plain text gives (and the same matrix in the twin).  Skips where the binary is
absent."""
import pytest

from oracle import refbin
from oracle import vcftext as O
from tests.helpers import load_golden

pytestmark = pytest.mark.skipif(not refbin.available(), reason="oracle/_ref/vcf2prot not built (make -C oracle ref)")


def extra_format(text: str) -> str:
    out = []
    for line in text.split("\n"):
        cols = line.split("\t")
        if line and not line.startswith("#") and len(cols) > 9:
            cols[8] = "GT:AD:BCSQ"
            cols[9:] = [c.split(":")[0] + ":3,1:" + c.split(":")[-1] for c in cols[9:]]
        out.append("\t".join(cols))
    return "\n".join(out)


def test_reference_binary_reads_the_dialect_variants():
    co = load_golden("cohort_a.json")
    plain = refbin.vcf_text(co["samples"], co["records"])
    variants = {"crlf": plain.replace("\n", "\r\n"), "extra_format_fields": extra_format(plain),
                "meta_lines": plain.replace("\n", "\n##contig=<ID=1>\n##INFO=<ID=AC,Number=A,Type=Integer>\n", 1)}
    base, _, rc = refbin.run_reference(plain, co["refs"], "st")
    assert rc == 0 and base
    ix = O.index(plain.encode())
    want = O.parse_masks(plain.encode(), ix, range(ix["n_lines"]))
    for name, text in variants.items():
        got, _, rc = refbin.run_reference(text, co["refs"], "st")
        assert rc == 0 and got == base, name
        vix = O.index(text.encode())
        assert (O.parse_masks(text.encode(), vix, range(vix["n_lines"])) == want).all(), name
