"""The text-format codes of the Python binding agree with include/kmerust_gpu.h (no device needed)."""
import os
import re

from krust_b200 import _lib
from krust_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_text_format_codes_match_the_header():
    with open(os.path.join(ROOT, "include", "kmerust_gpu.h")) as f:
        header = f.read()
    codes = dict((name, int(v)) for name, v in re.findall(r"\b(KMG_TEXT_[A-Z]+)\s*=\s*(\d+)", header))
    assert codes == {"KMG_TEXT_FASTA": 0, "KMG_TEXT_TSV": 1, "KMG_TEXT_JSON": 2}
    assert {name: getattr(_lib, name) for name in codes} == codes
    assert api._TEXT_FORMATS == {"fasta": codes["KMG_TEXT_FASTA"], "tsv": codes["KMG_TEXT_TSV"], "json": codes["KMG_TEXT_JSON"]}
