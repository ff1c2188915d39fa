"""CPU: every pass hands its statistics over through the one finish in bgmm_common.cuh.  The last-CTA election and the
publication to the peers are written only there, the tail of state.STATS is indexed only through its named slots, and
bgmm_pass takes no `accumulate` argument."""
import glob
import os
import re

from conftest import ROOT

CSRC = os.path.join(ROOT, "bayesml_b200", "csrc")


def _sources():
    paths = sorted(glob.glob(os.path.join(CSRC, "*.cu*")))
    assert paths
    return {os.path.basename(p): open(p).read() for p in paths}


def test_election_and_publication_live_in_the_common_header():
    for name, text in _sources().items():
        if name == "bgmm_common.cuh":
            continue
        for token in ("BGMM_CTRL_PASS_TICKET", "BGMM_CTRL_COMM_LO", "__threadfence_system", "st.release.sys"):
            assert token not in text, (name, token)


def test_stats_tail_is_indexed_through_named_slots():
    literal = re.compile(r"pitch\)?\s*\+\s*[12]\b")
    for name, text in _sources().items():
        assert not literal.search(text), (name, literal.search(text).group(0))


def test_bgmm_pass_has_no_accumulate_parameter():
    header = open(os.path.join(ROOT, "include", "bgmm.h")).read()
    decl = re.search(r"int bgmm_pass\(([^)]*)\)", header).group(1)
    assert "accumulate" not in decl and decl.rstrip().endswith("void* stream")
    api = open(os.path.join(CSRC, "bgmm_api.cu")).read()
    assert "accumulate" not in re.search(r'extern "C" int bgmm_pass\(([^)]*)\)', api).group(1)
    assert "accumulate" not in re.search(r"struct PassArgs \{(.*?)\};", _sources()["bgmm_common.cuh"], re.S).group(1)
