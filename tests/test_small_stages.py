"""CPU: bgmm_small's two kernels (the block kernel for D > 32, one warp per component for D <= 32) share one copy of every
stage but the dense algebra: the peer receive, the ELBO terms, the finaliser that owns the loop control, and one host
launcher."""
import os
import re

from conftest import ROOT

SRC = os.path.join(ROOT, "bayesml_b200", "csrc", "bgmm_small.cu")


def _source():
    return open(SRC).read()


def _function_body(text, name):
    start = re.search(r"\b" + name + r"\(", text).start()
    return start, text.index("\n}\n", start)


def test_peer_receive_is_written_once():
    assert _source().count("ld.acquire.sys") == 1


def test_loop_control_lives_in_the_finaliser():
    text = _source()
    start, end = _function_body(text, "finish_iteration")
    for token in ("BGMM_CTRL_TICKET", "BGMM_CTRL_CONVERGED"):
        where = [m.start() for m in re.finditer(token, text)]
        assert where and all(start < w < end for w in where), token


def test_elbo_terms_are_written_once():
    text = _source()
    for tag in (":673-683", ":692-701", ":710-715", ":717-723"):
        assert text.count(tag) == 1, tag


def test_one_host_launcher():
    text = _source()
    assert text.count("cudaFuncAttributeMaxDynamicSharedMemorySize") == 1
    # the block kernel runs for D > 32 only: 128 threads up to D = 64, 256 above
    assert not re.search(r"\?\s*(32|64)\s*:", text)
    assert "D <= 64 ? 128 : 256" in text


def test_hmm_trans_kernel_uses_block_max():
    text = _source()
    start, end = _function_body(text, "hmm_trans_kernel")
    body = text[start:end]
    assert "red[tid >> 5]" not in body and body.count("block_max(") == 2
