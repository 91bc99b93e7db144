"""CPU: the multi-batch zero-list and decoded-read forms reach every layer - the Python methods
take region-mode loci, include/dkb.hpp wraps both C calls, and the Rust safe crate's
Counter::submit_multi sends zero lists through dkb_batch_submit_sparse_multi."""
import inspect
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _read(*parts):
    with open(os.path.join(ROOT, *parts)) as f:
        return f.read()


def test_python_methods_take_loci(dkb):
    for name in ("submit_sparse_multi", "submit_reads_multi"):
        params = inspect.signature(getattr(dkb.KmerCounter, name)).parameters
        assert "loci" in params and params["loci"].default is None, name
    assert "four_bit" in inspect.signature(dkb.KmerCounter.submit_reads_multi).parameters


def test_cpp_layer_declares_both_calls():
    hpp = _read("include", "dkb.hpp")
    for fn in ("dkb_batch_submit_sparse_multi", "dkb_batch_submit_reads_multi"):
        assert re.search(r"check\(\s*" + fn + r"\(", hpp), fn
    assert "void submit_sparse_multi(" in hpp and "void submit_reads_multi(" in hpp


def _rust_fn(src, name):
    """The body of `pub fn name` in a Rust source (up to the next `pub fn` or `fn`)."""
    m = re.search(r"pub fn " + name + r"\b(.*?)(?=\n    (?:pub )?fn |\n    ///)", src, re.S)
    assert m, name
    return m.group(1)


def test_rust_submit_multi_sends_zero_lists():
    src = _read("bindings", "rust", "denovo-kmer-gpu", "src", "lib.rs")
    body = _rust_fn(src, "submit_multi")
    assert "sys::dkb_batch_submit_sparse_multi(" in body
    assert "sys::dkb_batch_submit_multi(" in body  # the dense flags when a batch has no zero list
    assert "sys::dkb_batch_submit_reads_multi(" in _rust_fn(src, "submit_reads_multi")
