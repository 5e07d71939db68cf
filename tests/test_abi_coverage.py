"""Every function include/grapes_b200.h declares is called by some test through the loaded library (a call written as
`.grapes_name(` in tests/*.py), or is listed below with the reason it is not: a debugging aid, or an entry point reached
through a Python wrapper, named together with the tests that run that wrapper.  An exported function that no test calls
can break without the suite noticing; this keeps a new one from slipping in that way."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

DEBUG_AIDS = {
    "grapes_debug_partials": "address of the timeline stamps of scripts/trace_fwd_ts.py",
    "grapes_debug_partials_bytes": "size of that buffer (scripts/trace_bwd_ts.py)",
    "grapes_debug_select_fused_stamps": "phase stamps of the fused selection launch, for the timeline scripts",
    "grapes_set_pdl": "launch-ordering switch (GRAPES_PDL) of the loader; every test runs with its default",
}

# name -> the test nodes that run the Python wrapper calling it
WRAPPED = {
    "grapes_aggregate_bf16": ["tests/test_gpu_eval_wide.py::test_rows64_bit_identical_to_int32_aggregation",
                              "tests/test_gpu_sharded_features.py::test_hop_form_bit_identical"],
    "grapes_aggregate_rows64": ["tests/test_gpu_eval_wide.py::test_rows64_bit_identical_to_int32_aggregation"],
    "grapes_aggregate_rows64_peer": ["tests/test_gpu_eval_dp.py::test_peer_aggregation_bit_identical_to_rows64"],
    "grapes_aggregate_rows64_peer_x": ["tests/test_gpu_sharded_features.py::test_slab_form_bit_identical"],
    "grapes_allreduce_adam_peer": [
        "tests/test_gpu_peer_exchange.py::test_peer_allreduce_adam_matches_nccl_and_is_identical_across_ranks"],
    "grapes_classifier_prep": ["tests/test_gpu_engine.py::test_step_parity_trajectory_balance"],
    "grapes_csr_from_edges": ["tests/test_gpu_csr_build.py::test_random_multigraph_matches_scipy",
                              "tests/test_gpu_entry_points.py::test_csr_forced_scatter_forms_match_scipy"],
    "grapes_csr_workspace_bytes": ["tests/test_gpu_csr_build.py::test_random_multigraph_matches_scipy"],
    "grapes_row_offsets": ["tests/test_gpu_eval.py::test_lib_builder_equals_torch_builder",
                           "tests/test_gpu_frontier.py::test_get_neighborhoods_bit_exact"],
    "grapes_expand_rows": ["tests/test_gpu_eval.py::test_lib_builder_equals_torch_builder",
                           "tests/test_gpu_frontier.py::test_get_neighborhoods_bit_exact"],
    "grapes_relabel": ["tests/test_gpu_eval.py::test_mini_batch_eval_engine_path_bit_exact_per_hop"],
    "grapes_slice_block": ["tests/test_gpu_eval.py::test_mini_batch_eval_engine_path_bit_exact_per_hop"],
    **{f"grapes_graph_norm_{s}": ["tests/test_gpu_eval_wide.py::test_builder_equals_torch_builder"]
       for s in ("begin", "add_csr", "add_edges", "offsets", "finish")},
    **{f"grapes_graph_norm_t_{s}": ["tests/test_gpu_full_graph.py::test_transposed_structure_bitwise"]
       for s in ("add_csr", "add_edges", "offsets")},
    **{f"grapes_graph_norm_window_{s}": ["tests/test_gpu_eval_dp.py::test_windows_concatenate_to_the_whole_structure"]
       for s in ("bounds", "add_csr", "add_edges")},
}


def _declared():
    from grapes_b200._lib import parse_header
    return set(parse_header())


def _test_sources():
    return {p: open(p).read() for p in sorted(glob.glob(os.path.join(ROOT, "tests", "*.py")))}


def test_every_entry_point_is_called_by_a_test():
    text = "\n".join(_test_sources().values())
    missing = sorted(n for n in _declared() - DEBUG_AIDS.keys() - WRAPPED.keys()
                     if not re.search(r"\." + re.escape(n) + r"\(", text))
    assert not missing, f"declared in include/grapes_b200.h but called by no test: {missing}"


def test_allowlist_names_declared_functions_and_existing_tests():
    """no stale entry: every listed name is declared, every wrapper-covered one is called from the package (or the
    script a listed test runs), and every named test exists"""
    declared = _declared()
    stale = sorted((DEBUG_AIDS.keys() | WRAPPED.keys()) - declared)
    assert not stale, f"listed but not declared: {stale}"
    callers = glob.glob(os.path.join(ROOT, "grapes_b200", "*.py")) + glob.glob(os.path.join(ROOT, "scripts", "*.py"))
    package = "\n".join(open(p).read() for p in callers)
    unwrapped = sorted(n for n in WRAPPED if not re.search(r"\b" + re.escape(n) + r"\b", package))
    assert not unwrapped, f"listed as covered through a wrapper, but nothing in grapes_b200/ or scripts/ calls them: {unwrapped}"
    for name, nodes in WRAPPED.items():
        assert nodes, name
        for node in nodes:
            path, test = node.split("::")
            src = open(os.path.join(ROOT, path)).read()
            assert re.search(r"^def " + re.escape(test) + r"\(", src, flags=re.M), f"{name}: no test {node}"
