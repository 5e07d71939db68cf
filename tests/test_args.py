"""CPU tests: the Tap-compatible ``Arguments`` parser accepts every config file of the reference
(read from the checkout GRAPES_REFERENCE_ROOT names, when it is set) and the spellings those files use."""
import glob
import os

import pytest

from grapes_b200.args import Arguments, parse_cli
from oracle.ref_import import REFERENCE_ROOT, reference_available

REF_CONFIGS = sorted(glob.glob(os.path.join(REFERENCE_ROOT, "configs", "*", "*.txt"))) if REFERENCE_ROOT else []
needs_reference = pytest.mark.skipif(not reference_available(),
                                     reason="needs GRAPES_REFERENCE_ROOT: a checkout of the reference GRAPES project")


def test_defaults_match_reference_main_py():
    a = Arguments()
    assert (a.dataset, a.sampling_hops, a.num_samples, a.use_indicators) == ('cora', 2, 16, True)
    assert (a.lr_gf, a.lr_gc, a.loss_coef, a.log_z_init, a.reg_param, a.dropout) == (1e-4, 1e-3, 1e4, 0., 0., 0.)
    assert (a.model_type, a.hidden_dim, a.embed_nodes, a.node_emb_dim, a.max_epochs, a.batch_size) == ('gcn', 256, False, 64, 30, 512)
    assert (a.eval_frequency, a.eval_on_cpu, a.eval_full_batch, a.random_sampling, a.runs) == (5, True, True, False, 10)
    assert (a.log_wandb, a.config_file, a.reinforce_baseline, a.seed) == (False, None, False, None)


def test_both_spellings_quotes_and_bool_prefixes(tmp_path):
    cfg = tmp_path / "c.txt"
    cfg.write_text('--batch_size 256\n--dataset "products"\n--eval_full_batch true\n--loss_coef=15227.12\n'
                   '--use_indicators=True\n--random_sampling=False\n--log_wandb t\n--runs 3\n')
    a = parse_cli(["--config_file", str(cfg), "--runs=7", "--sampling_hops", "3"])
    assert a.batch_size == 256 and a.dataset == "products" and a.eval_full_batch is True
    assert a.loss_coef == 15227.12 and a.use_indicators is True and a.random_sampling is False and a.log_wandb is True
    assert a.runs == 7 and a.sampling_hops == 3               # the command line wins over the file (main.py:369-373)


def test_unknown_flag_and_bad_bool_are_errors():
    with pytest.raises(SystemExit):
        Arguments.parse_args(["--no_such_flag", "1"])
    with pytest.raises(SystemExit):
        Arguments.parse_args(["--use_indicators", "maybe"])


@needs_reference
def test_every_reference_config_file_parses():
    bad = []
    for path in REF_CONFIGS:
        try:
            a = parse_cli(["--config_file", path])
            assert a.hidden_dim > 0 and a.num_samples > 0
        except SystemExit:
            bad.append(os.path.relpath(path, REFERENCE_ROOT))
    # configs/rl/flickr.txt:15 is malformed in the reference itself ("--runs=1 0", SURVEY.md section 5)
    assert bad == ["configs/rl/flickr.txt"], bad
    assert len(REF_CONFIGS) == 32


@needs_reference
def test_fields_and_defaults_match_the_live_reference_class():
    """main.py:23-54 read from the reference's own source (AST of ``class Arguments(Tap)``): same field names in the same
    order, same defaults."""
    import ast
    import dataclasses
    tree = ast.parse(open(os.path.join(REFERENCE_ROOT, "main.py")).read())
    cls = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "Arguments")
    ref = [(n.target.id, ast.literal_eval(n.value)) for n in cls.body if isinstance(n, ast.AnnAssign)]
    mine = [(f.name, f.default) for f in dataclasses.fields(Arguments)]
    assert mine == ref and len(ref) == 27


@needs_reference
def test_arguments_object_drives_the_live_reference_train():
    """The drop-in ``Arguments`` is accepted by the reference's OWN ``train(args)`` (main.py:57-340 executed live, see
    oracle/ref_import.py::load_reference_train): every attribute the loop reads, and ``as_dict()`` (main.py:61)."""
    from grapes_b200.synth import make_synth
    from oracle import ref_import
    d = make_synth("tiny", seed=0)
    a = Arguments.parse_args(["--dataset", "tiny", "--batch_size", "32", "--num_samples", "8", "--sampling_hops", "2",
                              "--max_epochs", "1", "--eval_full_batch", "True"])
    f1, logs, nets = ref_import.run_reference_train(d, weight_seed=100, rng_seed=4242, args_obj=a)
    assert len(logs) == 4 and 0.0 < f1 < 1.0 and len(nets) == 3
