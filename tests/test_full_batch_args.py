"""CPU tests of the full-graph training driver (grapes_b200.full_batch): argument handling, the refusals that come before
any device work, and the working-set estimate."""
import pytest


def test_cli_parses_the_arguments_of_main(tmp_path):
    from grapes_b200.args import parse_cli
    cfg = tmp_path / "cfg.txt"
    cfg.write_text('--dataset "synth:arxiv" --hidden_dim 128 --max_epochs 7 --embed_nodes true\n')
    a = parse_cli(["--config_file", str(cfg), "--max_epochs", "5", "--runs", "2"])
    assert (a.dataset, a.hidden_dim, a.max_epochs, a.runs, a.embed_nodes) == ("synth:arxiv", 128, 5, 2, True)
    with pytest.raises(SystemExit):
        parse_cli(["--no_such_flag", "1"])


def test_refuses_data_parallel(monkeypatch):
    from grapes_b200 import full_batch as fb
    from grapes_b200._lib import GrapesError
    from grapes_b200.args import Arguments
    monkeypatch.setenv("WORLD_SIZE", "2")
    with pytest.raises(GrapesError, match="one GPU"):
        fb.train(Arguments(dataset="synth:tiny"))


def test_working_set_estimate():
    """papers100M-shaped training does not fit a 180 GB device; the arxiv, Reddit and products shapes do."""
    from grapes_b200.full_batch import working_set_bytes
    from grapes_b200.synth import SHAPES
    fits = {k: working_set_bytes(s["N"], s["E_dir"], s["F"], 256, s["C"]) < 180e9 for k, s in SHAPES.items()}
    assert not fits["papers"]
    assert fits["arxiv"] and fits["reddit"] and fits["products"]
    s = SHAPES["arxiv"]
    assert working_set_bytes(s["N"], s["E_dir"], 64, 256, s["C"], embed_nodes=True) > \
        working_set_bytes(s["N"], s["E_dir"], 64, 256, s["C"])
