"""`metadamage fit` command line (cli.py:97-159): same options and defaults, plus
`--max-position` (documented upstream, README.md:121, but never wired: cli.py:105,143) and
`--gpus`, and `--map-only` (MAP-only screening). The `dashboard` sub-command is a visualisation front-end outside this build's scope."""
from pathlib import Path
from typing import List, Optional

import typer

from . import __version__, utils

out_dir_default = Path("./data/out/")
cli_app = typer.Typer(add_completion=False)


def version_callback(value: bool):
    if value:
        typer.echo(f"Metadamage CLI, version: {__version__}")
        raise typer.Exit()


@cli_app.callback()
def callback(version: Optional[bool] = typer.Option(None, "--version", callback=version_callback)):
    """Metagenomics Ancient Damage: metadamage (B200 build). Run `metadamage fit --help`."""


@cli_app.command("fit")
def cli_fit(
    filenames: List[Path] = typer.Argument(...),
    out_dir: Path = typer.Option(out_dir_default),
    max_fits: Optional[int] = typer.Option(None, help="[default: None (All fits)]"),
    max_cores: int = 1,
    max_position: int = typer.Option(15),
    min_alignments: int = 10,
    min_y_sum: int = 10,
    substitution_bases_forward: utils.SubstitutionBases = typer.Option(utils.SubstitutionBases.CT),
    substitution_bases_reverse: utils.SubstitutionBases = typer.Option(utils.SubstitutionBases.GA),
    forced: bool = typer.Option(False, "--forced"),
    gpus: int = typer.Option(1, help="number of B200s of this box to partition the TaxIDs over"),
    map_only: bool = typer.Option(False, "--map-only", help="MAP fits with Laplace uncertainties and a likelihood-ratio "
                                  "test only (no MCMC): writes map_results/<name>.parquet instead of the fit_* tables"),
):
    """Fitting Ancient Damage. FILENAMES are the mismatch-matrix files to fit, e.g.

    \b
        $ metadamage fit --max-fits 10 --max-cores 2 ./data/input/data_ancient.txt
    """
    from .main import main  # deferred: importing the backend needs the built CUDA library

    cfg = utils.Config(
        out_dir=out_dir, max_fits=max_fits, max_cores=max_cores, max_position=max_position,
        min_alignments=min_alignments, min_y_sum=min_y_sum,
        substitution_bases_forward=substitution_bases_forward.value,
        substitution_bases_reverse=substitution_bases_reverse.value,
        forced=forced, version="0.0.0", gpus=gpus,
    )
    cfg.add_filenames(filenames)
    main(filenames, cfg, map_only=map_only)


@cli_app.command("dashboard")
def cli_dashboard(dir: Path = typer.Argument(out_dir_default)):
    """Not part of this build: the parquet outputs are schema-compatible with the reference's dashboard."""
    typer.echo("The dashboard is not part of metadamage_b200; point the reference's `metadamage dashboard` at "
               f"{dir} (the parquet schemas are unchanged).")
    raise typer.Exit(code=2)


def cli_main():
    cli_app(prog_name="metadamage")
