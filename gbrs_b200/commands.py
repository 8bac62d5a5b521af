"""`gbrs quantify` command line -- same flags as the reference (/root/reference/src/gbrs/gbrs/commands.py:108-150):
-i -g -L -G -o -M -p -m -t -a -w -v, `gbrs compress` (:76-105): -i (repeatable / comma separated) -o -c -v,
`gbrs stencil` (:343-370): -i -G -g -o -v, and `gbrs reconstruct` (:153-183): -e -t -x -g -c -s -o -v.
Errors are logged, not raised, and the process exits 0 (:146-150)."""
from __future__ import annotations

import logging
from pathlib import Path
from typing import Annotated

import typer

import importlib

from . import utils

# the package re-exports the *function* `quantify`, which shadows the sub-module of the same name on `from . import`
quantify_mod = importlib.import_module(".quantify", __package__)

app = typer.Typer(help="GBRS (B200-native multiway EM quantifier)", add_completion=False)


@app.callback()
def _main() -> None:  # keeps `quantify` a sub-command, as in the reference's multi-command app
    pass


@app.command(help="quantify allele-specific expressions")
def quantify(
    alignment_file: Annotated[Path, typer.Option("-i", "--alignment-file", exists=True, dir_okay=False, resolve_path=True, help="EMASE alignment incidence file (hdf5 or npz twin)")],
    group_file: Annotated[Path, typer.Option("-g", "--group-file", exists=True, dir_okay=False, resolve_path=True, help="tab delimited file of gene to transcript mapping")] = None,
    length_file: Annotated[Path, typer.Option("-L", "--length-file", exists=True, dir_okay=False, resolve_path=True, help="tab delimited file of locus(transcript) and length")] = None,
    genotype_file: Annotated[Path, typer.Option("-G", "--genotype", exists=True, dir_okay=False, resolve_path=True, help="tab delimited file of locus(transcipt) and diplotype")] = None,
    outbase: Annotated[str, typer.Option("-o", "--outbase", help="basename of all the generated output files")] = "gbrs.quantified",
    multiread_model: Annotated[int, typer.Option("-M", "--multiread-model", help="emase model (default: 4)")] = 4,
    pseudocount: Annotated[float, typer.Option("-p", "--pseudocount", help="prior read count (default: 0.0)")] = 0.0,
    max_iters: Annotated[int, typer.Option("-m", "--max-iters", help="maximum iterations for EM iteration")] = 999,
    tolerance: Annotated[float, typer.Option("-t", "--tolerance", help="tolerance for EM termination (default: 0.0001 in TPM)")] = 0.0001,
    report_alignment_counts: Annotated[bool, typer.Option("-a", "--report-alignment-counts", help="whether to report alignment counts")] = False,
    report_posterior: Annotated[bool, typer.Option("-w", "--report-posterior", help="whether to report posterior probabilities")] = False,
    bootstrap: Annotated[int, typer.Option("--bootstrap", help="bootstrap replicates, written to <outbase>.bootstrap.npz after the reports (default: 0 = none)")] = 0,
    bootstrap_seed: Annotated[int, typer.Option("--bootstrap-seed", help="seed of the bootstrap replicates (default: 0)")] = 0,
    bootstrap_output: Annotated[str, typer.Option("--bootstrap-output", help="what --bootstrap writes: npz (the replicates), summary (mean / sd / interval tables) or both (default: npz)")] = "npz",
    bootstrap_interval: Annotated[float, typer.Option("--bootstrap-interval", help="central interval of the bootstrap summary tables (default: 0.95)")] = 0.95,
    verbose: Annotated[int, typer.Option("-v", "--verbose", count=True, help="specify multiple times for more verbose output")] = 0,
) -> None:
    logger = utils.configure_logging("gbrs", verbose)
    logger.debug("quantify")
    try:
        if multiread_model not in (1, 2, 3, 4):
            raise typer.Abort("-M, --multiread-model must be one of 1, 2, 3, or 4")
        quantify_mod.quantify(
            alignment_file=str(alignment_file),
            group_file=str(group_file) if group_file else None,
            length_file=str(length_file) if length_file else None,
            genotype_file=str(genotype_file) if genotype_file else None,
            outbase=outbase, multiread_model=multiread_model, pseudocount=pseudocount, max_iters=max_iters,
            tolerance=tolerance, report_alignment_counts=report_alignment_counts, report_posterior=report_posterior,
            bootstrap=bootstrap, bootstrap_seed=bootstrap_seed, bootstrap_output=bootstrap_output,
            bootstrap_interval=bootstrap_interval)
    except Exception as e:  # reference policy: log and return
        if logger.level == logging.DEBUG:
            logger.exception(e)
        else:
            logger.error(e)


@app.command(help="compress EMASE format alignment incidence matrix")
def compress(
    emase_files: Annotated[list[Path], typer.Option("-i", "--emase-file", exists=False, dir_okay=False, resolve_path=True, help='EMASE file to compress, can seperate files by "," or have multiple -i')],
    output_file: Annotated[Path, typer.Option("-o", "--output", exists=False, dir_okay=False, writable=True, resolve_path=True, help="name of the compressed EMASE file")],
    comp_lib: Annotated[str, typer.Option("-c", "--comp-lib", help="compression library to use")] = "zlib",
    verbose: Annotated[int, typer.Option("-v", "--verbose", count=True, help="specify multiple times for more verbose output")] = 0,
) -> None:
    """Flag surface of the reference's `gbrs compress` (/root/reference/src/gbrs/gbrs/commands.py:76-105)."""
    logger = utils.configure_logging("gbrs", verbose)
    logger.debug("compress")
    try:
        # file shortcut: -i abc.h5 -i def.h5  ==  -i abc.h5,def.h5   (:86-91)
        all_emase_files: list[str] = []
        for x in emase_files:
            all_emase_files.extend(str(x).split(","))
        for f in all_emase_files:
            if not Path(f).is_file():
                raise FileNotFoundError(f"{f} does not exist or is not a file")
        importlib.import_module(".compress", __package__).compress(
            emase_files=all_emase_files, output_file=str(output_file), comp_lib=comp_lib)
    except Exception as e:
        if logger.level == logging.DEBUG:
            logger.exception(e)
        else:
            logger.error(e)


@app.command(help="apply genotype calls to multi-way alignment incidence matrix")
def stencil(
    alignment_file: Annotated[Path, typer.Option("-i", "--alignment-file", exists=True, dir_okay=False, resolve_path=True, help="alignment incidence file (h5)")],
    genotype_file: Annotated[Path, typer.Option("-G", "--genotype", exists=True, dir_okay=False, resolve_path=True, help="genotype calls by GBRS (tsv)")],
    group_file: Annotated[Path, typer.Option("-g", "--group-file", exists=True, dir_okay=False, resolve_path=True, help="gene ID to isoform ID mapping info (tsv)")] = None,
    output_file: Annotated[Path, typer.Option("-o", "--output", exists=False, dir_okay=False, writable=True, resolve_path=True, help="genotyped version of alignment incidence file (h5)")] = None,
    verbose: Annotated[int, typer.Option("-v", "--verbose", count=True, help="specify multiple times for more verbose output")] = 0,
) -> None:
    """Flag surface of the reference's `gbrs stencil` (/root/reference/src/gbrs/gbrs/commands.py:343-370)."""
    logger = utils.configure_logging("gbrs", verbose)
    logger.debug("stencil")
    try:
        importlib.import_module(".stencil", __package__).stencil(
            alignment_file=str(alignment_file), genotype_file=str(genotype_file),
            group_file=str(group_file) if group_file else None, output_file=str(output_file) if output_file else None)
    except Exception as e:
        if logger.level == logging.DEBUG:
            logger.exception(e)
        else:
            logger.error(e)


@app.command(help="reconstruct the genome based upon gene-level TPM quantities")
def reconstruct(
    expression_file: Annotated[Path, typer.Option("-e", "--expr-file", exists=True, dir_okay=False, resolve_path=True, help="file containing gene-level TPM quantities")],
    tprob_file: Annotated[Path, typer.Option("-t", "--tprob-file", exists=True, dir_okay=False, resolve_path=True, help="transition probabilities file")],
    avec_file: Annotated[Path, typer.Option("-x", "--avec-file", exists=True, dir_okay=False, resolve_path=True, help="alignment specificity file")] = None,
    gpos_file: Annotated[Path, typer.Option("-g", "--gpos-file", exists=True, dir_okay=False, resolve_path=True, help="meta information for genes (chrom, id, location)")] = None,
    expr_threshold: Annotated[float, typer.Option("-c", "--expr-threshold")] = 1.5,
    sigma: Annotated[float, typer.Option("-s", "--sigma")] = 0.12,
    outbase: Annotated[str, typer.Option("-o", "--outbase", help="basename of all the generated output files")] = None,
    verbose: Annotated[int, typer.Option("-v", "--verbose", count=True, help="specify multiple times for more verbose output")] = 0,
) -> None:
    """Flag surface of the reference's `gbrs reconstruct` (/root/reference/src/gbrs/gbrs/commands.py:153-183)."""
    logger = utils.configure_logging("gbrs", verbose)
    logger.debug("reconstruct")
    try:
        importlib.import_module(".reconstruct", __package__).reconstruct(
            expression_file=str(expression_file), tprob_file=str(tprob_file),
            avec_file=str(avec_file) if avec_file else None, gpos_file=str(gpos_file) if gpos_file else None,
            expr_threshold=expr_threshold, sigma=sigma, outbase=outbase)
    except Exception as e:
        if logger.level == logging.DEBUG:
            logger.exception(e)
        else:
            logger.error(e)


@app.command(help="run EMASE (the same quantifier without genotype restriction; reference `emase run`)")
def run(
    alignment_file: Annotated[Path, typer.Option("-i", "--alignment-file", exists=True, dir_okay=False, resolve_path=True, help="EMASE alignment incidence file (hdf5 or npz twin)")],
    group_file: Annotated[Path, typer.Option("-g", "--group-file", exists=True, dir_okay=False, resolve_path=True, help="tab delimited file of gene to transcript mapping")] = None,
    length_file: Annotated[Path, typer.Option("-L", "--length-file", exists=True, dir_okay=False, resolve_path=True, help="tab delimited file of locus(transcript) and length")] = None,
    outbase: Annotated[str, typer.Option("-o", "--outbase", help="basename of all the generated output files")] = "emase",
    multiread_model: Annotated[int, typer.Option("-M", "--multiread-model", help="emase model (default: 4)")] = 4,
    pseudocount: Annotated[float, typer.Option("-p", "--pseudocount", help="prior read count (default: 0.0)")] = 0.0,
    read_length: Annotated[int, typer.Option("-l", "--read-length", help="specify read length")] = 100,
    max_iters: Annotated[int, typer.Option("-m", "--max-iters", help="maximum iterations for EM iteration")] = 999,
    tolerance: Annotated[float, typer.Option("-t", "--tolerance", help="tolerance for EM termination (default: 0.0001 in TPM)")] = 0.0001,
    report_alignment_counts: Annotated[bool, typer.Option("-c", "--report-alignment-counts", help="whether to report alignment counts")] = False,
    report_posterior: Annotated[bool, typer.Option("-w", "--report-posterior", help="whether to report posterior probabilities")] = False,
    bootstrap: Annotated[int, typer.Option("--bootstrap", help="bootstrap replicates, written to <outbase>.bootstrap.npz after the reports (default: 0 = none)")] = 0,
    bootstrap_seed: Annotated[int, typer.Option("--bootstrap-seed", help="seed of the bootstrap replicates (default: 0)")] = 0,
    bootstrap_output: Annotated[str, typer.Option("--bootstrap-output", help="what --bootstrap writes: npz (the replicates), summary (mean / sd / interval tables) or both (default: npz)")] = "npz",
    bootstrap_interval: Annotated[float, typer.Option("--bootstrap-interval", help="central interval of the bootstrap summary tables (default: 0.95)")] = 0.95,
    verbose: Annotated[int, typer.Option("-v", "--verbose", count=True, help="specify multiple times for more verbose output")] = 0,
) -> None:
    """Flag surface of the reference's `emase run` (/root/reference/src/gbrs/emase/commands.py:315-356)."""
    logger = utils.configure_logging("gbrs", verbose)
    logger.debug("run")
    try:
        if multiread_model not in (1, 2, 3, 4):
            raise typer.Abort("-M, --multiread-model must be one of 1, 2, 3, or 4")
        quantify_mod.run(
            alignment_file=str(alignment_file), group_file=str(group_file) if group_file else None,
            length_file=str(length_file) if length_file else None, outbase=outbase, multiread_model=multiread_model,
            read_length=read_length, pseudocount=pseudocount, max_iters=max_iters, tolerance=tolerance,
            report_alignment_counts=report_alignment_counts, report_posterior=report_posterior,
            bootstrap=bootstrap, bootstrap_seed=bootstrap_seed, bootstrap_output=bootstrap_output,
            bootstrap_interval=bootstrap_interval)
    except Exception as e:
        if logger.level == logging.DEBUG:
            logger.exception(e)
        else:
            logger.error(e)


if __name__ == "__main__":
    app()
