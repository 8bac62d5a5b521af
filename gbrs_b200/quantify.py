"""`quantify` workflow -- same arguments, defaults, masking, output files and headers as the reference's
`gbrs.gbrs.emase_utils.quantify` (/root/reference/src/gbrs/gbrs/emase_utils.py:180-332), with the EM itself on
the GPU (gbrs_b200.EMfactory)."""
from __future__ import annotations

import os
from itertools import dropwhile

import numpy as np

from . import utils
from .apm import AlignmentPropertyMatrix
from .bootstrap import SUMMARY_MAX_REPLICATES
from .emfactory import EMfactory

DATA_DIR = os.getenv("GBRS_DATA", ".")
logger = utils.get_logger("gbrs")


def load_genotype_mask(aln_mat: AlignmentPropertyMatrix, genotype_file: str):
    """Genotype TSV -> (gtmask H x T, gtcall_g, gtcall_t)   (emase_utils.py:240-269).  The reference sets the mask gene
    by gene (a meshgrid assignment and a loop over the gene's transcripts per line: a second at 32k genes); here the
    lines are parsed in the same order with the same look-ups -- an unknown gene or haplotype letter raises the same
    KeyError -- and the mask and the transcript notes are then filled in bulk."""
    hid = dict(zip(aln_mat.hname, np.arange(aln_mat.num_haplotypes)))
    gid = dict(zip(aln_mat.gname, np.arange(len(aln_mat.gname))))
    gtmask = np.zeros((aln_mat.num_haplotypes, aln_mat.num_loci))
    gtcall_g = dict.fromkeys(aln_mat.gname)
    gtcall_t = dict.fromkeys(aln_mat.lname)
    genes, calls, haps = [], [], []
    with open(genotype_file) as fh:
        for curline in dropwhile(utils.is_comment, fh):
            item = curline.rstrip().split("\t")
            g, gt = item[:2]
            gtcall_g[g] = gt
            haps.append([hid[c] for c in gt])
            genes.append(gid[g])
            calls.append(gt)
    if not genes:
        return gtmask, gtcall_g, gtcall_t
    groups = aln_mat.groups
    size = np.fromiter((len(groups[g]) for g in genes), dtype=np.int64, count=len(genes))
    loci = np.fromiter((t for g in genes for t in groups[g]), dtype=np.int64, count=int(size.sum()))
    line_of = np.repeat(np.arange(len(genes)), size)
    width = max(len(h) for h in haps)
    hap_tab = np.full((len(genes), max(width, 1)), -1, dtype=np.int64)
    for i, h in enumerate(haps):
        hap_tab[i, : len(h)] = h
    for k in range(width):
        h = hap_tab[line_of, k]
        ok = h >= 0
        gtmask[h[ok], loci[ok]] = 1.0
    lname = aln_mat.lname
    for t, i in zip(loci.tolist(), line_of.tolist()):  # later lines win, as in the reference's loop
        gtcall_t[lname[t]] = calls[i]
    return gtmask, gtcall_g, gtcall_t


def hapmask_bytes(gtmask: np.ndarray) -> np.ndarray:
    """H x T 0/1 genotype mask -> uint8 [T] with bit h set where haplotype h of the locus is kept."""
    H = gtmask.shape[0]
    bits = (np.asarray(gtmask) != 0).astype(np.uint8)
    return (bits << np.arange(H, dtype=np.uint8)[:, None]).sum(axis=0).astype(np.uint8)


def _write_reports(em_factory, outbase, alignment_file, group_file, report_group_counts, report_alignment_counts,
                   report_posterior, notes_t=None, notes_g=None, unmasked=None, unmasked_pattern=None):
    """The output section shared by `quantify` (gbrs/emase_utils.py:288-331) and `run` (emase/emase_utils.py:650-695)."""
    logger.info(f"Generating isoform TPMs: {outbase}.isoforms.tpm")
    em_factory.report_depths(filename=f"{outbase}.isoforms.tpm", tpm=True, notes=notes_t)
    logger.info(f"Generating isoform Read Counts: {outbase}.isoforms.expected_read_counts")
    em_factory.report_read_counts(filename=f"{outbase}.isoforms.expected_read_counts", notes=notes_t)
    if report_posterior:
        logger.info(f"Generating Posterior Probabilities: {outbase}.posterior.h5")
        em_factory.export_posterior_probability(filename=f"{outbase}.posterior.h5")
    if report_group_counts:
        logger.info(f"Generating gene TPMs: {outbase}.genes.tpm")
        em_factory.report_depths(filename=f"{outbase}.genes.tpm", tpm=True, grp_wise=True, notes=notes_g)
        logger.info(f"Generating gene Read Counts: {outbase}.genes.expected_read_counts")
        em_factory.report_read_counts(filename=f"{outbase}.genes.expected_read_counts", grp_wise=True, notes=notes_g)
    if report_alignment_counts:
        # The reference reloads the file, i.e. counts are taken on the *unmasked* matrix (gbrs/emase_utils.py:319).
        # Here the host matrix is still unmasked unless `-w` forced the in-place restriction, so it is reused; for a
        # multiway run even the EM's packed, device-resident pattern is reused.
        alnmat = unmasked if unmasked is not None else AlignmentPropertyMatrix(h5file=alignment_file, grpfile=group_file)
        logger.info(f"Generating isoform Alignment Counts: {outbase}.isoforms.alignment_counts")
        alnmat.report_alignment_counts(filename=f"{outbase}.isoforms.alignment_counts", pattern=unmasked_pattern)
        if report_group_counts:
            logger.info(f"Generating gene Alignment Counts: {outbase}.genes.alignment_counts")
            alnmat.report_alignment_counts(filename=f"{outbase}.genes.alignment_counts", gene_level=True,
                                           pattern=unmasked_pattern)


BOOTSTRAP_OUTPUTS = ("npz", "summary", "both")


def check_bootstrap_args(bootstrap, bootstrap_output, bootstrap_interval) -> None:
    """The refusals of the bootstrap flags that need no data, checked before the input is loaded and the EM runs."""
    if bootstrap_output not in BOOTSTRAP_OUTPUTS:
        raise ValueError(f"--bootstrap-output must be one of {', '.join(BOOTSTRAP_OUTPUTS)}")
    if not 0.0 < bootstrap_interval < 1.0:
        raise ValueError("--bootstrap-interval must be in (0, 1)")
    if bootstrap > 0 and bootstrap_output != "npz" and not 2 <= bootstrap <= SUMMARY_MAX_REPLICATES:
        raise ValueError(f"bootstrap summaries need 2 to {SUMMARY_MAX_REPLICATES} replicates")


def _write_bootstrap(em_factory, outbase, bootstrap, bootstrap_seed, multiread_model, pseudocount, tolerance, max_iters,
                     bootstrap_output="npz", bootstrap_interval=0.95, notes_t=None, notes_g=None):
    """`--bootstrap N`: N replicates (indices 0..N-1 of `bootstrap_seed`) after the point-estimate reports.
    `bootstrap_output`: "npz" writes them to {outbase}.bootstrap.npz (BootstrapResult.save); "summary" writes the
    summary tables {outbase}.bootstrap.{isoforms,genes}.{tpm,expected_read_counts,allelic_share}.summary
    (BootstrapSummary.write, interval `bootstrap_interval`); "both" writes both from one set of replicates."""
    if bootstrap <= 0:
        return
    path = f"{outbase}.bootstrap.npz"
    kw = dict(model=multiread_model, seed=bootstrap_seed, pseudocount=pseudocount, tol=tolerance, max_iters=max_iters)
    if bootstrap_output == "npz":
        logger.info(f"Running {bootstrap} bootstrap replicates (seed {bootstrap_seed}): {path}")
        em_factory.bootstrap(bootstrap, **kw).save(path)
        return
    logger.info(f"Running {bootstrap} bootstrap replicates (seed {bootstrap_seed}): {outbase}.bootstrap.*.summary")
    summary = em_factory.bootstrap_summary(bootstrap, interval=bootstrap_interval,
                                           keep_replicates=bootstrap_output == "both", **kw)
    summary.write(outbase, notes_t=notes_t, notes_g=notes_g)
    if bootstrap_output == "both":
        summary.result.save(path)


def run(alignment_file: str, group_file: str = None, length_file: str = None, outbase: str = "emase",
        multiread_model: int = 4, read_length: int = 100, pseudocount: float = 0.0, max_iters: int = 999,
        tolerance: float = 0.0001, report_alignment_counts: bool = False, report_posterior: bool = False,
        device=None, group=None, bootstrap: int = 0, bootstrap_seed: int = 0, bootstrap_output: str = "npz",
        bootstrap_interval: float = 0.95) -> None:
    """`emase run` workflow (reference `gbrs.emase.emase_utils.run`, emase/emase_utils.py:594-696): the same EM without
    the genotype restriction, with an explicit read length and no default group / length files.  `bootstrap` /
    `bootstrap_seed` / `bootstrap_output` / `bootstrap_interval`: replicates written after the reports (see
    `_write_bootstrap`; 0 = none)."""
    check_bootstrap_args(bootstrap, bootstrap_output, bootstrap_interval)
    report_group_counts = group_file is not None
    logger.info(f"Alignment File: {alignment_file}")
    logger.info(f"Group File: {group_file}")
    logger.info(f"Read Length File: {length_file}")
    logger.info(f"Read Length: {read_length}")
    logger.info(f"Outbase: {outbase}")
    logger.info(f"Multiread Model: {multiread_model}")
    logger.info(f"Loading EMASE file: {alignment_file}")
    aln_mat = AlignmentPropertyMatrix(h5file=alignment_file, grpfile=group_file)
    logger.info("Running EMASE")
    em_factory = EMfactory(aln_mat, device=device, group=group)
    em_factory.prepare(pseudocount=pseudocount, lenfile=length_file, read_length=read_length)
    em_factory.run(model=multiread_model, tol=tolerance, max_iters=max_iters, verbose=True)
    if em_factory.rank == 0:
        reuse_pattern = em_factory.world == 1 and em_factory._pattern.packed.has_genes
        _write_reports(em_factory, outbase, alignment_file, group_file, report_group_counts, report_alignment_counts,
                       report_posterior, unmasked=aln_mat, unmasked_pattern=em_factory._pattern if reuse_pattern else None)
        _write_bootstrap(em_factory, outbase, bootstrap, bootstrap_seed, multiread_model, pseudocount, tolerance, max_iters,
                         bootstrap_output, bootstrap_interval)
    logger.debug("Done")


def quantify(alignment_file: str, group_file: str = None, length_file: str = None, genotype_file: str = None,
             outbase: str = "gbrs.quantified", multiread_model: int = 4, pseudocount: float = 0.0,
             max_iters: int = 999, tolerance: float = 0.0001, report_alignment_counts: bool = False,
             report_posterior: bool = False, device=None, group=None, bootstrap: int = 0, bootstrap_seed: int = 0,
             bootstrap_output: str = "npz", bootstrap_interval: float = 0.95) -> None:
    """Quantify expected read counts.  Additions: `device` / `group`, the CUDA device to use and an optional
    torch.distributed process group over which the alignment classes are row-sharded; `bootstrap` / `bootstrap_seed` /
    `bootstrap_output` / `bootstrap_interval`, replicates written after the reports (see `_write_bootstrap`; 0 = none)."""
    check_bootstrap_args(bootstrap, bootstrap_output, bootstrap_interval)
    if group_file is None:
        group_file = os.path.join(DATA_DIR, "ref.gene2transcripts.tsv")
        if not os.path.exists(group_file):
            logger.warning("A group file is not given. Group-level results will not be reported.")
    if length_file is None:
        length_file = os.path.join(DATA_DIR, "gbrs.hybridized.targets.info")
        if not os.path.exists(length_file):
            logger.warning("A length file is not given. Transcript length adjustment will *not* be performed.")

    report_group_counts = group_file is not None  # always true here, as in the reference (:219-222)

    logger.info(f"Alignment File: {alignment_file}")
    logger.info(f"Group File: {group_file}")
    logger.info(f"Length File: {length_file}")
    logger.info(f"Genotype File: {genotype_file}")
    logger.info(f"Outbase: {outbase}")
    logger.info(f"Multiread Model: {multiread_model}")
    logger.info(f"Pseudocount: {pseudocount}")
    logger.info(f"Tolerance: {tolerance}")
    logger.info(f"Report Alignment Counts: {report_alignment_counts}")
    logger.info(f"Report Posterior: {report_posterior}")

    logger.info(f"Loading EMASE file: {alignment_file}")
    aln_mat = AlignmentPropertyMatrix(h5file=alignment_file, grpfile=group_file)
    locus_hapmask = None

    if genotype_file is not None:
        outbase = f"{outbase}.diploid"
        logger.info(f"Loading and processing genotype calls from: {genotype_file}")
        gtmask, gtcall_g, gtcall_t = load_genotype_mask(aln_mat, genotype_file)
        if report_posterior:
            # the exported pattern must be the restricted one, as in the reference (emase_utils.py:271-273)
            aln_mat.multiply(gtmask, axis=2)
            aln_mat.eliminate_zeros()
        else:
            # same restriction applied while packing: one byte per locus, bit h = haplotype h survives
            locus_hapmask = hapmask_bytes(gtmask)
    else:
        outbase = f"{outbase}.multiway"
        gtcall_g = None
        gtcall_t = None

    logger.info("Running EMASE")
    em_factory = EMfactory(aln_mat, device=device, group=group, locus_hapmask=locus_hapmask)
    em_factory.prepare(pseudocount=pseudocount, lenfile=length_file)
    em_factory.run(model=multiread_model, tol=tolerance, max_iters=max_iters, verbose=True)

    if em_factory.rank == 0:
        masked_on_host = genotype_file is not None and report_posterior
        reuse_pattern = genotype_file is None and em_factory.world == 1 and em_factory._pattern.packed.has_genes
        _write_reports(em_factory, outbase, alignment_file, group_file, report_group_counts, report_alignment_counts,
                       report_posterior, notes_t=gtcall_t, notes_g=gtcall_g,
                       unmasked=None if masked_on_host else aln_mat,
                       unmasked_pattern=em_factory._pattern if reuse_pattern else None)
        _write_bootstrap(em_factory, outbase, bootstrap, bootstrap_seed, multiread_model, pseudocount, tolerance, max_iters,
                         bootstrap_output, bootstrap_interval, notes_t=gtcall_t, notes_g=gtcall_g)
    logger.debug("Done")
