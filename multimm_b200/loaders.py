"""Input ingestion: genomic tracks -> bead-space arrays (Cs, ms, ns, ds, chr_ends, chrom_idxs).

Independent numpy implementation of the behaviour of the reference's ``import_bed``
(utils.py:220-347) and ``import_mns_from_bedpe`` (utils.py:425-547), including the quirks the
model depends on (SURVEY appendix A, Q4-Q6): the two loaders use different resolutions; chrX/chrY
rows keep raw coordinates in genome-wide mode; loops use anchor midpoints, the mean count per
(m, n), lexicographic column order, clamping to N-1 and the n > m + 2 filter; ``ds`` is 1.0
everywhere when all counts are equal.  ``np.random.seed(seed)`` is consumed in the same order as
the reference, so seed-controlled shuffling / down-sampling / noise reproduce its arrays.
tests/golden/ holds outputs of the reference's own functions on the same files.
"""
from __future__ import annotations

import logging
import os

import numpy as np
import pandas as pd

logger = logging.getLogger(__name__)

# hg38 chromosome table (utils.py:40-122)
CHROM_NAMES = {i: f"chr{i + 1}" for i in range(22)}
CHROM_NAMES[22] = "chrX"
CHROM_NAMES[23] = "chrY"
_LENGTHS = (248387328, 242696752, 201105948, 193574945, 182045439, 172126628, 160567428, 146259331,
            150617247, 134758134, 135127769, 133324548, 113566686, 101161492, 99753195, 96330374,
            84276897, 80542538, 61707364, 66210255, 45090682, 51324926, 154259566, 62460029)
CHROM_LENGTHS = np.array(_LENGTHS, dtype=np.int64)
CHROM_SIZES = {CHROM_NAMES[i]: _LENGTHS[i] for i in range(24)}


BEAD_MASS = 16427.889  # amu, the one atom type of forcefields/ff.xml:5


def _minmax(a):
    a = np.nan_to_num(np.asarray(a, dtype=np.float64))
    return (a - a.min()) / (a.max() - a.min())


# chrom_strength = 1 - minmax(lengths chr1..chrY)  (utils.py:125-137): chr1 -> 0, chr21 -> 1
CHROM_STRENGTH = 1.0 - _minmax(CHROM_LENGTHS)


def _chrom_index(chrom: str) -> int:
    for k, v in CHROM_NAMES.items():
        if v == chrom or v == f"chr{chrom}":
            return k
    return 0


def _chrom_layout(chrom, shuffle, n_chroms):
    """chrom_idxs and cumulative genomic offsets, consuming np.random exactly like the reference."""
    if chrom is not None:
        idxs = np.array([_chrom_index(chrom)])
        ends = np.array([0, CHROM_SIZES[chrom]], dtype=np.int64)
    else:
        idxs = np.arange(n_chroms).astype(int)
        if shuffle:
            np.random.shuffle(idxs)
        ends = np.concatenate([[0], np.cumsum(CHROM_LENGTHS[idxs])]).astype(np.int64)
    return idxs, ends


def _label_value(label: str):
    if label.startswith("A.1") or label.startswith("A1"):
        return 2
    if label.startswith("A"):
        return 1
    if label.startswith("B.2") or label.startswith("B2"):
        return -2
    if label.startswith("B"):
        return -1
    return None


def import_bed(bed_file, N_beads, coords=None, chrom=None, save_path="", shuffle=False, seed=0, n_chroms=22,
               flip_prob=0.0, noise_strength=0.0):
    """Compartment track -> (Cs int[N], chr_ends int[C+1], chrom_idxs int[C])."""
    np.random.seed(seed)
    df = pd.read_csv(bed_file, header=None, sep="\t")
    if chrom is not None:
        df = df[(df[0] == chrom) & (df[1] > coords[0]) & (df[2] < coords[1])].reset_index(drop=True)
    idxs, ends = _chrom_layout(chrom, shuffle, n_chroms)
    names = df[0].to_numpy()
    start = df[1].to_numpy(dtype=np.int64).copy()
    stop = df[2].to_numpy(dtype=np.int64).copy()
    labels = df[3].to_numpy()
    if chrom is None:
        for count, ci in enumerate(idxs):
            sel = names == CHROM_NAMES[int(ci)]
            start[sel] += ends[count]
            stop[sel] += ends[count]
        resolution = int(ends[-1]) // N_beads
    else:
        resolution = (coords[1] - coords[0]) // N_beads
        start -= coords[0]
        stop -= coords[0]
    chr_ends = ends // resolution
    chr_ends[-1] = N_beads
    start //= resolution
    stop //= resolution
    comps = np.zeros(N_beads, dtype=float)
    for a, b, lab in zip(start, stop, labels):  # later rows overwrite earlier ones
        val = _label_value(lab)
        if val is not None:
            comps[a:b] = val
    if noise_strength > 0:
        noise = np.random.normal(0.0, noise_strength, size=N_beads)
        from scipy.ndimage import gaussian_filter1d

        comps = comps + gaussian_filter1d(noise, sigma=8)
    if flip_prob > 0:
        mask = np.random.rand(N_beads) < flip_prob
        mask &= comps != 0
        step = np.random.choice([-1, 1], size=N_beads)
        comps[mask] += step[mask]
        comps = np.clip(comps, -2, 2)
    comps = np.where(comps > 1.5, 2, np.where(comps > 0.2, 1, np.where(comps < -1.5, -2,
                     np.where(comps < -0.2, -1, 0)))).astype(int)
    if save_path is not None:
        meta = os.path.join(save_path, "metadata")
        if os.path.isdir(meta):
            np.save(os.path.join(meta, "chrom_lengths.npy"), chr_ends)
            np.save(os.path.join(meta, "compartments.npy"), comps)
            np.save(os.path.join(meta, "chrom_idxs.npy"), idxs)
    return comps, chr_ends.astype(int), idxs.astype(int)


def import_mns_from_bedpe(bedpe_file, N_beads, coords=None, chrom=None, threshold=0, min_loop_dist=2, path="",
                          down_prob=1.0, shuffle=False, seed=0, n_chroms=22, layout=None):
    """Loop track -> (ms int[L], ns int[L], ds float[L], chr_ends int[C+1], chrom_idxs int[C]).

    ``layout``: an optional dict that receives the bead-to-genome mapping this call used (it changes
    neither the return value nor the draws from numpy's random stream): ``resolution`` (bp per bead),
    ``ends`` (bp offset of every block in the concatenated coordinate), ``chr_ends``, ``chrom_idxs`` and
    ``start_bp`` / ``stop_bp`` (the modelled region, or 0 / None genome-wide).  Bead i of block k then sits
    at bp ``start_bp + i * resolution + resolution // 2 - ends[k]`` of chromosome ``chrom_idxs[k]``."""
    np.random.seed(seed)
    df = pd.read_csv(bedpe_file, header=None, sep="\t")
    idxs, ends = _chrom_layout(chrom, shuffle, n_chroms)
    df = loop_rows(df, chrom, coords).reset_index(drop=True)
    counts_raw = df[6].to_numpy(dtype=np.float64)
    ms, ns, resolution, chr_ends = loop_anchor_beads(df, idxs, ends, N_beads, chrom, coords)
    # mean count per (m, n); unique columns in lexicographic order, first occurrence wins
    pair = np.stack([ms, ns], axis=1)
    uniq, first, inv = np.unique(pair, axis=0, return_index=True, return_inverse=True)
    inv = inv.reshape(-1)
    mean = np.bincount(inv, weights=counts_raw) / np.bincount(inv)
    keep = mean > threshold
    ms, ns, cs = uniq[keep, 0].copy(), uniq[keep, 1].copy(), mean[keep]
    if cs.size == 0:
        raise ValueError("The region of interest does not include loops. Please try with longer modelling "
                         "region or increase the window around the gene.")
    ms[ms >= N_beads] = N_beads - 1
    ns[ns >= N_beads] = N_beads - 1
    sel = ns > ms + min_loop_dist
    ms, ns, cs = ms[sel], ns[sel], cs[sel]
    if cs.size == 0:  # the reference fails with an IndexError on cs[0] here (utils.py:520); say why instead
        raise ValueError("No loop spans more than min_loop_dist beads at this resolution. Please increase N_BEADS "
                         "or model a shorter region.")
    ds = 0.1 + 0.1 * _minmax_raw(1 / cs ** (2 / 3)) if not np.all(cs == cs[0]) else np.ones(len(ms))
    if down_prob < 1.0:
        pick = np.where(np.random.rand(len(ms)) < down_prob)[0]
        ms, ns, cs, ds = ms[pick], ns[pick], cs[pick], ds[pick]
    if path is not None:
        meta = os.path.join(path, "metadata")
        if os.path.isdir(meta):
            np.save(os.path.join(meta, "chrom_lengths.npy"), chr_ends)
            np.save(os.path.join(meta, "chrom_idxs.npy"), idxs)
            np.save(os.path.join(meta, "ms.npy"), ms)
            np.save(os.path.join(meta, "ns.npy"), ns)
            np.save(os.path.join(meta, "ds.npy"), ds)
    logger.info(f"Number of loops is {len(ms)}")
    if layout is not None:
        layout.update(resolution=int(resolution), ends=ends.astype(np.int64), chr_ends=chr_ends.astype(np.int64),
                      chrom_idxs=idxs.astype(np.int64), start_bp=int(coords[0]) if chrom is not None else 0,
                      stop_bp=int(coords[1]) if chrom is not None else None)
    return ms.astype(int), ns.astype(int), ds, chr_ends.astype(int), idxs.astype(int)


def loop_rows(df, chrom=None, coords=None):
    """The rows of a bedpe table (columns 0..6) that import_mns_from_bedpe reads, in file order and with the
    file's row index: all of them genome-wide; in a chromosome, region or gene run those whose first anchor is
    on ``chrom`` and whose four coordinates lie inside ``coords`` (the second anchor's chromosome is not
    checked)."""
    if chrom is None:
        return df
    return df[(df[0] == chrom) & (df[1] > coords[0]) & (df[2] < coords[1]) & (df[4] > coords[0])
              & (df[5] < coords[1])]


def loop_anchor_beads(df, idxs, ends, N_beads, chrom=None, coords=None):
    """The loader's bp -> bead arithmetic for every row of ``df`` (rows of loop_rows), with the chromosome
    layout ``idxs``, ``ends`` of _chrom_layout: (m, n, resolution, chr_ends), m and n the bead midpoints
    ``(a // res + b // res) // 2`` of the two anchors, not yet clamped to N - 1.  Genome-wide an anchor is
    offset by its chromosome's block start ``ends[k]``; an anchor on a chromosome that is not modelled keeps
    its raw coordinates (SURVEY appendix A, Q5).  In a region run every coordinate is taken relative to
    ``coords[0]``."""
    c = [df[k].to_numpy(dtype=np.int64).copy() for k in (1, 2, 4, 5)]
    if chrom is None:
        n0, n3 = df[0].to_numpy(), df[3].to_numpy()
        for count, ci in enumerate(idxs):
            name = CHROM_NAMES[int(ci)]
            s0, s3 = n0 == name, n3 == name
            c[0][s0] += ends[count]
            c[1][s0] += ends[count]
            c[2][s3] += ends[count]
            c[3][s3] += ends[count]
        resolution = int(np.max(c[3])) // N_beads
    else:
        resolution = (coords[1] - coords[0]) // N_beads
        for a in c:
            a -= coords[0]
    chr_ends = ends // resolution
    chr_ends[-1] = N_beads
    c = [a // resolution for a in c]
    return (c[0] + c[1]) // 2, (c[2] + c[3]) // 2, resolution, chr_ends


def _minmax_raw(x):
    return (x - x.min()) / (x.max() - x.min())


def get_gene_region(gene_tsv, gene_id=None, gene_name=None, window_size=200000):
    """Region around a gene (utils.py:688-710): (chrom, [start-w, end+w], [start, end])."""
    genes = pd.read_csv(gene_tsv, sep="\t")
    if gene_id is not None:
        col, key = "gene_id", gene_id
    elif gene_name is not None:
        col, key = "gene_name", gene_name
    else:
        raise ValueError("Either 'gene_id' or 'gene_name' must be provided.")
    hit = genes[genes[col] == key]
    if len(hit) == 0:
        what = "Gene ID" if col == "gene_id" else "Gene name"
        raise ValueError(f"{what} '{key}' not found in the provided TSV file.")
    chrom, start, end = hit["chromosome"].values[0], hit["start"].values[0], hit["end"].values[0]
    return chrom, [max(0, int(start - window_size)), int(end + window_size)], [start, end]
