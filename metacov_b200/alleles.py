"""Metrics derived from the allele statistics of a region (``AlignmentFile.allele_stats``,
``CoverageEngine.allele_stats``): the one place the CLI and the tests take them from."""
import numpy as np

DERIVED = ("breadth", "con_ani", "depth", "pi", "pop_ani", "snv_per_kbp")


def _ratio(num, den):
    num = np.asarray(num, dtype=np.float64)
    den = np.asarray(den, dtype=np.float64)
    out = np.full(np.broadcast(num, den).shape, np.nan)
    np.divide(num, den, out=out, where=den != 0)
    return out


def derive(stats):
    """{name: float64 array (or 0-d array for one record)}: breadth = covered / length, depth = depth_sum / length,
    pi = pi_sum / covered, snv_per_kbp = 1000 snv / covered, con_ani = 1 - sub / ref_covered,
    pop_ani = 1 - popsub / ref_covered.  A division by zero gives NaN."""
    s = stats
    return {
        "breadth": _ratio(s["covered"], s["length"]),
        "depth": _ratio(s["depth_sum"], s["length"]),
        "pi": _ratio(s["pi_sum"], s["covered"]),
        "snv_per_kbp": _ratio(1000.0 * np.asarray(s["snv"], dtype=np.float64), s["covered"]),
        "con_ani": 1.0 - _ratio(s["sub"], s["ref_covered"]),
        "pop_ani": 1.0 - _ratio(s["popsub"], s["ref_covered"]),
    }


COMPARE_DERIVED = ("con_ani", "percent_compared", "pop_ani")


def derive_compare(stats):
    """{name: float64 array} of the pair records of ``compare`` / ``CoverageEngine.compare_stats``:
    con_ani = 1 - con_snp / compared, pop_ani = 1 - pop_snp / compared, percent_compared = compared / length.  A
    division by zero gives NaN."""
    s = stats
    return {
        "con_ani": 1.0 - _ratio(s["con_snp"], s["compared"]),
        "percent_compared": _ratio(s["compared"], s["length"]),
        "pop_ani": 1.0 - _ratio(s["pop_snp"], s["compared"]),
    }


LINKAGE_DERIVED = ("distance", "r2", "d_prime")


def derive_linkage(pairs):
    """{name: float64 array} of the pair records of ``AlignmentFile.linkage`` / ``CoverageEngine.linkage``, with fixed
    allele calls (upper case the major allele) and total = n_AB + n_Ab + n_aB + n_ab: p_A = (n_AB + n_Ab) / total,
    p_B = (n_AB + n_aB) / total, D = n_AB / total - p_A p_B, r2 = D^2 / (p_A (1 - p_A) p_B (1 - p_B)) and
    d_prime = |D| / D_max, D_max = min(p_A (1 - p_B), (1 - p_A) p_B) for D > 0, else min(p_A p_B, (1 - p_A)(1 - p_B));
    distance = pos_b - pos_a.  These are inStrain's definitions of r2 and D', without its rarefied columns.  A division
    by zero gives NaN."""
    s = pairs
    ab, a_b, ab_, ab2 = (np.asarray(s[k], dtype=np.float64) for k in ("n_AB", "n_Ab", "n_aB", "n_ab"))
    total = ab + a_b + ab_ + ab2
    p_a = _ratio(ab + a_b, total)
    p_b = _ratio(ab + ab_, total)
    d = _ratio(ab, total) - p_a * p_b
    d_max = np.where(d > 0, np.minimum(p_a * (1.0 - p_b), (1.0 - p_a) * p_b), np.minimum(p_a * p_b, (1.0 - p_a) * (1.0 - p_b)))
    return {
        "distance": np.asarray(s["pos_b"], dtype=np.float64) - np.asarray(s["pos_a"], dtype=np.float64),
        "r2": _ratio(d * d, p_a * (1.0 - p_a) * p_b * (1.0 - p_b)),
        "d_prime": _ratio(np.abs(d), d_max),
    }


GENE_DERIVED = ("N_sites", "S_sites", "pN", "pS", "pn_ps", "dN", "dS", "dn_ds")


def derive_genes(records):
    """{name: float64 array} of the gene records of ``AlignmentFile.gene_stats`` / ``CoverageEngine.gene_stats``:
    N_sites = n_sites3 / 3, S_sites = s_sites3 / 3, pN = snv_n / N_sites, pS = snv_s / S_sites, pn_ps = pN / pS,
    dN = sub_n / N_sites, dS = sub_s / S_sites, dn_ds = dN / dS; no Jukes-Cantor correction.  A division by zero gives
    NaN."""
    s = records
    n_sites = np.asarray(s["n_sites3"], dtype=np.float64) / 3.0
    s_sites = np.asarray(s["s_sites3"], dtype=np.float64) / 3.0
    p_n, p_s = _ratio(s["snv_n"], n_sites), _ratio(s["snv_s"], s_sites)
    d_n, d_s = _ratio(s["sub_n"], n_sites), _ratio(s["sub_s"], s_sites)
    return {"N_sites": n_sites, "S_sites": s_sites, "pN": p_n, "pS": p_s, "pn_ps": _ratio(p_n, p_s),
            "dN": d_n, "dS": d_s, "dn_ds": _ratio(d_n, d_s)}
