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
