"""Seeded VCF inputs with declared ##FORMAT fields, shared by the FORMAT tests and tools/measure_vcf.py: an edge file covering the
record rules, and genotype lines with GT, DP, AD (Number=R), GQ and PL (Number=G) per sample, built from a pool of sample strings."""
from operator import itemgetter

import numpy as np

from vcf_inputs import CHROM, HEADER

FORMAT_HEADER = (b"##FORMAT=<ID=GT,Number=1,Type=String,Description=\"Genotype\">\n"
                 b"##FORMAT=<ID=DP,Number=1,Type=Integer,Description=\"Read depth\">\n"
                 b"##FORMAT=<ID=AD,Number=R,Type=Integer,Description=\"Allelic depths, \\\"ref,alt\\\"\">\n"
                 b"##FORMAT=<ID=GQ,Number=1,Type=Integer,Description=\"Genotype quality\">\n"
                 b"##FORMAT=<ID=PL,Number=G,Type=Integer,Description=\"Phred-scaled likelihoods\">\n"
                 b"##FORMAT=<ID=GL,Number=G,Type=Float,Description=\"Genotype likelihoods\">\n"
                 b"##FORMAT=<ID=HQ,Number=1,Type=Float,Description=\"Haplotype quality\">\n"
                 b"##FORMAT=<ID=FT,Number=1,Type=Character,Description=\"Filter\">\n")
FIVE = ["GT", "DP", "AD", "GQ", "PL"]
ALL = FIVE + ["GL", "HQ", "FT"]

# three samples; every record rule of DESIGN 3.11a on one line or another
EDGE_FMT = (HEADER + FORMAT_HEADER + CHROM + b"\tFORMAT\tNA1\tNA\"2\tS 3\n" +
            b"1\t100\trs1\tA\tT\t50\tPASS\tDP=14\tGT:DP:AD:GQ:PL:GL:HQ:FT\t0|1:12:5,7:99:0,30,300:-0.5,.,-2e1:1.5:x\t./.:.:.:.:.:.:.:.\t1/2:0:0,0:0:.,1,2:0,0,0:-0.0:.\n"
            b"1\t200\t.\tAC\t.\t.\t.\t.\tPL:GT:DP\t1,2,3:0/0:7\t.\t4,5,6:1|1\r\n"
            b"1\t300\t.\tG\tGA,GT\t9.5\tq10\tAC=1,2,3\tGT:AD\t0|1\t1|2:.,3,.\t.:.\n"
            b"chr2\t1\t.\tN\tA\t.\tPASS\t.\t.\t.\t.\t.\n"
            b"chr2\t5\t.\tN\tA\t.\tPASS\t.\tXX:GT:XX:DP\ta:0|0:b:-2147483648\tc:.|.\t::2147483647\n"
            b"chr2\t9\t.\tN\tA\t.\tPASS\t.\tGT:GQ:FT:HQ\t.:.:.:.\t0/1:.:y:1e10\t\n"
            b"chrX\t7\t.\tA\tC\t.\tPASS\t.\tGT:PL:GL\t0:.,.,.:.\t1:0:3\t0|0:+7,-7:1,2\n")


def format_text(n, n_samples=2504, seed=21) -> bytes:
    """Genotype lines with FORMAT GT:DP:AD:GQ:PL per sample (about 20 bytes each), every seventh line GT:PL:DP; about 1 % of the
    samples are './.', '.', or lack their trailing values or hold '.' values and leaves."""
    rng = np.random.default_rng(seed)
    pool0, pool1 = [], []
    for k in range(4096):
        g = [b"0|0", b"0|1", b"1|0", b"1|1", b"0/1"][k % 5]
        dp, a0, gq = int(rng.integers(0, 99)), int(rng.integers(0, 60)), int(rng.integers(0, 99))
        pl = b"%d,%d,%d" % (rng.integers(0, 9), rng.integers(0, 99), rng.integers(0, 999))
        full = b"%s:%d:%d,%d:%d:%s" % (g, dp, a0, dp - a0 if dp >= a0 else 0, gq, pl)
        if k % 97 == 5:
            full = b"./.:.:.:.:."
        elif k % 97 == 11:
            full = b"."
        elif k % 97 == 17:
            full = b"%s:%d" % (g, dp)
        elif k % 97 == 23:
            full = b"%s:%d:%d,.:.:.,3,." % (g, dp, a0)
        pool0.append(full)
        pool1.append(b"." if k % 97 == 11 else b"%s:%s:%d" % (g, pl, dp))
    samples = b"\t".join(b"HG%05d" % k for k in range(n_samples))
    pos = np.cumsum(rng.integers(1, 1000, n)) + 1
    picks = rng.integers(0, 4096, (n, n_samples))
    lines = []
    for i in range(n):
        pool, keys = (pool1, b"GT:PL:DP") if i % 7 == 3 else (pool0, b"GT:DP:AD:GQ:PL")
        body = b"\t".join(itemgetter(*picks[i])(pool)) if n_samples > 1 else pool[picks[i][0]]
        lines.append(b"22\t%d\t.\tA\tG\t%d\tPASS\tDP=%d;AF=0.%02d\t%s\t%s\n" % (pos[i], i % 99, i % 1000, i % 100, keys, body))
    return HEADER + FORMAT_HEADER + CHROM + b"\tFORMAT\t" + samples + b"\n" + b"".join(lines)
