"""Seeded VCF inputs shared by the VCF tests and tools/measure_vcf.py: an edge file, sites-only lines with many INFO keys and a
VEP-like CSQ string, and genotype lines with thousands of samples; BGZF members compressed on a thread pool."""
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from oracle.fastq_write_oracle import BGZF_BLOCK, BGZF_EOF, bgzf_bytes, bgzf_member

HEADER = (b"##fileformat=VCFv4.3\n"
          b"##FILTER=<ID=PASS,Description=\"All filters passed\">\n"
          b"##INFO=<ID=DP,Number=1,Type=Integer,Description=\"Total depth, as in \\\"DP=\\\">\">\n"
          b"##INFO=<ID=AF,Number=A,Type=Float,Description=\"Allele frequency\">\n"
          b"##INFO=<ID=DB,Number=0,Type=Flag,Description=\"dbSNP membership\">\n"
          b"##INFO=<ID=CSQ,Number=.,Type=String,Description=\"Consequence annotations: Allele|Consequence|Gene\">\n"
          b"##INFO=<ID=END,Number=1,Type=Integer,Description=\"End position\">\n"
          b"##INFO=<ID=AC,Number=R,Type=Integer,Description=\"Allele counts\">\n"
          b"##INFO=<ID=GL,Number=G,Type=Float,Description=\"Genotype likelihoods\">\n"
          b"##INFO=<ID=NS,Number=2,Type=Integer,Description=\"Two numbers\">\n"
          b"##INFO=<ID=TC,Number=1,Type=Character,Description=\"A character\">\n"
          b"##INFO=<ID=SVTYPE,Number=1,Type=String,Description=\"Type of structural variant\">\n"
          b"##INFO=<ID=H2,Number=0,Type=Flag,Description=\"HapMap2 membership\">\n"
          b"##INFO=<ID=MQ,Number=1,Type=Float,Description=\"Mapping quality\">\n")
CHROM = b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO"

EDGE = (HEADER + CHROM + b"\tFORMAT\tS1\tS2\n" +
        b"1\t100\trs1\tA\tT\t50\tPASS\tDP=14;AF=0.5;DB;CSQ=T|missense|G1,T|synonymous|G2;AC=3,1;MQ=60.25\tGT\t0|1\t1|1\n"
        b"1\t200\t.\tAC\t.\t.\t.\t.\r\n"
        b"1\t300\t.\tG\tGA,GT\t9.5e1\tq10;s50\tAF=.,0.25;AC=.,1,.;GL=-1.5,.,-0.5,0,1e-3,.;NS=1,2;TC=x;H2\n"
        b"chr2\t1\tid;2\tN\t<DEL>\t.\tPASS\tEND=1000;SVTYPE=DEL;CSQ=.;DB;XX=unknown;FOO\r\n"
        b"chr2\t5000\t.\tACGT\tA\t0\tPASS\tDP=.;AF=1e10;CSQ=a,,b|c;;;UNDECLARED=1,2\n"
        b"chrX\t2147483647\t.\tt\tc\t1.5\tPASS\tEND=2147483647;DP=-2147483648;SVTYPE=;GL=1,2,3\n"
        b"chrX\t7\t.\tA\tC\t.\tPASS\tDP=+7;TC=.;MQ=-0.0")


def bgzf_parallel(text: bytes, level=1) -> bytes:
    if len(text) <= (8 << 20):
        return bgzf_bytes(text, level)
    with ThreadPoolExecutor(16) as ex:
        members = list(ex.map(lambda i: bgzf_member(text[i:i + BGZF_BLOCK], level), range(0, len(text), BGZF_BLOCK)))
    return b"".join(members) + BGZF_EOF


def _info_keys(n_extra):
    return b"".join(b"##INFO=<ID=K%d,Number=1,Type=Integer,Description=\"extra key %d\">\n" % (k, k) for k in range(n_extra))


def sites_text(n, seed=11, n_extra=24, csq_lo=500, csq_hi=2000) -> bytes:
    """Sites-only lines: 8 declared keys plus n_extra integer keys per line and a CSQ list of csq_lo..csq_hi bytes."""
    rng = np.random.default_rng(seed)
    pos = np.cumsum(rng.integers(1, 200, n)) % 2000000000 + 1
    dp = rng.integers(0, 500, n)
    af = rng.integers(1, 1000, n)
    ext = rng.integers(0, 100000, (n, n_extra))
    csq_len = rng.integers(csq_lo, csq_hi + 1, n)
    alphabet = np.frombuffer(b"ACGTacgt|_-:0123456789", np.uint8)
    pool = alphabet[rng.integers(0, len(alphabet), csq_hi * 64)].tobytes()
    offs = rng.integers(0, csq_hi * 63, n)
    bases = [b"A", b"C", b"G", b"T"]
    lines = []
    for i in range(n):
        c = pool[offs[i]:offs[i] + csq_len[i]]
        c = c[:60] + b"," + c[61:200] + b"," + c[201:] if len(c) > 210 else c
        ext_s = b";".join(b"K%d=%d" % (k, ext[i, k]) for k in range(n_extra))
        lines.append(b"%d\t%d\trs%d\t%s\t%s\t%d.5\tPASS\tDP=%d;AF=0.%03d;%sCSQ=%s;AC=%d,%d;MQ=%d.25;%s\n" % (
            1 + i % 22, pos[i], i, bases[i % 4], bases[(i + 1) % 4], dp[i] % 100, dp[i], af[i], b"DB;" if i % 3 == 0 else b"",
            c, dp[i], af[i], dp[i] % 61, ext_s))
    return HEADER + _info_keys(n_extra) + CHROM + b"\n" + b"".join(lines)


def genotypes_text(n, n_samples=2504, seed=12) -> bytes:
    """Lines with FORMAT GT and n_samples genotypes (about 4 bytes each)."""
    rng = np.random.default_rng(seed)
    gts = np.frombuffer(b"0|0\t0|1\t1|0\t1|1\t", np.uint8).reshape(4, 4)
    samples = b"\t".join(b"S%d" % k for k in range(n_samples))
    pos = np.cumsum(rng.integers(1, 1000, n)) + 1
    lines = []
    for i in range(n):
        g = gts[rng.integers(0, 4, n_samples)].tobytes()[:-1]
        lines.append(b"22\t%d\t.\tA\tG\t%d\tPASS\tDP=%d;AF=0.%02d;NS=%d,%d\tGT\t%s\n" % (pos[i], i % 99, i % 1000, i % 100, i, 2 * i, g))
    return HEADER + CHROM + b"\tFORMAT\t" + samples + b"\n" + b"".join(lines)
