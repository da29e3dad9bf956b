#!/usr/bin/env python
"""Writes a benchmark cohort (find_tfbs_b200/synth.py) as the reference's input FILES -- BGZF-compressed BCF2.2 + CSI index, FASTA + .fai,
BED files, HOCOMOCO-style PWM + threshold files -- so that the C++ driver (find-tfbs-b200) can be timed end to end on the same data
bench.py scores from arrays ("chromosome wall time" of BASELINE.json's metric).

    python scripts/make_cohort_files.py configs2            -> scratch_data/cfg2/   (2,504 samples, ~170k records, 401 PWMs)
    python scripts/make_cohort_files.py configs1            -> scratch_data/cfg1/
    python scripts/make_cohort_files.py configs2 0.05       -> scratch_data/cfg2_0.05/

The directory is git-ignored (hundreds of MB uncompressed); args.txt holds the driver's command line.  Without it, bench.py writes the
same files into a temporary directory (write_file_set) before it times the driver.
The BCF body is assembled with numpy (one int8 GT vector per record, 2 values per sample) and compressed member by member on all
cores; tests/file_writers.py is the readable per-record version of the same format and is used to cross-check this one."""
import os
import struct
import sys
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import file_writers as fw  # noqa: E402
from find_tfbs_b200 import synth  # noqa: E402

MEMBER = 0xff00


def bcf_body(chrom, contig_len, samples, pos, ref_len, alleles_of, bits):
    """Uncompressed BCF: header + one record per variant; bits[v, 2s + side] = the haplotype carries ALT."""
    text = ("##fileformat=VCFv4.2\n##FILTER=<ID=PASS,Description=\"All filters passed\">\n##contig=<ID=%s,length=%d>\n"
            "##FORMAT=<ID=GT,Number=1,Type=String,Description=\"Genotype\">\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t%s\n"
            % (chrom, contig_len, "\t".join(samples))).encode() + b"\0"
    head = b"BCF\2\2" + struct.pack("<I", len(text)) + text
    n, S = len(pos), len(samples)
    shared = []
    for v in range(n):
        ref, alt = alleles_of(v)
        sh = struct.pack("<iiiIII", 0, int(pos[v]), int(ref_len[v]), 0x7F800001, (2 << 16), (1 << 24) | S) + bytes([0x07]) + \
            fw._typed_str(ref) + fw._typed_str(alt) + bytes([0x00])
        shared.append(sh)
    l_indiv = 3 + 2 * S
    sizes = np.array([8 + len(sh) + l_indiv for sh in shared], dtype=np.int64)
    offs = np.concatenate([[0], np.cumsum(sizes)]) + len(head)
    out = np.zeros(int(offs[-1]), dtype=np.uint8)
    out[:len(head)] = np.frombuffer(head, dtype=np.uint8)
    for v in range(n):
        o = int(offs[v])
        sh = shared[v]
        out[o:o + 8] = np.frombuffer(struct.pack("<II", len(sh), l_indiv), dtype=np.uint8)
        out[o + 8:o + 8 + len(sh)] = np.frombuffer(sh, dtype=np.uint8)
        g = o + 8 + len(sh)
        out[g:g + 3] = (0x11, 1, 0x21)
    # genotypes: left = Unphased(allele) = (allele + 1) << 1, right = Phased(allele) = (allele + 1) << 1 | 1 (haplotype.rs:34-41 reads 4 / 5)
    step = max(1, (256 << 20) // max(1, 2 * S))
    for v0 in range(0, n, step):
        v1 = min(n, v0 + step)
        gt = np.empty((v1 - v0, 2 * S), dtype=np.uint8)
        gt[:, 0::2] = 2 + 2 * bits[v0:v1, 0::2]
        gt[:, 1::2] = 3 + 2 * bits[v0:v1, 1::2]
        starts = offs[v0:v1] + 8 + np.array([len(s) for s in shared[v0:v1]], dtype=np.int64) + 3
        idx = (starts[:, None] + np.arange(2 * S, dtype=np.int64)[None, :]).ravel()
        out[idx] = gt.ravel()
    return out, len(head), int(offs[-1])


def bgzf_member(data, level):
    co = zlib.compressobj(level, zlib.DEFLATED, -15)
    comp = co.compress(data) + co.flush()
    return (b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", len(comp) + 25) + comp +
            struct.pack("<II", zlib.crc32(data) & 0xFFFFFFFF, len(data)))


def write_bgzf_bcf(path, body, first_record, end, n_records, level=4):
    chunks = [bytes(body[i:i + MEMBER]) for i in range(0, len(body), MEMBER)]
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:
        members = list(ex.map(lambda c: bgzf_member(c, level), chunks))
    member_off, o = [], 0
    with open(path, "wb") as f:
        for m in members:
            member_off.append(o)
            f.write(m)
            o += len(m)
        member_off.append(o)
        f.write(bgzf_member(b"", level))

    def voff(byte):
        k = byte // MEMBER
        return (member_off[k] << 16) | (byte - k * MEMBER)

    # CSI (min_shift 14, depth 5): one bin holding one chunk = all records of the only contig, plus the pseudo-bin with the statistics
    idx = bytearray(b"CSI\1" + struct.pack("<iii", 14, 5, 0) + struct.pack("<i", 1))
    pseudo = ((1 << 18) - 1) // 7 + 1
    b, e = voff(first_record), voff(end)
    idx += struct.pack("<i", 2)
    idx += struct.pack("<IQi", 0, b, 1) + struct.pack("<QQ", b, e)
    idx += struct.pack("<IQi", pseudo, 0, 2) + struct.pack("<QQ", b, e) + struct.pack("<QQ", n_records, 0)
    idx += struct.pack("<Q", 0)
    with open(path + ".csi", "wb") as f:
        f.write(bgzf_member(bytes(idx), 6) + bgzf_member(b"", 6))


def write_file_set(pats, blk, out, rel):
    """Writes the file set of a synth cohort into directory `out`; returns the driver's arguments, naming the files under `rel`."""
    os.makedirs(out, exist_ok=True)
    m = blk.meta
    chrom = "chrS"
    fw.write_fasta(os.path.join(out, "genome.fa"), chrom, m["genome"].tobytes())
    beds = []
    for b, pm in enumerate(m["peak_map"]):
        p = os.path.join(out, "regions%d.bed" % (b + 1))
        fw.write_bed(p, chrom, pm)
        beds.append(os.path.join(rel, "regions%d.bed" % (b + 1)))
    fw.write_pwms(os.path.join(out, "pwms.txt"), os.path.join(out, "thr"), pats)
    S = blk.n_samples
    samples = ["S%05d" % i for i in range(S)]
    allele = m["allele"].tobytes()
    ro, rl, ao, al = m["var_ref_off"], m["var_ref_len"], m["var_alt_off"], m["var_alt_len"]
    bits = np.unpackbits(blk.carriers.view(np.uint8), axis=1, bitorder="little")[:len(m["var_pos"]), :2 * S]
    body, first, end = bcf_body(chrom, m["genome_len"], samples, m["var_pos"], rl,
                                lambda v: (allele[ro[v]:ro[v] + rl[v]].decode(), allele[ao[v]:ao[v] + al[v]].decode()), bits)
    write_bgzf_bcf(os.path.join(out, "cohort.bcf"), body, first, end, len(m["var_pos"]))
    names = [p["name"] for p in pats if p["direction"] == 0]
    args = ["--chromosome", chrom, "--input", os.path.join(rel, "cohort.bcf"), "--reference", os.path.join(rel, "genome.fa"), "--bed", ",".join(beds),
            "--pwm_names", ",".join(names), "--pwm_file", os.path.join(rel, "pwms.txt"), "--pwm_threshold_directory", os.path.join(rel, "thr"),
            "--pwm_threshold", "0.0001"]
    print("%s: %d samples, %d records, %d merged regions, BCF %.1f MB (%.1f MB inflated)" %
          (rel, S, len(m["var_pos"]), blk.n_regions, os.path.getsize(os.path.join(out, "cohort.bcf")) / 1e6, len(body) / 1e6))
    return args


def main():
    name = sys.argv[1] if len(sys.argv) > 1 else "configs2"
    scale = float(sys.argv[2]) if len(sys.argv) > 2 else 1.0
    if name == "configs2":
        pats, blk = synth.config3(scale=scale, seed=3)
        d = "cfg2"
    else:
        pats, blk = synth.config2(scale=scale, seed=2)
        d = "cfg1"
    if scale != 1.0:
        d += "_%g" % scale
    rel = os.path.join("scratch_data", d)
    out = os.path.join(ROOT, rel)
    args = write_file_set(pats, blk, out, rel)
    open(os.path.join(out, "args.txt"), "w").write(" ".join(args) + "\n")


if __name__ == "__main__":
    main()
