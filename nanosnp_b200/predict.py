"""Drop-in for the reference entry point PileupModel/predict.py (same CLI, same VCF text).

    python -m nanosnp_b200.predict -config CFG -model_path CKPT -data DIR -reference REF.fa -output OUT.vcf [-batch_size 1000]

`-data` is a directory of per-contig files: the reference's `.pd` text, or packed reads `.reads.npz` (then s1 runs on
the GPU too).  Records are produced per file in consecutive batches of `-batch_size` sites, because the reference's
record logic depends on batch composition (predict.py:106,119; SURVEY 8a P13); the per-batch text comes from the
native formatter nsnp_vcf_format_batch.  `--no_cuda` is refused: there is no CPU path.
"""
from __future__ import annotations

import argparse
import ctypes as C
import os
import sys

import numpy as np
import torch

from . import _lib
from .dataset import PredictDataset
from .model import LSTMNetwork
from .runner import COV_CHANNELS


def write_head(reference_index_file, fwriter):                     # predict.py:13-27
    fwriter.write("##fileformat=VCFv4.3\n")
    fwriter.write('##FILTER=<ID=PASS,Description="All filters passed">\n')
    fwriter.write('##FILTER=<ID=RefCall,Description="Reference call">\n')
    with open(reference_index_file) as f:
        for line in f:
            fields = line.strip().split()
            fwriter.write("##contig=<ID={},length={}>\n".format(fields[0], fields[1]))
    fwriter.write('##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">\n')
    fwriter.write('##FORMAT=<ID=GQ,Number=1,Type=Integer,Description="Genotype Quality">\n')
    fwriter.write('##FORMAT=<ID=DP,Number=1,Type=Integer,Description="Read Depth">\n')
    fwriter.write('##FORMAT=<ID=AF,Number=A,Type=Float,Description="Allele Frequency">\n')
    fwriter.write("#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tSample\n")


from .predict_io import ContigVcfAssembler, format_records, format_records_into, vcf_buffer_bytes  # noqa: E402,F401


def _read_inputs(testing_paths, only=None):
    """Yields (contig, reads or None, bam_reader or None, ref_id) per contig of the read inputs, one contig in memory at a time.
    BAM files are streamed (bam.BamReader); with a .bai the reads are left in the file and fetched region by region."""
    from .dataset import load_reads_npz
    for path in testing_paths:
        if path.endswith(".bam"):
            from .bam import BamReader
            reader = BamReader(path)
            if reader.has_index:
                for rid, (name, _) in enumerate(reader.refs):
                    if only is None or name in only:
                        yield name, None, reader, rid
            else:
                for rid, name, reads in reader.contigs(only):
                    yield name, reads, None, rid
        elif not path.endswith(".pd"):
            reads, contig, _ = load_reads_npz(path)
            if only is None or contig in only:
                yield contig, reads, None, -1


def _region_reads(reads, reader, rid, regions, targets=None):
    """Reads of each region: fetched through the .bai (with targets: only the reads near the unit's intervals), else the
    contiguous slice of the in-memory reads that can overlap the region's computed span."""
    from .reads import max_reference_span, slice_reads
    from .shard import fetch_ranges, read_range_for_region
    if reader is not None:
        if targets is not None:
            return [reader.fetch_ranges(rid, fetch_ranges(rg, iv)) for rg, iv in zip(regions, targets)]
        return [reader.fetch(rid, rg.start, rg.end) for rg in regions]
    span = max_reference_span(reads) + 1
    return [slice_reads(reads, *read_range_for_region(reads.pos, span, rg)) for rg in regions]


def predict(model: LSTMNetwork, testing_paths, reference_index_file, batch_size, output_file, device, reference=None, region_len=12_500_000,
            targets=None):
    """predict.py:37-195.  `.pd` text files: windows -> model -> records.  Read inputs (`.bam`, `.reads.npz`): the whole
    s1 + s2 path incl. the VCF text runs on the GPU region by region (caller.call_contig_text); under torchrun every rank
    computes and formats its LPT share of the regions and writes its own segments of the one output file
    (caller.write_sharded_vcf).
    targets: None (every position), or contig -> merged [k, 2] 0-based [start, end) intervals (targets.build_targets): only
    sites inside them are called, and the GPU computes only the pileup tiles near them.  The VCF is the one the reference
    writes from `.pd` files holding only those sites (batches are consecutive kept sites)."""
    import io
    from .caller import call_contig_text, write_sharded_vcf, _pinned
    from .dataset import load_fasta
    from .pipeline import PileupEngine
    from .runner import RegionRunner
    from .shard import assign_lpt, listed_tiles, plan_regions, plan_target_units
    from .targets import in_targets
    runner = None
    fasta = None

    def get_runner():
        nonlocal runner
        if runner is None:
            runner = RegionRunner(PileupEngine(device), model._forward(), records=True)
        return runner

    head = io.StringIO(); write_head(reference_index_file, head)
    header = head.getvalue().encode()
    import torch.distributed as dist
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    rank = dist.get_rank() if world > 1 else 0
    model.eval()
    if world > 1:
        # one process per GPU (torchrun): the contigs come from the reference index (every rank plans the same regions);
        # a rank only decodes the contigs / byte ranges of its own regions
        if any(f.endswith(".pd") for f in testing_paths):
            raise NotImplementedError("multi-GPU runs take read inputs (.bam / .reads.npz); .pd files hold ready-made windows")
        if reference is None:
            raise ValueError("read inputs need the reference FASTA")
        fasta = load_fasta(reference)
        with open(reference_index_file) as f:
            contigs = [(l.split()[0], int(l.split()[1])) for l in f if l.strip()]
        if targets is None:
            regions, unit_iv = plan_regions(contigs, region_len), None
            mine = assign_lpt(regions, world)[rank]
        else:
            regions, unit_iv = plan_target_units(contigs, targets, region_len)
            mine = assign_lpt(regions, world, [len(listed_tiles(rg, iv)) for rg, iv in zip(regions, unit_iv)])[rank]
        need = {regions[i].contig for i in mine}
        index_of = {name: ci for ci, (name, _) in enumerate(contigs)}
        recs = {}
        for contig, reads, reader, rid in _read_inputs(testing_paths, need):
            ci = index_of.get(contig)
            if ci is None:
                raise KeyError(f"contig {contig} is not in the reference index")
            idx = [i for i in mine if regions[i].contig_index == ci]
            if not idx:
                continue
            rgs = [regions[i] for i in idx]
            ivs = None if unit_iv is None else [unit_iv[i] for i in idx]
            host = [_pinned(r) for r in _region_reads(reads, reader, rid, rgs, ivs)]
            ref_dev = torch.from_numpy(np.ascontiguousarray(fasta[contig])).to(device)
            r = get_runner()
            for k, (i, rg, hr) in enumerate(zip(idx, rgs, host)):
                out = r.run_device(r.upload(hr), ref_dev, rg, targets=None if ivs is None else ivs[k])
                recs[i] = out.rec.clone()                    # records stay on this GPU until the text is made
        for i in mine:
            recs.setdefault(i, torch.zeros((0, 32), dtype=torch.uint8, device=device))
        write_sharded_vcf(output_file, header, contigs, regions, recs, batch_size, device)
        model._forward().reevaluated()                          # f16x1: raises if a region had more low-margin sites than are re-run
        return

    with open(output_file, "wb") as fwriter:
        fwriter.write(header)
        for testing_file in testing_paths:
            if testing_file.endswith(".pd"):
                dataset = PredictDataset(datapath=testing_file, reference=reference, device=device)
                if len(dataset) == 0:
                    continue
                names = dataset.contig_names
                if any(nm != names[0] for nm in names):
                    raise NotImplementedError("one predict-data file must hold one contig (as make_predict_data.sh writes them)")
                if targets is not None:                       # POS is 1-based
                    keep = in_targets(np.asarray(dataset.positions, np.int64) - 1, targets.get(names[0]))
                    if not keep.any():
                        continue
                    dataset.position_matrix = np.ascontiguousarray(dataset.position_matrix[keep])
                    dataset.positions = np.asarray(dataset.positions)[keep]
                    dataset.reference_bases = np.asarray(dataset.reference_bases)[keep]
                x = torch.from_numpy(dataset.position_matrix).to(device)
                gt, zy = model.predict(x)
                cov8 = x[:, 16, COV_CHANNELS].to(torch.float32)
                fwriter.write(format_records(names[0], dataset.positions, dataset.reference_bases, gt.cpu().numpy(), zy.cpu().numpy(),
                                             cov8.cpu().numpy(), batch_size))
        read_paths = [f for f in testing_paths if not f.endswith(".pd")]
        if read_paths:
            if reference is None:
                raise ValueError("read inputs need the reference FASTA")
            fasta = load_fasta(reference)
            for contig, reads, reader, rid in _read_inputs(read_paths, None if targets is None else set(targets)):
                if contig not in fasta:
                    if reader is not None:
                        continue                              # an indexed BAM lists every @SQ; only contigs of the FASTA are called
                    raise KeyError(f"contig {contig} is not in the reference")
                if targets is None:
                    regions, unit_iv = plan_regions([(contig, len(fasta[contig]))], region_len), None
                else:
                    regions, unit_iv = plan_target_units([(contig, len(fasta[contig]))], targets, region_len)
                call_contig_text(get_runner(), reads, fasta[contig], contig, fwriter, batch_size, region_len, regions,
                                 _region_reads(reads, reader, rid, regions, unit_iv), unit_iv)
        model._forward().reevaluated()                          # f16x1: raises if a region had more low-margin sites than are re-run


def main(argv=None):
    parser = argparse.ArgumentParser()
    parser.add_argument("-config", type=str, required=True, help="path to config file")
    parser.add_argument("-model_path", required=True, help="path to trained model")
    parser.add_argument("-data", required=True, help="directory of per-contig files (.pd text, .reads.npz, .bam) or one such file")
    parser.add_argument("-reference", required=True, help="path to reference file")
    parser.add_argument("-output", required=True, help="output vcf file")
    parser.add_argument("-batch_size", type=int, default=1000, help="batch size")
    parser.add_argument("--no_cuda", action="store_true", help="refused: the B200 path has no CPU fallback")
    parser.add_argument("--precision", default="f16x3", choices=["fp32", "f16x3", "f16x1"],
                        help="f16x1: single-pass tensor-core LSTM, low-margin sites re-evaluated in f16x3 (same calls, QUAL may move by ~0.06)")
    parser.add_argument("--region_len", type=int, default=12_500_000, help="positions per GPU work unit (read inputs)")
    parser.add_argument("--bed", default=None, help="call only inside these intervals (BED: 0-based, half-open; first three fields)")
    parser.add_argument("--region", action="append", default=[],
                        help="call only inside CTG or CTG:START-END (1-based, inclusive); repeatable, combines with --bed")
    opt = parser.parse_args(argv)
    if opt.no_cuda:
        raise SystemExit("nanosnp_b200.predict: --no_cuda is not supported (no CPU fallback); use the reference's predict.py on CPU")
    import yaml
    from .utils import AttrDict
    device = torch.device("cuda")
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:              # torchrun: one process per GPU, NCCL only gathers the call lists
        import torch.distributed as dist
        local = int(os.environ.get("LOCAL_RANK", "0")) % max(1, torch.cuda.device_count())
        torch.cuda.set_device(local)
        device = torch.device("cuda", local)
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        backend = os.environ.get("NSNP_DIST_BACKEND", "nccl")       # gloo: several ranks may share one GPU (tests)
        if backend == "nccl":
            dist.init_process_group("nccl", device_id=device)
        else:
            dist.init_process_group(backend)
    config = AttrDict(yaml.load(open(opt.config), Loader=yaml.FullLoader))
    pred_model = LSTMNetwork(config.model, precision=opt.precision).to(device)
    if opt.model_path.endswith(".npz"):
        z = np.load(opt.model_path)
        checkpoint = {"encoder": {k[8:]: z[k] for k in z.files if k.startswith("encoder.")},
                      "forward_layer": {k[14:]: z[k] for k in z.files if k.startswith("forward_layer.")}}
    else:
        checkpoint = torch.load(opt.model_path, map_location="cpu")
    pred_model.encoder.load_state_dict(checkpoint["encoder"])
    pred_model.forward_layer.load_state_dict(checkpoint["forward_layer"])
    if os.path.isfile(opt.data):
        testing_paths = [opt.data]                      # a single BAM / .reads.npz / .pd
    else:
        testing_paths = sorted(opt.data + "/" + f for f in os.listdir(opt.data) if f.endswith((".pd", ".reads.npz", ".bam")))
    assert os.path.exists(opt.reference + ".fai"), "reference index file does not exist."
    targets = None
    if opt.bed is not None or opt.region:
        from .targets import build_targets
        with open(opt.reference + ".fai") as f:
            contigs = [(l.split()[0], int(l.split()[1])) for l in f if l.strip()]
        quiet = int(os.environ.get("RANK", "0")) != 0                   # report skipped intervals once, not once per rank
        targets = build_targets(contigs, opt.bed, opt.region, report=None if quiet else sys.stderr)
    predict(pred_model, testing_paths, opt.reference + ".fai", opt.batch_size, opt.output, device, reference=opt.reference,
            region_len=opt.region_len, targets=targets)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
