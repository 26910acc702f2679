"""baf feature-counting configuration (fields / defaults of xcltk/baf/fc/config.py:8-164)."""

import sys

from ...config import APP


class DefaultConfig(object):
    DEBUG = 0
    CELL_TAG = "CB"
    UMI_TAG = "UB"
    UMI_TAG_BC = "UB"
    NPROC = 1
    MIN_COUNT = 1
    MIN_MAF = 0
    OUTPUT_ALL_REG = False
    NO_DUP_HAP = True
    MIN_MAPQ = 20
    MIN_LEN = 30
    INCL_FLAG = 0
    EXCL_FLAG_UMI = 772
    EXCL_FLAG_XUMI = 1796
    NO_ORPHAN = True


class Config(object):
    _SHOW = [
        ("sam_fn", "sam_file", "%s"), ("sam_list_fn", "sam_list_file", "%s"),
        ("barcode_fn", "barcode_file", "%s"), ("sample_id_str", "sample_id_str", "%s"),
        ("sample_id_fn", "sample_id_file", "%s"), ("region_fn", "region_file", "%s"),
        ("snp_fn", "snp_file", "%s"), ("out_dir", "out_dir", "%s"), ("debug", "debug_level", "%d"), None,
        ("cellsnp_dir", "cellsnp_dir", "%s"), ("ref_cell_fn", "ref_cell_fn", "%s"),
        ("phase_from_reads", "phase_from_reads", "%s"), ("cell_tag", "cell_tag", "%s"), ("umi_tag", "umi_tag", "%s"),
        ("nproc", "number_of_processes", "%d"), ("min_count", "min_count", "%d"),
        ("min_maf", "min_maf", "%f"), ("output_all_reg", "output_all_reg", "%s"),
        ("no_dup_hap", "no_dup_hap", "%s"), None,
        ("min_mapq", "min_mapq", "%d"), ("min_len", "min_len", "%d"),
        ("incl_flag", "include_flag", "%d"), ("excl_flag", "exclude_flag", "%d"),
        ("no_orphan", "no_orphan", "%s"), None,
        ("#sam_fn_list", "#BAMs", "%d"), ("#barcodes", "#barcodes", "%d"),
        ("#sample_ids", "#sample IDs", "%d"), ("#reg_list", "#regions", "%d"),
        ("#snp_set", "#snps", "%d"), ("!snp_adata", "shape of snp adata", "%s"),
        ("#ref_cells", "#reference cells", "%d"), None,
        ("out_region_fn", "output_region_file", "%s"), ("out_sample_fn", "output_sample_file", "%s"),
        ("out_ad_fn", "output_ad_file", "%s"), ("out_dp_fn", "output_dp_file", "%s"),
        ("out_oth_fn", "output_oth_file", "%s"), None,
        ("rlp_min_len", "rlp_min_len", "%d"), ("rlp_min_n_snps", "rlp_min_n_snps", "%d"),
        ("rlp_min_gap", "rlp_min_gap", "%d"), None,
    ]

    def __init__(self):
        d = self.defaults = DefaultConfig()
        self.argv = None
        self.sam_fn = self.sam_list_fn = self.barcode_fn = None
        self.sample_id_str = self.sample_id_fn = None
        self.region_fn = self.snp_fn = self.out_dir = None
        self.debug = d.DEBUG
        self.cellsnp_dir = self.ref_cell_fn = None
        self.phase_from_reads = False      # local phasing from the call's own reads instead of cellsnp_dir
        self.cell_tag, self.umi_tag = d.CELL_TAG, d.UMI_TAG
        self.nproc = d.NPROC
        self.min_count, self.min_maf = d.MIN_COUNT, d.MIN_MAF
        self.output_all_reg, self.no_dup_hap = d.OUTPUT_ALL_REG, d.NO_DUP_HAP
        self.min_mapq, self.min_len = d.MIN_MAPQ, d.MIN_LEN
        self.incl_flag, self.excl_flag = d.INCL_FLAG, -1
        self.no_orphan = d.NO_ORPHAN
        # derived
        self.barcodes = self.sample_ids = self.reg_list = self.snp_set = None
        self.sam_fn_list = self.samples = None
        self.snp_adata = self.ref_cells = None
        # internal
        self.out_prefix = APP + "."
        self.out_region_fn = self.out_sample_fn = None
        self.out_ad_fn = self.out_dp_fn = self.out_oth_fn = None
        # region-wise local phasing thresholds (host pre-step, config.py:66-68)
        self.rlp_min_len = 50000
        self.rlp_min_n_snps = 2
        self.rlp_min_gap = 50000

    def show(self, fp=None, prefix=""):
        fp = fp or sys.stderr
        lines = [prefix]
        for item in self._SHOW:
            if item is None:
                lines.append(prefix)
                continue
            attr, label, fmt = item
            if attr.startswith("#"):
                v = getattr(self, attr[1:])
                v = (v.get_n() if hasattr(v, "get_n") else len(v)) if v is not None else -1
            elif attr.startswith("!"):
                v = getattr(self, attr[1:])
                v = str(v.shape) if v is not None else "None"
            else:
                v = getattr(self, attr)
            lines.append(("%s%s = " + fmt) % (prefix, label, v))
        fp.write("\n".join(lines) + "\n")

    def use_barcodes(self):
        return self.cell_tag is not None

    def use_local_phasing(self):
        return self.cellsnp_dir is not None or self.phase_from_reads

    def use_umi(self):
        return self.umi_tag is not None
