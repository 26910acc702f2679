"""basefc configuration (field names and defaults of xcltk/rdr/fc/config.py:5-111)."""

import sys


class DefaultConfig(object):
    DEBUG = 0
    CELL_TAG = "CB"
    UMI_TAG = "UB"
    UMI_TAG_BC = "UB"          # default UMI tag for 10x data
    NPROC = 1
    OUTPUT_ALL_REG = True
    MIN_MAPQ = 20
    MIN_LEN = 30
    MIN_INCLUDE = 0.9
    INCL_FLAG = 0
    EXCL_FLAG_UMI = 772        # UNMAP | SECONDARY | QCFAIL
    EXCL_FLAG_XUMI = 1796      # ... | DUP
    NO_ORPHAN = True


class Config(object):
    # (attribute, label, printf format) in the order the reference prints them; None = blank line
    _SHOW = [
        ("sam_fn", "sam_file", "%s"), ("sam_list_fn", "sam_list_file", "%s"),
        ("barcode_fn", "barcode_file", "%s"), ("sample_id_str", "sample_id_str", "%s"),
        ("sample_id_fn", "sample_id_file", "%s"), ("region_fn", "region_file", "%s"),
        ("out_dir", "out_dir", "%s"), ("debug", "debug_level", "%d"), None,
        ("cell_tag", "cell_tag", "%s"), ("umi_tag", "umi_tag", "%s"),
        ("nproc", "number_of_processes", "%d"), ("output_all_reg", "output_all_reg", "%s"), None,
        ("min_mapq", "min_mapq", "%d"), ("min_len", "min_len", "%d"),
        ("min_include", "min_include", "%f"), ("incl_flag", "include_flag", "%d"),
        ("excl_flag", "exclude_flag", "%d"), ("no_orphan", "no_orphan", "%s"), None,
        ("#sam_fn_list", "number_of_BAMs", "%d"), ("#barcodes", "number_of_barcodes", "%d"),
        ("#sample_ids", "number_of_sample_IDs", "%d"), ("#reg_list", "number_of_regions", "%d"), None,
        ("out_region_fn", "output_region_file", "%s"), ("out_sample_fn", "output_sample_file", "%s"),
        ("out_mtx_fn", "output_mtx_file", "%s"), None,
    ]

    def __init__(self):
        d = self.defaults = DefaultConfig()
        self.argv = None
        self.sam_fn = self.sam_list_fn = self.barcode_fn = None
        self.sample_id_str = self.sample_id_fn = self.region_fn = self.out_dir = None
        self.debug = d.DEBUG
        self.cell_tag, self.umi_tag = d.CELL_TAG, d.UMI_TAG
        self.nproc = d.NPROC
        self.output_all_reg = d.OUTPUT_ALL_REG
        self.min_mapq, self.min_len, self.min_include = d.MIN_MAPQ, d.MIN_LEN, d.MIN_INCLUDE
        self.incl_flag, self.excl_flag = d.INCL_FLAG, -1
        self.no_orphan = d.NO_ORPHAN
        self.barcodes = self.sample_ids = self.reg_list = None
        self.sam_fn_list = self.samples = None
        self.out_prefix = ""
        self.out_region_fn = self.out_sample_fn = self.out_mtx_fn = None
        # B200 additions (not in the reference): GPUs to shard over, host decode threads
        self.n_gpus = None
        self.devices = None
        # --summary: also write summary.tsv (the table is left in summary_table)
        self.summary = False
        self.summary_table = None

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
                v = len(v) if v is not None else -1
            else:
                v = getattr(self, attr)
            lines.append(("%s%s = " + fmt) % (prefix, label, v))
        fp.write("\n".join(lines) + "\n")

    def use_barcodes(self):
        return self.cell_tag is not None

    def use_umi(self):
        return self.umi_tag is not None
