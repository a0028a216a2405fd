"""write_vcf(): the variants of a set of haplotypes as one VCF file, its lines merged and formatted on the GPU
(jlp_write_vcf; the format is defined in DESIGN.md section 11)."""
from __future__ import annotations

import ctypes as C
import datetime
import os

import numpy as np

from . import _lib
from .genome import Haplotypes
from .illumina import _single_integer, default_context
from .profiles import JackalopeError


def _err(par, what):
    raise JackalopeError("\nFor the `write_vcf` function in jackalope, argument `%s` must be %s." % (par, what))


def write_vcf(haps, out_prefix, compress=False, comp_method="bgzip", sample_matrix=None, overwrite=False, *, ctx=None,
              device=0, file_date=None, comp_engine="auto", n_threads=1, batch_bytes=None):
    """Write the haplotypes' variants to ``<out_prefix>.vcf`` (``.vcf.gz`` when compressed).  ``sample_matrix``: an
    ``n_samples x ploidy`` array of 0-based haplotype indices (samples ``sample1 .. sampleN``); None is one haploid
    sample per haplotype, named by the haplotype.  ``compress``: a logical or a level 1-9 (levels 1-6 are compressed on
    the GPU unless ``comp_engine="host"``, 7-9 by zlib on ``n_threads`` writer threads).  ``file_date`` (YYYYMMDD)
    defaults to today.  Returns the call's figures as a dict."""
    if not isinstance(haps, Haplotypes):
        _err("haps", "a \"haplotypes\" object")
    if not isinstance(out_prefix, str) or not out_prefix:
        _err("out_prefix", "a single, non-empty string")
    if not isinstance(compress, (bool, np.bool_)) and not _single_integer(compress, 1, 9):
        _err("compress", "a single logical or integer from 1 to 9")
    if comp_method not in ("gzip", "bgzip"):
        _err("comp_method", "\"gzip\" or \"bgzip\"")
    if not isinstance(overwrite, (bool, np.bool_)):
        _err("overwrite", "a single logical")
    if comp_engine not in ("auto", "host", "device"):
        _err("comp_engine", "\"auto\", \"host\" or \"device\"")
    if not _single_integer(n_threads, 1, 64):
        _err("n_threads", "a single integer from 1 to 64")
    if sample_matrix is None:
        S = np.arange(haps.n_haps(), dtype=np.uint64).reshape(-1, 1)
        names = list(haps.hap_names)
    else:
        try:
            a = np.asarray(sample_matrix)
        except ValueError:
            a = None
        if a is None or a.dtype == object or a.ndim != 2 or a.size == 0 or not np.issubdtype(a.dtype, np.integer):
            _err("sample_matrix", "NULL or a 2-dimensional matrix of integers")
        if (a < 0).any() or (a >= haps.n_haps()).any():
            _err("sample_matrix", "a matrix of haplotype indices from 0 to %d" % (haps.n_haps() - 1))
        S = np.ascontiguousarray(a, dtype=np.uint64)
        names = ["sample%d" % (i + 1) for i in range(S.shape[0])]
    for n in names:
        if any(ch in n for ch in "\t\r\n"):
            raise JackalopeError("\nFor the `write_vcf` function in jackalope, sample (haplotype) names cannot contain "
                                 "tabs or line breaks: %r" % n)
    for n in haps.reference.names:
        if any(ch.isspace() for ch in n):
            raise JackalopeError("\nFor the `write_vcf` function in jackalope, chromosome names cannot contain "
                                 "whitespace: %r" % n)
    if isinstance(compress, (bool, np.bool_)):
        compress = 6 if compress else 0
    compress = int(compress)
    path = os.path.expanduser(out_prefix) + (".vcf.gz" if compress else ".vcf")
    d = os.path.dirname(path)
    if d and not os.path.isdir(d):
        os.makedirs(d, exist_ok=True)
    if not overwrite and os.path.exists(path):
        raise JackalopeError("\nFile %s already exists." % path)
    if file_date is None:
        file_date = datetime.date.today().strftime("%Y%m%d")

    p = _lib.VcfParams()
    p.path = path.encode()
    p.n_samples, p.ploidy = S.shape
    p.sample_haps = S.ctypes.data_as(_lib.u64p)
    c_names = (C.c_char_p * len(names))(*[n.encode() for n in names])
    p.sample_names = c_names
    p.file_date = str(file_date).encode()
    p.compress, p.comp_method = compress, comp_method.encode()
    p.comp_engine = {"auto": 0, "host": 1, "device": 2}[comp_engine]
    p.n_threads = int(n_threads)
    p.batch_bytes = int(batch_bytes or 0)
    ctx = ctx or default_context(device)
    ctx.set_haplotypes(haps)
    st = _lib.VcfStats()
    ctx._check(ctx.lib.jlp_write_vcf(ctx.h, C.byref(p), C.byref(st)), "write_vcf")
    return st.as_dict()
