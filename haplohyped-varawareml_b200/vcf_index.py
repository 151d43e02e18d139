"""vcf_index FILE [--csi] [--min-shift 14] [--device 0] [--force]: write FILE.tbi (or FILE.csi) of a bgzipped VCF, or
FILE.csi of a BGZF BCF, built on the GPU -- what `tabix -p vcf`, `tabix -C -p vcf` and `bcftools index` write.  An existing
index is kept unless --force is given."""
import os
import sys

import click

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


@click.command()
@click.argument("file", type=click.Path(exists=True, dir_okay=False))
@click.option("--csi", is_flag=True, help="Write a CSI index (always for a .bcf).")
@click.option("--min-shift", default=14, show_default=True, help="CSI: log2 of the smallest bin.")
@click.option("--device", default=0, show_default=True, help="CUDA device ordinal.")
@click.option("--force", is_flag=True, help="Overwrite an existing index.")
def main(file, csi, min_shift, device, force):
    from haplohyped_varawareml_b200 import capi
    fmt = "csi" if csi or file.endswith(".bcf") else "tbi"
    out = file + "." + fmt
    if os.path.exists(out) and not force:
        raise click.ClickException("%s exists: use --force to overwrite it" % out)
    try:
        capi.index_file(file, fmt, min_shift, device)
    except capi.HaploError as e:
        raise click.ClickException(str(e))
    click.echo(out)


if __name__ == "__main__":
    main()
