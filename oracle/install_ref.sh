#!/bin/bash
# Installs the UNMODIFIED reference package (torch_geometric 2.9.0, pure Python) into oracle/_ref (git-ignored) from a
# checkout of pyg-team/pytorch_geometric given as $1 or $B200MP_REFERENCE_SRC.  The CPU arm of bench.py and the
# plug-in tests import it from there.  Nothing is compiled: the package directory is copied with default file modes
# (the source may be read-only) and then compared file by file with the source.
set -e
ROOT="$(cd "$(dirname "$0")/.." && pwd)"
SRC=${1:-$B200MP_REFERENCE_SRC}
[ -n "$SRC" ] && [ -d "$SRC/torch_geometric" ] || { echo "no reference checkout given (B200MP_REFERENCE_SRC)"; exit 0; }
DEST="$ROOT/oracle/_ref"
TMP="$DEST.tmp.$$"
trap 'rm -rf "$TMP"' EXIT
rm -rf "$TMP"
mkdir -p "$TMP"
cp -r --no-preserve=mode "$SRC/torch_geometric" "$TMP/"
# every file of the installed package must equal the reference's
(cd "$SRC" && find torch_geometric -type f \( -name '*.py' -o -name '*.jinja' \) | sort | while read -r f; do
    cmp -s "$f" "$TMP/$f" || echo "DIFF $f"; done) > "$TMP.diff"
if [ -s "$TMP.diff" ]; then cat "$TMP.diff"; rm -f "$TMP.diff"; echo "installed package differs from the reference"; exit 1; fi
rm -f "$TMP.diff"
rm -rf "$DEST"
mv "$TMP" "$DEST"
echo "oracle/_ref installed: $(find "$DEST/torch_geometric" -name '*.py' | wc -l) python files identical to $SRC"
