#!/bin/sh
# Installs the unmodified reference package (mapbox/robosat 1.2.0, pure Python) into oracle/_ref/robosat for the benchmark's
# reference arms (bench.py cpu_baseline and reference_cudnn, imported through baseline/ref_loader.py). oracle/_ref/ is
# git-ignored and is not part of the product. The source tree is $RSB_REFERENCE_SRC, else BASELINE.json's "reference_path".
# Where that tree is not readable nothing is installed, an oracle/_ref/ installed earlier is kept, and the benchmark states
# which implementation its reference arms ran.
set -e
cd "$(dirname "$0")"
SRC=${RSB_REFERENCE_SRC:-$(python3 -c 'import json; print(json.load(open("../BASELINE.json"))["reference_path"])')}
if [ ! -r "$SRC/robosat/unet.py" ]; then
  if [ -f _ref/robosat/unet.py ]; then
    echo "reference source $SRC is not readable: keeping the installed $(pwd)/_ref"
  else
    echo "reference source $SRC is not readable: the reference is not installed (bench.py's reference arms report this)"
  fi
  exit 0
fi
rm -rf _ref
mkdir -p _ref
cp -R "$SRC/robosat" _ref/robosat
echo "installed the reference from $SRC into $(pwd)/_ref"
