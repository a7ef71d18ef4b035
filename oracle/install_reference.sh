#!/bin/bash
# Copy the UNMODIFIED reference package (baybe) into oracle/_ref (git-ignored build product) for the tests that
# drive baybe's own Campaign.  The source tree is $BAYBE_REFERENCE, by default /root/reference; without a readable
# one this does nothing and those tests skip.  Only the package directory is copied: baybe needs no install
# metadata (its version then reads "unknown").  Its dependencies are not installed: botorch / gpytorch / cattrs
# may be absent, so only the parts of baybe that do not import them are used (Campaign, search spaces, the
# recommender base classes); tests/shims/cattrs stands in for cattrs.
set -e
cd "$(dirname "$0")/.."
SRC=${BAYBE_REFERENCE:-/root/reference}
if ! [ -r "$SRC/baybe/__init__.py" ] || ! [ -x "$SRC/baybe" ]; then
  echo "no readable baybe source tree at $SRC: oracle/_ref not built"
  exit 0
fi
if [ -f oracle/_ref/.complete ]; then echo "oracle/_ref present"; exit 0; fi
rm -rf oracle/_ref
mkdir -p oracle/_ref
cp -r "$SRC/baybe" oracle/_ref/
chmod -R u+w oracle/_ref
touch oracle/_ref/.complete
echo "copied $(find oracle/_ref/baybe -name '*.py' | wc -l) modules of $SRC/baybe into oracle/_ref"
