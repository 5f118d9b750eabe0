#!/usr/bin/env bash
# Installs the UNMODIFIED reference (KinWaiCheuk/nnAudio v0.3.3) into oracle/_ref (git-ignored) so that
# `bench.py --impl reference`, its `cpu_baseline` and its `reference_gpu` leg time the reference's own
# code.  The reference is pure Python with no compiled parts, so installing it is copying its package.
# Without a reference checkout ($NNAUDIO_REF) this does nothing and bench.py times the NumPy oracle.
set -euo pipefail
root="$(cd "$(dirname "${BASH_SOURCE[0]}")/.." && pwd)"
src="${NNAUDIO_REF:-/root/reference/Installation}"
[ -d "$src/nnAudio" ] || { echo "no reference at $src: oracle/_ref not installed"; exit 0; }
dst="$root/oracle/_ref"
tmp="$dst.tmp.$$"
trap 'rm -rf "$tmp"' EXIT
mkdir -p "$tmp"
cp -r "$src/nnAudio" "$tmp/nnAudio"
chmod -R u+w "$tmp"   # the checkout may be read-only; the copy must stay removable
rm -rf "$dst"
mv "$tmp" "$dst"
echo "installed reference into $dst"
