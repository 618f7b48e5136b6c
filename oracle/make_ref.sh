#!/bin/bash
# oracle/make_ref.sh -- make the LIVE reference importable on the GPU box: copy the reference's own Python package
# (pure Python, nothing to compile) from /root/reference into the git-ignored oracle/_ref/.  The directory is
# NOT in .gpurunignore, so it travels with the gpurun snapshot like the built libsmcb.so; nothing from the
# reference enters the repository history.  Used by (i) tests/test_gpu_dropin.py: real reference objects
# (particles.state_space_models.StochVol ...) through particles_b200.install() -> fused kernels, and (ii)
# bench.py --impl reference: the real particles.SMC timed on the box's host cores (kind "reference").
# TEST / BASELINE INFRASTRUCTURE: the product never imports it.
set -e
cd "$(dirname "$0")"
SRC=${1:-/root/reference}
if [ ! -d "$SRC/particles" ]; then echo "no reference at $SRC: oracle/_ref left as it is"; exit 0; fi
# a read-only reference checkout must not give a read-only copy: the next line, and the next build, delete in it
if [ -d _ref ]; then chmod -R u+w _ref; fi
rm -rf _ref && mkdir -p _ref
cp -r --no-preserve=mode "$SRC/particles" _ref/particles
rm -rf _ref/particles/datasets _ref/particles/__pycache__        # 3 MB of data files the hot path never reads
cp "$SRC/LICENSE" _ref/LICENSE 2>/dev/null || true
echo "oracle/_ref/particles: $(find _ref -name '*.py' | wc -l) modules"
