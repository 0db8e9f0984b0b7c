#!/bin/bash
# Regenerate every golden fixture from the reference checkout (authoring container only: needs /root/reference; CPU, ~15 min,
# most of it the B = 32 / 512^2 GAN goldens).  Each script's docstring says which reference code it executes and how.
set -e
cd "$(dirname "$0")/../.."
for s in pointcloud silhouette_losses mesh template renderer pose recon recon_step gan wrapper gan_loop syncbn fid fid_loop pseudogt; do
  echo "== make_golden_$s.py"
  python tests/golden/make_golden_$s.py
done
echo "== make_golden_reference_state.py"
python tests/golden/make_golden_reference_state.py "${REFERENCE_CODE:?set REFERENCE_CODE to the original project's code directory}"
cp "$REFERENCE_CODE"/mesh_templates/uvsphere_{16,31}rings.obj tests/golden/
git status --short tests/golden
