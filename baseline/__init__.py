"""Harness around the UNMODIFIED reference (copied into oracle/_ref by oracle/install_ref.sh)."""
