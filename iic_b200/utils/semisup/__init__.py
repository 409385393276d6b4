"""Drop-in for code/utils/semisup/ of the reference (the device part of the semi-supervised finetune)."""
