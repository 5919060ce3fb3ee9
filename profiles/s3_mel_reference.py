"""Checker for the S3 tokenizer's log-mel front end: the reference's ``log_mel_spectrogram``
(tools/S3Tokenizer/s3tokenizer/utils.py, the Whisper front end) restated line for line with ``torch.stft``.  It is what
tests/test_s3_mel_*.py and profiles/time_s3_audio.py compare the kernel (csrc/s3_mel.cu) against; it is never on the
product path."""
import torch


def s3_log_mel(audio, filters):
    """One 16 kHz clip, in the dtype and on the device of ``audio``: audio [S] (S > 200), filters [n_mels, 201] ->
    [n_mels, S // 160]."""
    window = torch.hann_window(400, dtype=audio.dtype, device=audio.device)
    stft = torch.stft(audio, 400, 160, window=window, return_complex=True)
    magnitudes = stft[..., :-1].abs() ** 2
    mel_spec = filters.to(audio.dtype) @ magnitudes
    log_spec = torch.clamp(mel_spec, min=1e-10).log10()
    log_spec = torch.maximum(log_spec, log_spec.max() - 8.0)
    return (log_spec + 4.0) / 4.0
