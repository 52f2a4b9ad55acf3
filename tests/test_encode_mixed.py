"""CPU: the argument checks of files.encode_files with one bitrate per file, which run before any GPU work."""
import pytest

from conftest import synth_wav


def _wavs(tmp_path, n):
    from mp3stego_b200.wavio import write_wav
    paths = []
    for i, sr in zip(range(n), (44100, 48000, 32000)):
        p = str(tmp_path / f"in{i}.wav")
        write_wav(p, sr, synth_wav(i, 1, sr=sr))
        paths.append(p)
    return paths


@pytest.mark.parametrize("bad", [100, 330, 0])
def test_unsupported_entry_exits_like_the_reference(tmp_path, bad):
    from mp3stego_b200 import files
    wavs = _wavs(tmp_path, 3)
    outs = [str(tmp_path / f"out{i}.mp3") for i in range(3)]
    with pytest.raises(SystemExit, match="^Unsupported bitrate configuration.$"):
        files.encode_files(None, wavs, outs, bitrate=[128, bad, 320])
    assert not any((tmp_path / f"out{i}.mp3").exists() for i in range(3))


def test_one_bitrate_per_file(tmp_path):
    from mp3stego_b200 import files
    wavs = _wavs(tmp_path, 2)
    with pytest.raises(ValueError, match="one bitrate per input file"):
        files.encode_files(None, wavs, [str(tmp_path / "a.mp3"), str(tmp_path / "b.mp3")], bitrate=[128])
