"""Host-side utilities of the audio2vid / vid2vid scripts on the device: face-mesh pose maps (draw_util) and head-pose
smoothing and projection (pose_util)."""
