"""CPU oracle for the VLFM perception -> value-map hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``vlfm_b200/`` may import this package; the
only legal importers are ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs, and there only as the checker or as the
CPU baseline being reported -- never as the product path.

Contents
--------
``cv_prims``            numpy restatement of the OpenCV rasterisation rules the path
                        depends on (8-connected line, even-odd polygon fill, fixed-point
                        bilinear warpAffine, box dilation), pinned against cv2 itself.
``value_map_oracle``    restatement of ``vlfm/mapping/value_map.py`` (+ the pieces of
                        ``vlfm/utils/img_utils.py`` / ``geometry_utils.py`` it calls).
``obstacle_map_oracle`` restatement of ``vlfm/mapping/obstacle_map.py`` including the
                        third-party ``frontier_exploration`` functions it calls
                        (that package is absent from /root/reference: parity for the
                        fog-of-war / frontier half is UNPINNED, see DESIGN.md).
``blip2_oracle``        architecture-equivalent fp32 BLIP-2 ITC forward built on
                        HF transformers (LAVIS is absent: parity UNPINNED w.r.t. LAVIS).
``ref_import``          imports the real reference from a checkout named by VLFM_REFERENCE
                        (used only by ``make_golden`` to generate tests/golden/*).
``golden``              compact storage of, and exact comparison with, the stored
                        reference outputs under tests/golden/.

Pinning status is recorded per module in its header and in DESIGN.md.
"""
