"""CPU oracle for stages 01-03 -- TEST INFRASTRUCTURE ONLY.

Nothing under oracle/ may be imported by the product package; only tests/, __graft_entry__.smoke()
and bench.py's CPU-baseline legs use it, and only as the checker / the timed CPU baseline.

  oracle.cmodel   plain-C integer/float restatement of the OpenCV/NumPy arithmetic (omni_oracle.c)
  oracle.refport  replay of the reference's own cv2/NumPy call sites (needs cv2), i.e. the
                  reference CPU implementation of the path with the file/PNG I/O stripped
  oracle.kmeans_model  NumPy restatement of the opt-in device k-means (kmeans.cu), bit for bit
"""
