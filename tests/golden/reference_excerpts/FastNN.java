		NetMakerOriginal.NMMode myMode = NetMakerOriginal.NMMode.CANONICAL;
		//NamesAndDistances myND;
				beginTimer = System.nanoTime();
				ordering = myNMO.runNeighborNet();
				endTimer = System.nanoTime();
//			} else {
				ordering = myNMO.runNeighborNet();
//			}
		}
		int dim = (nTaxa * (nTaxa - 1)) /2;
